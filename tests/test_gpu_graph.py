"""The train step replayed as one CUDA graph (pseudo_speaker_vae_b200/graphs.py) against the eager DataParallelTrainer, and the device-counter
entry points it is built on (psvae_adam_step_dc, psvae_train_fwd_bwd_dc, psvae_step_counters_advance)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _lib():
    from pseudo_speaker_vae_b200 import _lib as L
    return L


# ---- Adam with t and lr in device memory ------------------------------------------------------------
@pytest.mark.parametrize("amsgrad,maximize,wd", [(False, False, 0.0), (False, False, 0.01), (True, False, 0.0), (False, True, 0.01), (True, True, 0.01)])
def test_adam_dc_is_bit_identical_to_host_scalar_adam(amsgrad, maximize, wd):
    """psvae_adam_step_dc (t from the counter block, lr from a device fp64 array changed mid-run) against psvae_adam_step / _ex with the same
    t and lr: p, m, v, vmax bit-identical, the bf16 shadow the rounding of p, the counters advanced once per step."""
    L = _lib()
    lib = L.lib()
    z = np.load(os.path.join(GOLDEN, "adam_cosine.npz"))
    lrs = [3e-3, 3e-3, 1.1e-3, 4.7e-4]             # a scheduler step between steps 2 and 3, another before 4
    gscale = 0.5
    p0 = torch.from_numpy(z["p0"].copy()).to(DEV)
    bufs = {k: [p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0), torch.zeros_like(p0), torch.empty(p0.numel(), dtype=torch.bfloat16, device=DEV)]
            for k in ("ref", "dc")}
    counters = torch.zeros(L.COUNTER_SLOTS, dtype=torch.int64, device=DEV)
    lr_dev = torch.zeros(1, dtype=torch.float64, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    for s, g in enumerate(z["grads"]):
        gt = torch.from_numpy(g.astype(np.float32)).to(DEV)
        p, m, v, x, sh = bufs["ref"]
        if amsgrad or maximize:
            rc = lib.psvae_adam_step_ex(p.data_ptr(), gt.data_ptr(), m.data_ptr(), v.data_ptr(), L.ptr(x) if amsgrad else None, p.numel(), lrs[s], 0.9, 0.999,
                                        1e-8, wd, s + 1, gscale, int(amsgrad), int(maximize), sh.data_ptr(), st)
        else:
            rc = lib.psvae_adam_step(p.data_ptr(), gt.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lrs[s], 0.9, 0.999, 1e-8, wd, s + 1, gscale,
                                     sh.data_ptr(), st)
        L.check(rc, "psvae_adam_step")
        lr_dev.fill_(lrs[s])
        p, m, v, x, sh = bufs["dc"]
        L.check(lib.psvae_adam_step_dc(p.data_ptr(), gt.data_ptr(), m.data_ptr(), v.data_ptr(), L.ptr(x) if amsgrad else None, p.numel(), lr_dev.data_ptr(),
                                       counters.data_ptr(), 0.9, 0.999, 1e-8, wd, gscale, int(amsgrad), int(maximize), sh.data_ptr(), st), "psvae_adam_step_dc")
        L.check(lib.psvae_step_counters_advance(counters.data_ptr(), st), "psvae_step_counters_advance")
        for a, b, name in zip(bufs["ref"], bufs["dc"], ("p", "m", "v", "vmax", "shadow")):
            assert torch.equal(a, b), (name, s)
        assert torch.equal(bufs["dc"][4], bufs["dc"][0].to(torch.bfloat16))
    assert counters[L.COUNTER_RNG_OFFSET].item() == len(lrs) and counters[L.COUNTER_ADAM_STEP].item() == len(lrs)


# ---- graphed vs eager trajectories --------------------------------------------------------------------
CASES = {
    # the benchmark's model (bf16 tensor cores, 2-class linear classifier) at the reference's batch size
    "bf16_d256_c2": dict(hp=dict(model=dict(input_dim=256, latent_dim=64), classifier=dict(input_dim=64, num_classes=2)), precision="bf16", rows=2048),
    # fp32 parity engine, no classifier, a ragged batch
    "fp32_d192_noclf": dict(hp=dict(model=dict(input_dim=192, latent_dim=32, hidden_dim=256)), precision="fp32", rows=1000),
    # the consistency classifier on x_hat and the L2-normalised decoder
    "bf16_cons_norm": dict(hp=dict(model=dict(input_dim=256, latent_dim=64, normalize_decoder=True), classifier=dict(input_dim=64, num_classes=2)),
                           precision="bf16", rows=512, cons=True),
}


def _module(case, seed=0):
    import pseudo_speaker_vae_b200 as P

    c = CASES[case]
    torch.manual_seed(seed)
    m = P.PseudoSpeakerVAE(**c["hp"], optimizer=dict(lr=2e-3), scheduler=dict(T_max=5), precision=c["precision"])
    if c.get("cons"):
        ec = P.EmbeddingClassifier(input_dim=c["hp"]["model"]["input_dim"], num_classes=2, hidden_dim=128)
        for p in ec.parameters():
            p.requires_grad = False
        ec.eval()
        m.consistency_classifier = ec
    return m.to(DEV)


def _batches(case, n, rows=None, seed=5):
    c = CASES[case]
    D = c["hp"]["model"]["input_dim"]
    rows = rows or c["rows"]
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        x = torch.randn(rows, D, generator=g)
        x = x / x.norm(dim=1, keepdim=True)
        y = torch.randint(0, 2, (rows,), generator=g)
        out.append((x.to(DEV), y.to(DEV)))
    return out


class _deterministic:
    def __init__(self, value):
        self.value = value

    def __enter__(self):
        L = _lib()
        self.prev = L.get_option("deterministic")
        L.set_option("deterministic", self.value)

    def __exit__(self, *exc):
        _lib().set_option("deterministic", self.prev)


def _run(case, graphed, batches, sched_every=3):
    """K steps with Philox eps (no injection), a cosine scheduler stepped every `sched_every` steps.  Returns the end state and per-step losses."""
    import pseudo_speaker_vae_b200 as P

    L = _lib()
    m = _module(case)
    m.hot_path.manual_seed(77, 0)
    tr = P.DataParallelTrainer(m, local_only=True)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(tr.optimizer, T_max=5)
    step = P.GraphedTrainStep(tr, rows=CASES[case]["rows"]) if graphed else tr.train_step
    losses, launches = [], []
    for s, (x, y) in enumerate(batches):
        losses.append(step(x, y).clone())
        launches.append(int(L.lib().psvae_launch_count()))
        if s % sched_every == sched_every - 1:
            sched.step()
    torch.cuda.synchronize()
    opt = tr.optimizer
    p0 = next(iter(m.parameters()))
    return dict(p=m.hot_path.arena.flat.detach().clone(), m=opt._m.clone(), v=opt._v.clone(), losses=torch.stack(losses), offset=m.hot_path.offset,
                step=float(opt.state[p0]["step"]), launches=launches, graph=step if graphed else None)


@pytest.mark.parametrize("case", list(CASES))
def test_graphed_trajectory_is_bit_identical(case):
    """Deterministic summation mode, 8 steps: the graphed run (call 1 eager, call 2 capture + replay, then replays) equals the eager run bit for bit
    in parameters, moments, per-step losses, the host Philox offset and Adam's step count; replays launch nothing from the host."""
    batches = _batches(case, 8)
    with _deterministic(1):
        eager = _run(case, False, batches)
        graph = _run(case, True, batches)
    for k in ("p", "m", "v", "losses"):
        assert torch.equal(eager[k], graph[k]), (case, k, (eager[k] - graph[k]).abs().max().item())
    assert eager["offset"] == graph["offset"] == 8 and eager["step"] == graph["step"] == 8.0
    assert graph["graph"].replays == 7
    assert len(set(graph["launches"][1:])) == 1, graph["launches"]          # psvae_launch_count does not move across replays
    assert torch.isfinite(graph["losses"]).all()


def test_graphed_fast_mode_within_eager_run_to_run_spread():
    """Fast mode (atomic sums; the fused encoder head draws its own eps in the GEMM epilogue): graphed vs eager differ by no more than twice
    what two eager runs differ by (the floor is one fp32 rounding of the parameter norm: the atomic order is random per run, so two eager
    runs may by chance agree more closely than a third run does)."""
    case = "bf16_d256_c2"
    batches = _batches(case, 8)
    with _deterministic(0):
        a = _run(case, False, batches)
        b = _run(case, False, batches)
        g = _run(case, True, batches)
    rel = lambda u, w: float((u["p"] - w["p"]).double().norm() / w["p"].double().norm())
    d_ee, d_ge = rel(a, b), rel(g, a)
    assert d_ge <= 2 * d_ee + 6e-8, (d_ge, d_ee)
    assert torch.allclose(g["losses"], a["losses"], rtol=1e-3, atol=1e-5)
    assert g["offset"] == a["offset"] and g["step"] == a["step"]


def test_interleaved_eager_steps_lr_change_and_checkpoint_resume():
    """graph, graph, an eager tail batch of another size, an lr change, graph; then state_dict() into a fresh module + trainer (the Philox offset
    resumed with hot_path.manual_seed) and two more graphed calls: bit-identical to one uninterrupted eager run."""
    import pseudo_speaker_vae_b200 as P

    case = "bf16_d256_c2"
    rows = 1024
    main = _batches(case, 7, rows=rows)
    tail = _batches(case, 1, rows=640, seed=9)[0]
    plan = [main[0], main[1], main[2], tail, main[3], main[4], main[5], main[6]]
    with _deterministic(1):
        ref = _module(case)
        ref.hot_path.manual_seed(31, 0)
        tr = P.DataParallelTrainer(ref, local_only=True)
        for i, (x, y) in enumerate(plan):
            if i == 4:
                for g in tr.optimizer.param_groups:
                    g["lr"] = 7e-4
            tr.train_step(x, y)

        m = _module(case)
        m.hot_path.manual_seed(31, 0)
        tr1 = P.DataParallelTrainer(m, local_only=True)
        step = P.GraphedTrainStep(tr1, rows=rows)
        for i, (x, y) in enumerate(plan[:6]):
            if i == 4:
                for g in tr1.optimizer.param_groups:
                    g["lr"] = 7e-4
            step(x, y)
        assert step.replays == 4          # calls 2, 3, 5 and 6 replayed; call 1 warmed up, call 4 was the tail
        sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
        osd = tr1.optimizer.state_dict()
        offset = m.hot_path.offset
        assert offset == 6 and int(osd["state"][0]["step"]) == 6

        m2 = _module(case, seed=1)
        m2.load_state_dict(sd)
        m2.hot_path.manual_seed(31, offset)
        tr2 = P.DataParallelTrainer(m2, local_only=True)
        tr2.optimizer.load_state_dict(osd)
        step2 = P.GraphedTrainStep(tr2, rows=rows)
        for x, y in plan[6:]:
            step2(x, y)
        torch.cuda.synchronize()
    assert torch.equal(m2.hot_path.arena.flat, ref.hot_path.arena.flat)
    assert torch.equal(tr2.optimizer._m, tr.optimizer._m) and torch.equal(tr2.optimizer._v, tr.optimizer._v)
    assert m2.hot_path.offset == ref.hot_path.offset == 8


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_graphed_data_parallel_step_on_real_ranks():
    """2 ranks: graphed data-parallel steps (all-reduce inside the graph) equal eager data-parallel steps bit for bit, on identical ranks."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29543",
           os.path.join(ROOT, "tests", "graph_dp_case.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in res.stdout.splitlines() if l.startswith("RESULT ")]
    assert res.returncode == 0 and len(lines) == 2, res.stdout[-2000:] + res.stderr[-2000:]
    for l in lines:
        r = json.loads(l[len("RESULT "):])
        assert r["bit_identical"] and r["ranks_identical"] and r["replays"] >= 3, r


def test_larger_eager_calls_between_replays_do_not_move_the_graphs_scratch():
    """An eager step on a LARGER batch and a forward pass on more rows grow HotPath's cached workspace (the old tensor is replaced); the graph
    keeps the one it was captured with.  graph, graph, eager 1,536 rows, forward on 8,192 rows, a decoy allocation of the captured workspace's
    size, graph, graph: bit-identical to the same sequence run eagerly, and the decoy untouched."""
    import pseudo_speaker_vae_b200 as P

    case, rows = "bf16_d256_c2", 1024
    main = _batches(case, 6, rows=rows)
    big = _batches(case, 1, rows=1536, seed=8)[0]
    probe = _batches(case, 1, rows=8192, seed=10)[0][0]
    results = []
    with _deterministic(1):
        for graphed in (False, True):
            m = _module(case)
            m.hot_path.manual_seed(41, 0)
            tr = P.DataParallelTrainer(m, local_only=True)
            step = P.GraphedTrainStep(tr, rows=rows) if graphed else tr.train_step
            for x, y in main[:3]:
                step(x, y)
            ws0 = m.hot_path._ws[torch.device(DEV)]
            step(*big)
            with torch.no_grad():
                xh, _, _ = m.hot_path.forward(probe)
            assert m.hot_path._ws[torch.device(DEV)].numel() > ws0.numel()       # the cached workspace was replaced by a larger one
            nbytes = ws0.numel()
            del ws0                # the graph's own reference, if any, is now the only one
            decoy = torch.full((nbytes,), 7, dtype=torch.uint8, device=DEV)
            losses = [step(x, y).clone() for x, y in main[3:]]
            torch.cuda.synchronize()
            assert bool((decoy == 7).all())
            results.append((m.hot_path.arena.flat.detach().clone(), torch.stack(losses), xh))
            if graphed:
                assert step.replays == 5          # calls 2, 3 and the three after the larger eager calls
    assert torch.equal(results[0][0], results[1][0]) and torch.equal(results[0][1], results[1][1]) and torch.equal(results[0][2], results[1][2])


def test_batch_dtype_and_label_structure():
    """A batch of another dtype than the graph's static buffer is refused, not converted; a call whose labels differ in structure from the
    captured ones (here: labels, then none, on a model without a classifier) re-captures instead of replaying stale labels."""
    import pseudo_speaker_vae_b200 as P

    case = "fp32_d192_noclf"
    bs = _batches(case, 5)
    with _deterministic(1):
        m = _module(case)
        tr = P.DataParallelTrainer(m, local_only=True)
        step = P.GraphedTrainStep(tr, rows=CASES[case]["rows"])
        step(*bs[0])
        step(*bs[1])
        g0 = step.graph
        with pytest.raises(ValueError, match="dtype|float"):
            step(bs[2][0].to(torch.bfloat16), bs[2][1])
        step(bs[2][0], None)
        assert step.graph is not g0 and step.replays == 2
        step(bs[3][0], None)
        assert step.replays == 3
    with pytest.raises(ValueError):
        P.GraphedTrainStep(tr, rows=CASES[case]["rows"], x_dtype=torch.bfloat16)(*bs[4])


def test_fused_head_reads_the_philox_offset_from_the_counter_block():
    """Fast mode, the benchmark's model: the fused encoder head (Philox in the GEMM epilogue) with counters holding offset k gives the same
    mu, log_sigma and x_hat, bit for bit, as the host-offset entry point at offset k -- while the host offset passed alongside is
    a different one -- and offset k + 1 in the block gives other noise."""
    L = _lib()
    case = "bf16_d256_c2"
    x, y = _batches(case, 1)[0]
    with _deterministic(0):
        m = _module(case)
        hot = m.hot_path
        counters = torch.zeros(L.COUNTER_SLOTS, dtype=torch.int64, device=DEV)
        outs = {}
        for name, dev_off, host_off in (("host", None, 5), ("dev", 5, 900), ("dev_next", 6, 900)):
            hot.manual_seed(123, host_off)
            c = None
            if dev_off is not None:
                counters[L.COUNTER_RNG_OFFSET] = dev_off
                c = counters
            losses, _, (xh, mu, ls) = hot.step(x, y, want_outputs=True, counters=c)
            torch.cuda.synchronize()
            outs[name] = (losses.clone(), xh.clone(), mu.clone(), ls.clone())
    for a, b, what in zip(outs["host"][1:], outs["dev"][1:], ("x_hat", "mu", "log_sigma")):
        assert torch.equal(a, b), what
    assert torch.equal(outs["dev"][2], outs["dev_next"][2])          # mu does not depend on the noise ...
    assert not torch.equal(outs["dev"][1], outs["dev_next"][1])      # ... x_hat (through z) does


def test_adam_dc_scalars_match_the_host_over_a_long_run():
    """The device forms lr/(1-beta1^t) and sqrt(1-beta2^t) with its own pow; the host uses the C library's.  Over t = 1 ... 100,000 (the
    reference trains 59,400 steps) the device-counter update and the host-scalar update of the same 1,024 parameters stay bit-identical: a
    one-ulp difference in either scalar would change the rounding of most of the updated elements."""
    L = _lib()
    lib = L.lib()
    n, T = 1024, 100_000
    g = torch.Generator().manual_seed(3)
    p0 = torch.randn(n, generator=g).to(DEV)
    m0 = (torch.randn(n, generator=g) * 1e-2).to(DEV)
    v0 = (torch.rand(n, generator=g) * 1e-3).to(DEV)
    grad = (torch.randn(n, generator=g) * 1e-2).to(DEV)
    st = torch.cuda.current_stream().cuda_stream
    for beta1, beta2 in ((0.9, 0.999), (0.8, 0.99)):
        ref = [p0.clone(), m0.clone(), v0.clone()]
        dc = [p0.clone(), m0.clone(), v0.clone()]
        counters = torch.zeros(L.COUNTER_SLOTS, dtype=torch.int64, device=DEV)
        lr_dev = torch.full((1,), 1e-3, dtype=torch.float64, device=DEV)
        for t in range(1, T + 1):
            L.check(lib.psvae_adam_step(ref[0].data_ptr(), grad.data_ptr(), ref[1].data_ptr(), ref[2].data_ptr(), n, 1e-3, beta1, beta2, 1e-8, 0.0, t, 1.0,
                                        None, st))
            L.check(lib.psvae_adam_step_dc(dc[0].data_ptr(), grad.data_ptr(), dc[1].data_ptr(), dc[2].data_ptr(), None, n, lr_dev.data_ptr(),
                                           counters.data_ptr(), beta1, beta2, 1e-8, 0.0, 1.0, 0, 0, None, st))
            L.check(lib.psvae_step_counters_advance(counters.data_ptr(), st))
            if t % 10_000 == 0:
                assert all(torch.equal(a, b) for a, b in zip(ref, dc)), (beta1, beta2, t)
                # restart from the same state: the next window is compared on fresh values, not on a settled steady state
                for a, b, s in zip(ref, dc, (p0, m0, v0)):
                    a.copy_(s)
                    b.copy_(s)
        assert counters[L.COUNTER_ADAM_STEP].item() == T
