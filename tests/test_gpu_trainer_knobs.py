"""Gradient accumulation and clipping of DataParallelTrainer / GraphedTrainStep on the GPU: the accumulating fused step against the
writing one, accumulation against the drop-in's Lightning-style path, norm and value clipping against torch, graphed against eager, no
host synchronisation, and two ranks."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ps_vae_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
MULTI = dict(D=256, L=64, wseed=3, clf=dict(input_dim=64, num_classes={"age": 3, "gender": 2}))


def _gu():
    from tests import gpu_util as G
    return G


class _deterministic:
    def __init__(self, value):
        self.value = value

    def __enter__(self):
        from pseudo_speaker_vae_b200 import _lib as L
        self.prev = L.get_option("deterministic")
        L.set_option("deterministic", self.value)

    def __exit__(self, *exc):
        from pseudo_speaker_vae_b200 import _lib as L
        L.set_option("deterministic", self.prev)


def _cfg(name):
    from tests.golden_util import load
    return MULTI if name == "multilabel" else load(name)[1]


def _batch(cfg, rows, seed):
    G = _gu()
    nc = cfg["clf"]["num_classes"] if cfg.get("clf") else 2
    x, y, eps = O.synth_batch(rows, cfg["D"], cfg["L"], nc, seed=seed)
    return torch.from_numpy(x).to(DEV), G.labels_to_torch(y), torch.from_numpy(eps).to(DEV)


def _padding_mask(module):
    arena = module.hot_path.arena
    mask = torch.ones(arena.numel, dtype=torch.bool, device=DEV)
    for p, off in arena.entries:
        mask[off:off + p.numel()] = False
    return mask


# ---- 1. the accumulating step adds exactly what the writing step writes --------------------------------------------------------------
@pytest.mark.parametrize("name", ["train_d256_c2", "train_d192_c3_cons_norm_cos", "train_d512_c3_mlp", "train_d192_noclf", "multilabel"])
@pytest.mark.parametrize("mode", ["fp32", "bf16_det", "bf16_fast"])
def test_accumulating_step_adds_the_writing_steps_gradient(name, mode):
    """Pre-fill the gradient buffer with a seeded R, run the accumulating step, compare with R + g (g: the writing step on the same inputs).
    Deterministic modes bit for bit, padding included; fast mode (atomics) to 1e-5, padding still R bit for bit."""
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    cfg = _cfg(name)
    precision = "fp32" if mode == "fp32" else "bf16"
    with _deterministic(0 if mode == "bf16_fast" else 1):
        m = G.module_from_cfg(cfg, precision)
        tr = P.DataParallelTrainer(m, local_only=True, accumulate_grad_batches=2)
        x, y, eps = _batch(cfg, 300, seed=41)
        xs = [x] + ([x.to(torch.bfloat16)] if mode == "bf16_fast" and name == "train_d256_c2" else [])     # + the bf16-x clear-only path
        for xx in xs:
            _, gflat = tr._fwd_bwd(xx, y, eps)
            g = gflat.clone()
            gen = torch.Generator(device=DEV).manual_seed(7)
            R = torch.randn(g.numel(), device=DEV, generator=gen) * g.abs().mean()
            gflat.copy_(R)
            _, gacc = tr._fwd_bwd(xx, y, eps, accumulate=True)
            assert gacc.data_ptr() == gflat.data_ptr()
            pad = _padding_mask(m)
            assert torch.equal(gacc[pad], R[pad])
            if mode == "bf16_fast":
                from tests.golden_util import rel_err
                assert rel_err(gacc.cpu().numpy(), (R + g).cpu().numpy()) <= 1e-5
            else:
                assert torch.equal(gacc, R + g)


# ---- 2. accumulation against the Lightning-style path --------------------------------------------------------------------------------
def _lightning_run(cfg, precision, batches, k):
    """Returns the parameters at the end and the gradient the last optimiser step consumed (Lightning's .grad: the mean)."""
    G = _gu()
    m = G.module_from_cfg(cfg, precision)
    opt = m.configure_optimizers()["optimizer"]
    last_grad = None
    for i, (x, y, eps) in enumerate(batches):
        loss = m.training_step((x, y), i, eps=eps)["loss"]
        (loss / k).backward()
        if (i + 1) % k == 0:
            last_grad = m.hot_path.arena.flat_grad().clone()
            opt.step()
            opt.zero_grad(set_to_none=True)
    return m.hot_path.arena.flat.detach().clone(), last_grad


def _trainer_run(cfg, precision, batches, k, **kw):
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    m = G.module_from_cfg(cfg, precision)
    tr = P.DataParallelTrainer(m, local_only=True, accumulate_grad_batches=k, **kw)
    for x, y, eps in batches:
        tr.train_step(x, y, eps)
    return m.hot_path.arena.flat.detach().clone(), tr


@pytest.mark.parametrize("k", [2, 3, 4])
def test_accumulation_matches_the_lightning_style_path(k):
    """k micro-batches through the trainer against training_step + (loss / k).backward() + FusedAdam.step() every k calls (injected eps,
    deterministic mode): bit-identical for k = 2, 4 (scaling by a power of two is exact).  For k = 3 the two paths round differently
    (sum of g_i / 3 against (sum of g_i) / 3): the gradient the first Adam step consumes is within 1e-6; the parameters after two steps
    are within 1e-5, because Adam's first steps divide by sqrt(v) ~ |g| and so turn last-bit differences of near-zero gradient elements
    into updates of up to lr."""
    from tests.golden_util import rel_err

    cfg = _cfg("train_d256_c2")
    batches = [_batch(cfg, 512, seed=100 + i) for i in range(2 * k)]
    with _deterministic(1):
        ref, _ = _lightning_run(cfg, "bf16", batches, k)
        got, _ = _trainer_run(cfg, "bf16", batches, k)
        if k == 3:
            _, ref_grad = _lightning_run(cfg, "bf16", batches[:k], k)
            _, tr = _trainer_run(cfg, "bf16", batches[:k], k)
    if k in (2, 4):
        assert torch.equal(got, ref)
    else:
        eff = (tr.hot.arena.flat_grad() * tr.optimizer.grad_scale).cpu().numpy()
        assert rel_err(eff, ref_grad.cpu().numpy()) <= 1e-6
        assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) <= 1e-5


def test_row_slices_of_one_batch_match_the_single_batch_step():
    """k = 4 micro-batches that are the row slices of one batch land within 1e-6 (fp32 mode) of one step on the whole batch."""
    from tests.golden_util import rel_err

    cfg = _cfg("train_d256_c2")
    x, y, eps = _batch(cfg, 1024, seed=9)
    with _deterministic(1):
        one, tr1 = _trainer_run(cfg, "fp32", [(x, y, eps)], 1)
        sl = [slice(i * 256, (i + 1) * 256) for i in range(4)]
        four, tr4 = _trainer_run(cfg, "fp32", [(x[s], y[s], eps[s]) for s in sl], 4)
    g1 = tr1.hot.arena.flat_grad().cpu().numpy()
    g4 = tr4.hot.arena.flat_grad().cpu().numpy() / 4           # .grad holds the SUM of the micro-batch gradients
    assert rel_err(g4, g1) <= 1e-6
    assert rel_err(four.cpu().numpy(), one.cpu().numpy()) <= 1e-6


# ---- 3. clipping --------------------------------------------------------------------------------------------------------------------
def test_norm_clipping_matches_clip_grad_norm_and_torch_adam():
    G = _gu()
    from tests.golden_util import rel_err

    cfg = _cfg("train_d512_c3_mlp")
    x, y, eps = _batch(cfg, 512, seed=3)
    max_norm = 1e-3
    with _deterministic(1):
        m0 = G.module_from_cfg(cfg, "fp32")
        p0 = {k: p.detach().clone() for k, p in m0.named_parameters()}
        got, tr = _trainer_run(cfg, "fp32", [(x, y, eps)], 1, gradient_clip_val=max_norm)
    m = tr.module
    names = {id(p): k for k, p in m.named_parameters()}
    grads = {names[id(p)]: p.grad.detach().clone() for p, _ in tr.hot.arena.entries}
    gflat = tr.hot.arena.flat_grad().double()
    n64 = float(torch.linalg.vector_norm(gflat))
    tn = float(tr.grad_norm)
    assert abs(tn - n64) <= 1e-6 * n64 and tn > max_norm
    ref = {k: v.clone().requires_grad_(True) for k, v in p0.items()}
    for k, v in ref.items():
        v.grad = grads[k].clone()
    tn_torch = float(torch.nn.utils.clip_grad_norm_(list(ref.values()), max_norm))
    assert abs(tn - tn_torch) <= 1e-6 * tn_torch
    g0 = tr.optimizer.param_groups[0]
    torch.optim.Adam(list(ref.values()), lr=g0["lr"], betas=g0["betas"], eps=g0["eps"], weight_decay=g0["weight_decay"], foreach=False).step()
    for k, p in m.named_parameters():
        assert rel_err(p.detach().cpu().numpy(), ref[k].detach().cpu().numpy()) <= 1e-6, k


def test_norm_clipping_above_the_norm_is_the_unclipped_step():
    cfg = _cfg("train_d256_c2")
    batches = [_batch(cfg, 512, seed=20 + i) for i in range(3)]
    with _deterministic(1):
        plain, _ = _trainer_run(cfg, "bf16", batches, 1)
        clipped, tr = _trainer_run(cfg, "bf16", batches, 1, gradient_clip_val=1e9)
    tn = float(tr.grad_norm)
    diff = (plain != clipped)
    assert tn > 0 and float(tr._clip_coef) == 1.0, (tn, float(tr._clip_coef))
    assert torch.equal(plain, clipped), (int(diff.sum()), float((plain - clipped).abs().max()), diff.nonzero()[:8].flatten().tolist())


def test_value_clipping_is_fused_adam_on_a_clamped_gradient():
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    cfg = _cfg("train_d256_c2")
    x, y, eps = _batch(cfg, 512, seed=4)
    with _deterministic(1):
        m = G.module_from_cfg(cfg, "bf16")
        probe = P.DataParallelTrainer(m, local_only=True)
        _, g = probe._fwd_bwd(x, y, eps)
        v = float(g.abs().median())
        got, tr = _trainer_run(cfg, "bf16", [(x, y, eps)], 1, gradient_clip_val=v, gradient_clip_algorithm="value")
        ref = G.module_from_cfg(cfg, "bf16")
        opt = ref.configure_optimizers()["optimizer"]
        for (p, _), (q, _) in zip(tr.hot.arena.entries, ref.hot_path.arena.entries):
            q.grad = torch.clamp(p.grad, -v, v)
        opt.step()
    assert torch.equal(got, ref.hot_path.arena.flat.detach())


# ---- 4. graphed against eager -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,clip,algo,flush_at", [(1, 0.05, "norm", None), (3, 1e-4, "value", None), (4, 0.05, "norm", 5)])
def test_graphed_knobs_match_eager(k, clip, algo, flush_at):
    """Deterministic mode, Philox eps, a cosine scheduler stepped after every optimiser step, one eager micro-batch of another row count in
    the middle of a window: graphed and eager runs bit-identical (parameters, Adam moments, every returned loss)."""
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    cfg = _cfg("train_d256_c2")
    rows = 512
    calls = [_batch(cfg, rows, seed=60 + i)[:2] for i in range(12)]
    calls[7] = _batch(cfg, 256, seed=99)[:2]
    out = []
    with _deterministic(1):
        for graphed in (False, True):
            m = G.module_from_cfg(cfg, "bf16")
            m.hot_path.manual_seed(77, 0)
            tr = P.DataParallelTrainer(m, local_only=True, accumulate_grad_batches=k, gradient_clip_val=clip, gradient_clip_algorithm=algo)
            sched = torch.optim.lr_scheduler.CosineAnnealingLR(tr.optimizer, T_max=5)
            step = P.GraphedTrainStep(tr, rows=rows) if graphed else tr.train_step
            losses = []
            for i, (x, y) in enumerate(calls):
                flush = i == flush_at
                ends = tr._window_phase(flush)[1]
                losses.append(step(x, y, flush=flush).clone())
                if ends:
                    sched.step()
            torch.cuda.synchronize()
            out.append((m.hot_path.arena.flat.detach().clone(), tr.optimizer._m.clone(), torch.stack(losses), m.hot_path.offset))
            if graphed:
                assert step.replays >= 8
    for a, b in zip(out[0][:3], out[1][:3]):
        assert torch.equal(a, b)
    assert out[0][3] == out[1][3] == len(calls)


# ---- 5. no host synchronisation -----------------------------------------------------------------------------------------------------
def test_eager_knob_steps_do_not_synchronise():
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    cfg = _cfg("train_d256_c2")
    m = G.module_from_cfg(cfg, "bf16")
    tr = P.DataParallelTrainer(m, local_only=True, accumulate_grad_batches=2, gradient_clip_val=0.1)
    batches = [_batch(cfg, 512, seed=200 + i)[:2] for i in range(6)]
    for x, y in batches[:2]:                # first window: buffers and optimiser state are allocated
        tr.train_step(x, y)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for x, y in batches[2:]:
            tr.train_step(x, y)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.isfinite(tr.grad_norm)


# ---- 6. two ranks -------------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_knobs_on_two_ranks():
    """2 ranks with accumulation and norm clipping: ranks bit-identical, within 2e-6 of a single-process run on the whole batches."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29547",
           os.path.join(ROOT, "tests", "knobs_dp_case.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in res.stdout.splitlines() if l.startswith("RESULT ")]
    assert res.returncode == 0 and len(lines) == 2, res.stdout[-2000:] + res.stderr[-2000:]
    for l in lines:
        r = json.loads(l[len("RESULT "):])
        assert r["ranks_identical"] and r["param_rel_err"] <= 2e-6, r
