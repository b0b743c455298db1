"""The classifier-only train step (frozen VAE, ``freeze_vae``) on the GPU: the same losses, outputs and classifier gradients as the full
step, a gradient buffer of which only the classifier span changes, training runs against the full step, fewer launches and no shadow
refresh, the graphed step, and two ranks."""
import json
import os
import subprocess
import sys

import pytest
import torch

from oracle import ps_vae_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
MULTI = dict(D=256, L=64, wseed=3, clf=dict(input_dim=64, num_classes={"age": 3, "gender": 2}))
CASES = ["train_d256_c2", "train_d192_c3_cons_norm_cos", "train_d512_c3_mlp", "multilabel"]
MODES = ["fp32", "bf16_det", "bf16_fast"]


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


def _freeze(m, frozen=True):
    for p in m.model.parameters():
        p.requires_grad = not frozen


def _step(m, x, y, eps, scope, grads, accumulate=False, scratch=None):
    cons = m.consistency_classifier
    return m.hot_path.step(x, y, eps, kl_weight=m.kl_loss_weight, clf_weight=m.classifier_loss_weight, use_cos_loss=m.use_cos_loss,
                           compute_grads=True, grads=grads, want_outputs=True, consistency=cons, consistency_y=y if cons is not None else None,
                           consistency_weight=m.consitency_loss_weight, accumulate=accumulate, grad_scratch=scratch, grad_scope=scope)


def _close(a, b, tol):
    return bool(((a - b).abs() <= tol * b.abs() + 1e-7).all())


# ---- 1 + 2. the same numbers as the full step; only the classifier span of the buffer changes --------------------------------------
@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("mode", MODES)
def test_frozen_step_matches_the_full_step(name, mode):
    """Same inputs, injected eps: losses and classifier gradients bit-identical in the deterministic modes (fast mode: 1e-6 / 1e-5),
    x_hat / mu / log_sigma bit-identical (x_hat within 1e-6 in fast mode, where the full step's decoder epilogue also emits the bias
    gradient).  A seeded pattern R in the buffer: outside the classifier span it survives bit for bit, the writing step puts g in the span
    and the accumulating step R + g."""
    from tests.golden_util import rel_err

    G = _gu()
    cfg = _cfg(name)
    precision = "fp32" if mode == "fp32" else "bf16"
    det = mode != "bf16_fast"
    with _deterministic(1 if det else 0):
        m = G.module_from_cfg(cfg, precision)
        hot = m.hot_path
        a, b = hot.classifier_span()
        x, y, eps = _batch(cfg, 300, seed=43)
        full = torch.zeros(hot.arena.numel, device=DEV)
        l_full, _, o_full = _step(m, x, y, eps, "all", full)
        gen = torch.Generator(device=DEV).manual_seed(5)
        R = torch.randn(hot.arena.numel, device=DEV, generator=gen)
        buf = R.clone()
        l_clf, _, o_clf = _step(m, x, y, eps, "classifier", buf)
        scratch = torch.randn(hot.arena.numel, device=DEV, generator=gen)
        acc = R.clone()
        l_acc, _, _ = _step(m, x, y, eps, "classifier", acc, accumulate=True, scratch=scratch)
        torch.cuda.synchronize()
    outside = torch.ones(hot.arena.numel, dtype=torch.bool, device=DEV)
    outside[a:b] = False
    assert torch.equal(buf[outside], R[outside]) and torch.equal(acc[outside], R[outside])
    g_full, g_clf = full[a:b], buf[a:b]
    assert torch.equal(o_clf[1], o_full[1]) and torch.equal(o_clf[2], o_full[2])         # mu, log_sigma
    if det:
        assert torch.equal(l_clf, l_full) and torch.equal(l_acc, l_full)
        assert torch.equal(g_clf, g_full)
        assert torch.equal(acc[a:b], R[a:b] + g_full)
        assert torch.equal(o_clf[0], o_full[0])
    else:
        assert _close(l_clf, l_full, 1e-6) and _close(l_acc, l_full, 1e-6)
        assert rel_err(g_clf.cpu().numpy(), g_full.cpu().numpy()) <= 1e-5
        assert rel_err(acc[a:b].cpu().numpy(), (R[a:b] + g_full).cpu().numpy()) <= 1e-5
        assert rel_err(o_clf[0].cpu().numpy(), o_full[0].cpu().numpy()) <= 1e-6
    assert g_full.abs().sum() > 0


def test_classifier_scope_without_a_classifier_is_refused():
    from pseudo_speaker_vae_b200 import _lib as L

    G = _gu()
    cfg = _cfg("train_d192_noclf")
    m = G.module_from_cfg(cfg, "fp32")
    x, _, eps = _batch(cfg, 64, seed=1)
    hot = m.hot_path
    grads = torch.zeros(hot.arena.numel, device=DEV)
    losses = torch.empty(L.NUM_LOSSES, device=DEV)
    ws = hot._workspace(torch.device(DEV), 64, L.MODE_TRAIN)
    rc = L.lib().psvae_train_fwd_bwd_scoped(hot._dref, hot.arena.flat.data_ptr(), None, grads.data_ptr(), x.data_ptr(), L.X_F32, None,
                                            eps.data_ptr(), 0, 0, 0, 64, 1.0, 1.0, 0, 1, L.FP32, None, None, None, losses.data_ptr(),
                                            ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream, None, None, None, 0.0, None, 0,
                                            None, L.GRAD_CLASSIFIER)
    assert rc < 0


# ---- 3. training: freeze_vae against the full step with the VAE frozen ---------------------------------------------------------------
def _batches(cfg, n, rows=512, seed=70):
    return [_batch(cfg, rows, seed=seed + i) for i in range(n)]


def _trainer_run(cfg, precision, batches, force_all, **kw):
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    m = G.module_from_cfg(cfg, precision, freeze_vae=True)
    if force_all:
        m.hot_path.train_scope = lambda: "all"
    tr = P.DataParallelTrainer(m, local_only=True, **kw)
    for x, y, eps in batches:
        tr.train_step(x, y, eps)
    torch.cuda.synchronize()
    return m.hot_path.arena.flat.detach().clone(), tr.optimizer._m.clone(), tr.optimizer._v.clone()


def _lightning_run(cfg, precision, batches, force_all, k=1):
    G = _gu()
    m = G.module_from_cfg(cfg, precision, freeze_vae=True)
    if force_all:
        m.hot_path.train_scope = lambda: "all"
    opt = m.configure_optimizers()["optimizer"]
    for i, (x, y, eps) in enumerate(batches):
        loss = m.training_step((x, y), i, eps=eps)["loss"]
        (loss / k).backward()
        assert all(p.grad is None for p in m.model.parameters())
        if (i + 1) % k == 0:
            opt.step()
            opt.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    return m.hot_path.arena.flat.detach().clone(), opt._m.clone(), opt._v.clone()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("knobs", ["plain", "clip", "acc3"])
@pytest.mark.parametrize("path", ["trainer", "lightning"])
def test_frozen_training_matches_the_full_step(mode, knobs, path):
    from tests.golden_util import rel_err

    cfg = _cfg("train_d256_c2")
    precision = "fp32" if mode == "fp32" else "bf16"
    k = 3 if knobs == "acc3" else 1
    batches = _batches(cfg, 5 * k)
    kw = dict(gradient_clip_val=0.05) if knobs == "clip" else dict(accumulate_grad_batches=k)
    if path == "lightning" and knobs == "clip":
        pytest.skip("the Lightning-style loop has no clipping of its own (Lightning's Trainer does it)")
    start = _gu().module_from_cfg(cfg, precision).hot_path.arena.ensure().detach().clone()
    runs = []
    with _deterministic(0 if mode == "bf16_fast" else 1):
        for force_all in (True, False):
            if path == "trainer":
                runs.append(_trainer_run(cfg, precision, batches, force_all, **kw))
            else:
                runs.append(_lightning_run(cfg, precision, batches, force_all, k=k))
    a, b = _gu().module_from_cfg(cfg, precision).hot_path.classifier_span()
    (pf, mf, vf), (pc, mc, vc) = runs
    # the VAE and its Adam moments: untouched by both
    assert torch.equal(pc[:a], start[:a]) and torch.equal(pf[:a], start[:a])
    assert not mc[:a].any() and not vc[:a].any() and not mf[:a].any()
    assert not torch.equal(pc[a:b], start[a:b])
    if mode == "bf16_fast":
        assert rel_err(pc[a:b].cpu().numpy(), pf[a:b].cpu().numpy()) <= 1e-4
    else:
        assert torch.equal(pc, pf) and torch.equal(mc, mf) and torch.equal(vc, vf)


# ---- 4. fewer launches, no shadow refresh, no host synchronisation --------------------------------------------------------------------
@pytest.mark.parametrize("name,det", [("train_d256_c2", 0), ("train_d256_c2", 1), ("multilabel", 0), ("train_d512_c3_mlp", 1)])
def test_frozen_step_launches(name, det):
    from pseudo_speaker_vae_b200 import _lib as L

    G = _gu()
    cfg = _cfg(name)
    lib = L.lib()
    with _deterministic(det):
        m = G.module_from_cfg(cfg, "bf16")
        hot = m.hot_path
        x, y, eps = _batch(cfg, 4096, seed=3)
        grads = torch.zeros(hot.arena.numel, device=DEV)
        hot._shadow()

        def count(**kw):
            c0 = lib.psvae_launch_count()
            hot.step(x, y, eps, grads=grads if kw.get("compute_grads", True) else None, **kw)
            return lib.psvae_launch_count() - c0

        fwd = count(compute_grads=False)
        full = count(grad_scope="all")
        frozen = count(grad_scope="classifier")
    # the classifier's gradient kernels on top of the forward: none (the fused pass writes them), one (row-gradient kernel under the fused
    # encoder head), or the general chain of an MLP classifier (per Linear: GEMM + column sums + their reduce, plus the dgrad GEMMs)
    extra = {"train_d512_c3_mlp": 16}.get(name, 1)
    assert frozen <= fwd + extra and frozen < full


def test_frozen_eager_steps_keep_the_shadow_and_do_not_synchronise():
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    cfg = _cfg("train_d256_c2")
    m = G.module_from_cfg(cfg, "bf16", freeze_vae=True)
    tr = P.DataParallelTrainer(m, local_only=True, accumulate_grad_batches=2, gradient_clip_val=0.1)
    batches = [_batch(cfg, 512, seed=200 + i)[:2] for i in range(6)]
    for x, y in batches[:2]:
        tr.train_step(x, y)
    torch.cuda.synchronize()
    arena = m.hot_path.arena
    assert arena.shadow_current()
    shadow = arena.shadow.clone()
    refreshes = []
    real = arena.shadow_ptr

    def watch(desc_ref):
        if not arena.shadow_current():
            refreshes.append(1)
        return real(desc_ref)

    arena.shadow_ptr = watch
    torch.cuda.set_sync_debug_mode("error")
    try:
        for x, y in batches[2:]:
            tr.train_step(x, y)
    finally:
        torch.cuda.set_sync_debug_mode(0)
        del arena.shadow_ptr
    torch.cuda.synchronize()
    assert not refreshes and arena.shadow_current()
    a, _ = m.hot_path.classifier_span()
    assert torch.equal(arena.shadow[:a], shadow[:a])
    assert torch.equal(arena.shadow, arena.flat.to(torch.bfloat16))        # the classifier's slice was rewritten by Adam


# ---- 5. the graphed step --------------------------------------------------------------------------------------------------------------
def test_graphed_frozen_step_matches_eager_and_unfreezing_recaptures():
    """Deterministic mode: 10 frozen steps (a scheduler step after each, one eager step of another row count in the middle), then the VAE
    is unfrozen for 4 more: graphed and eager bit-identical throughout (parameters, Adam moments, losses)."""
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    cfg = _cfg("train_d256_c2")
    rows = 512
    calls = [_batch(cfg, rows, seed=300 + i)[:2] for i in range(14)]
    calls[6] = _batch(cfg, 256, seed=399)[:2]
    out = []
    with _deterministic(1):
        for graphed in (False, True):
            m = G.module_from_cfg(cfg, "bf16", freeze_vae=True)
            m.hot_path.manual_seed(77, 0)
            tr = P.DataParallelTrainer(m, local_only=True)
            sched = torch.optim.lr_scheduler.CosineAnnealingLR(tr.optimizer, T_max=5)
            step = P.GraphedTrainStep(tr, rows=rows) if graphed else tr.train_step
            losses, keys = [], []
            for i, (x, y) in enumerate(calls):
                if i == 10:
                    _freeze(m, False)
                losses.append(step(x, y).clone())
                sched.step()
                if graphed:
                    keys.append(step._key)
                if i == 9:
                    frozen_state = m.hot_path.arena.flat.detach().clone()
            torch.cuda.synchronize()
            out.append((frozen_state, m.hot_path.arena.flat.detach().clone(), tr.optimizer._m.clone(), torch.stack(losses)))
            if graphed:
                assert step.replays >= 11
                assert keys[9] is not None and keys[10] != keys[9]          # unfreezing re-captured
    for a, b in zip(out[0], out[1]):
        assert torch.equal(a, b)
    start = G.module_from_cfg(cfg, "bf16").hot_path.arena.ensure().detach()
    a = G.module_from_cfg(cfg, "bf16").hot_path.classifier_span()[0]
    assert torch.equal(out[1][0][:a], start[:a]) and not torch.equal(out[1][1][:a], start[:a])


def test_graph_still_refuses_other_partial_freezes():
    import pseudo_speaker_vae_b200 as P

    G = _gu()
    cfg = _cfg("train_d256_c2")
    m = G.module_from_cfg(cfg, "bf16")
    for p in m.classifier.parameters():
        p.requires_grad = False
    tr = P.DataParallelTrainer(m, local_only=True)
    step = P.GraphedTrainStep(tr, rows=256)
    x, y, _ = _batch(cfg, 256, seed=9)
    step(x, y)
    with pytest.raises(NotImplementedError, match="no frozen parameters"):
        step(x, y)


# ---- 6. two ranks -----------------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_frozen_vae_on_two_ranks():
    """2 ranks, frozen VAE, deterministic mode: ranks bit-identical and equal to the single-process frozen run."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29549",
           os.path.join(ROOT, "tests", "frozen_dp_case.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    lines = [l for l in res.stdout.splitlines() if l.startswith("RESULT ")]
    assert res.returncode == 0 and len(lines) == 2, res.stdout[-2000:] + res.stderr[-2000:]
    for l in lines:
        r = json.loads(l[len("RESULT "):])
        assert r["ranks_identical"] and r["vae_unchanged"] and r["param_rel_err"] <= 2e-6, r
