"""Per-row classifier targets and in-kernel target mixes on the GPU (-m gpu).

A row of a per-row call must be bit-identical to the shared-target call with that row's target (same seed, offset0, row0): z, the
history, stop_step and last_prob are compared with torch.equal for the thread-per-sample kernel, the generic kernel with an MLP
classifier, and the generic kernel forced on linear heads.  Against the fp64 reference (oracle/row_targets.py) the usual sampling
tolerances hold.  A target mix draws exactly what oracle/row_targets.draw_target_mix draws, at the frequencies of its weights, and
a sharded run draws what a single call draws."""
import itertools

import numpy as np
import pytest
import torch

from oracle import ps_vae_oracle as O
from oracle import row_targets as RT
from tests.golden_util import rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
FP32_TOL = 1e-5
BF16_FWD_TOL = 1e-2
HEADS = {"gender": 3, "age": 3}
# every target combination of the two heads, including rows that leave one head out
COMBOS = [c for c in itertools.product(range(-1, 3), range(-1, 3)) if c != (-1, -1)]


def _P():
    import pseudo_speaker_vae_b200 as P

    return P


def _model(kind, precision="fp32", seed=0):
    torch.manual_seed(seed)
    clf = dict(input_dim=64, num_classes=dict(HEADS))
    if kind == "mlp":
        clf.update(num_layers=2, hidden_dim=128)
    m = _P().PseudoSpeakerVAE(model=dict(input_dim=256, latent_dim=64), classifier=clf, optimizer={}, scheduler=dict(T_max=1), precision=precision)
    with torch.no_grad():                      # heads strong enough that p(y|z) crosses the threshold within a few steps for some rows
        for n, p in m.classifier.named_parameters():
            if "weight" in n:
                p.mul_(4.0)
    return m.to(DEV)


def _oracle_params(m):
    return {k: v.detach().double().cpu().numpy() for k, v in m.state_dict().items()}


def _dict_target(combo):
    return {name: t for name, t in zip(HEADS, combo) if t >= 0}


def _row_assignment(N, seed=1):
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(len(COMBOS), (N,), generator=g)
    idx[:len(COMBOS)] = torch.arange(len(COMBOS))          # every combination present
    tg = torch.tensor([COMBOS[i][0] for i in idx.tolist()])
    ta = torch.tensor([COMBOS[i][1] for i in idx.tolist()])
    return idx, {"gender": tg.to(DEV), "age": ta.to(DEV)}


class _generic:
    def __init__(self, on):
        self.on = on

    def __enter__(self):
        _P()._lib.set_option("langevin_generic", int(self.on))

    def __exit__(self, *a):
        _P()._lib.set_option("langevin_generic", 0)


def _run(hot, N, target, off, inject, steps, **kw):
    hot.offset = off
    return hot.langevin(N, target, 0.3, steps, 0.7, return_history=True, return_stop=True, threshold=0.6, row0=kw.pop("row0", 0), **inject, **kw)


CASES = [("fast", "lin", 0), ("mlp", "mlp", 0), ("generic", "lin", 1)]


@pytest.mark.parametrize("case,kind,generic", CASES)
@pytest.mark.parametrize("injected", [False, True])
def test_rows_bit_identical_to_shared_calls(case, kind, generic, injected):
    m = _model(kind)
    hot = m.hot_path
    hot.seed = 1234
    N, steps, L = 997, 6, 64
    inject = {}
    if injected:
        g = torch.Generator().manual_seed(5)
        inject = dict(z0=torch.randn(N, L, generator=g).to(DEV), noise=torch.randn(steps, N, L, generator=g).to(DEV))
    idx, target = _row_assignment(N)
    with _generic(generic):
        z, hist, (_, stop, prob) = _run(hot, N, target, 40, inject, steps, row0=3)
        assert hot.offset == 40 + steps + 1
        for k, combo in enumerate(COMBOS):
            rows = (idx == k).nonzero().flatten().to(DEV)
            zs, hs, (_, ss, ps) = _run(hot, N, _dict_target(combo), 40, inject, steps, row0=3)
            assert torch.equal(z[rows], zs[rows]), (case, combo)
            assert torch.equal(hist[:, rows], hs[:, rows]), (case, combo)
            assert torch.equal(stop[rows], ss[rows]) and torch.equal(prob[rows], ps[rows]), (case, combo)


@pytest.mark.parametrize("case,kind,generic", CASES)
def test_rows_against_the_oracle(case, kind, generic):
    P = _P()
    N, steps, L = 257, 5, 64
    g = torch.Generator().manual_seed(7)
    z0 = torch.randn(N, L, generator=g)
    noise = torch.randn(steps, N, L, generator=g)
    idx, target = _row_assignment(N, seed=2)
    per_row = [_dict_target(COMBOS[i]) for i in idx.tolist()]
    for precision, tol in (("fp32", FP32_TOL), ("bf16", BF16_FWD_TOL)):
        m = _model(kind, precision)
        params = _oracle_params(m)
        zr, hr = RT.langevin_rows(params, z0.double().numpy(), list(noise.double().numpy()), per_row, 0.05, 1.0, return_history=True)
        with _generic(generic):
            x_hat, hist = P.conditional_synthesis(m, N, target, 0.05, steps, 1.0, return_history=True, device=DEV, z0=z0.to(DEV),
                                                  noise=noise.to(DEV))
        assert rel_err(np.stack(hist), np.stack(hr)) <= FP32_TOL, (case, precision)        # the Langevin loop is fp32 in both modes
        assert rel_err(hist[-1], zr) <= FP32_TOL
        assert rel_err(x_hat.numpy(), O.decode(params, zr)) <= tol, (case, precision)


def test_latent_transformation_per_row_gender_flip():
    """The batched form of analysis/sample_gender_transformation.py: every speaker moves towards the opposite of its own gender."""
    P = _P()
    m = _model("lin")
    N = 300
    g = torch.Generator().manual_seed(3)
    x = torch.randn(N, 256, generator=g).to(DEV)
    src = torch.randint(2, (N,), generator=g).to(DEV)
    kw = dict(step_size=0.3, max_steps=40, noise_weight=0.0, prior_weight=0.5, threshold=0.9)
    for generic in (0, 1):
        with _generic(generic):
            xh, z, stop, prob = P.latent_transformation(m, x, {"gender": 1 - src}, **kw)
            for gender in (0, 1):
                rows = (src.cpu() == 1 - gender).nonzero().flatten()
                xs, zs, ss, ps = P.latent_transformation(m, x, {"gender": gender}, **kw)
                assert torch.equal(z[rows], zs[rows]) and torch.equal(stop[rows], ss[rows]) and torch.equal(prob[rows], ps[rows]), generic
                assert torch.equal(xh[rows], xs[rows])
    with pytest.raises(IndexError):
        P.latent_transformation(m, x, {"gender": src + 2}, **kw)


def _expected_targets(hot, entries, thr, N, off, steps, row0):
    k = RT.draw_target_mix(thr, N, hot.seed, off + steps + 1, row0)
    e = np.asarray(entries)[k]                    # [N, n_heads]
    return {name: torch.from_numpy(e[:, h]).to(torch.int64) for h, name in enumerate(HEADS)}


def test_mix_draw_matches_the_reference_and_its_weights():
    P = _P()
    m = _model("lin")
    hot = m.hot_path
    hot.seed = 99
    mix = [({"gender": 0, "age": 1}, 0.2), ({"gender": 2}, 0.0), ({"gender": 1, "age": 0}, 0.5), ({"age": 2}, 0.3)]
    entries, thr = hot.target_mix_for(mix)
    # N not a multiple of 4, odd row0
    N, steps = 1001, 3
    hot.offset = 10
    x, t = P.sample_on_device(m, N, num_steps=steps, target_mix=mix, row0=7)
    assert hot.offset == 10 + steps + 2 and x.is_cuda and t["gender"].is_cuda and t["gender"].dtype == torch.int64
    want = _expected_targets(hot, entries, thr, N, 10, steps, 7)
    assert all(torch.equal(t[k].cpu(), want[k]) for k in HEADS)
    # 2^20 rows: frequencies within 5 sigma of the weights; the zero-weight entry never appears
    N = 1 << 20
    hot.offset = 0
    _, t = P.sample_on_device(m, N, num_steps=1, target_mix=mix)
    codes = (t["gender"] + 1) * 4 + (t["age"] + 1)
    for (target, w), code in zip(mix, [1 * 4 + 2, 3 * 4 + 0, 2 * 4 + 1, 0 * 4 + 3]):
        n = int((codes == code).sum())
        sd = (N * w * (1 - w)) ** 0.5
        assert abs(n - N * w) <= 5 * sd, (target, w, n)
    assert int((codes == 3 * 4 + 0).sum()) == 0


def test_mix_single_label_and_conditional_synthesis_form():
    P = _P()
    torch.manual_seed(0)
    m = P.PseudoSpeakerVAE(model=dict(input_dim=256, latent_dim=64), classifier=dict(input_dim=64, num_classes=3), optimizer={},
                           scheduler=dict(T_max=1)).to(DEV)
    hot = m.hot_path
    hot.seed, hot.offset = 5, 0
    x, hist, t = P.conditional_synthesis(m, 101, num_steps=2, return_history=True, device=DEV, target_mix=[(0, 1), (2, 3)])
    assert x.shape == (101, 256) and len(hist) == 2 and t.dtype == torch.int64 and t.device.type == "cpu"
    k = RT.draw_target_mix([2 ** 30], 101, 5, 3, 0)
    assert torch.equal(t, torch.from_numpy(np.array([0, 2])[k]))
    # the drawn rows are the shared-target rows
    z_mix, _, _, t2 = hot.langevin(101, None, 0.01, 2, 1.0, row0=0, target_mix=[(0, 1), (2, 3)])
    for c in (0, 2):
        hot.offset = 4
        zc, _, _ = hot.langevin(101, c, 0.01, 2, 1.0)
        rows = (t2 == c).nonzero().flatten()
        assert torch.equal(z_mix[rows], zc[rows])
    with pytest.raises(ValueError):
        P.conditional_synthesis(m, 8, 1, device=DEV, target_mix=[(0, 1)])


@pytest.mark.parametrize("kind", ["lin", "mlp"])
def test_mix_sharding_reproduces_the_single_call(kind):
    P = _P()
    m = _model(kind)
    hot = m.hot_path
    hot.seed = 2024
    mix = [({"gender": 0}, 1.0), ({"gender": 1, "age": 2}, 2.0), ({"age": 0}, 1.5)]
    N, steps = 1237, 4
    hot.offset = 50
    z_full, _, _, t_full = hot.langevin(N, None, 0.05, steps, 1.0, row0=0, target_mix=mix)
    hot.offset = 50
    x_full, tx_full = P.sample_on_device(m, N, step_size=0.05, num_steps=steps, target_mix=mix)
    assert all(torch.equal(t_full[k], tx_full[k]) for k in HEADS)
    for world in (1, 2, 3, 8):
        zs, xs, ts = [], [], []
        for r in range(world):
            row0, rows = P.shard_rows(N, r, world)
            hot.offset = 50
            z, _, _, t = hot.langevin(rows, None, 0.05, steps, 1.0, row0=row0, target_mix=mix)
            hot.offset = 50
            x, _ = P.sample_on_device(m, rows, step_size=0.05, num_steps=steps, target_mix=mix, row0=row0)
            zs.append(z), xs.append(x), ts.append(t)
        assert torch.equal(torch.cat(zs), z_full) and torch.equal(torch.cat(xs), x_full), (kind, world)
        assert all(torch.equal(torch.cat([t[k] for t in ts]), t_full[k]) for k in HEADS), (kind, world)


@pytest.mark.parametrize("case,kind,generic", CASES)
def test_bad_device_target_gives_a_nan_row_only(case, kind, generic):
    m = _model(kind)
    hot = m.hot_path
    hot.seed = 77
    N, steps = 300, 4
    idx, target = _row_assignment(N, seed=4)
    bad = {"gender": target["gender"].clone(), "age": target["age"].clone()}
    bad["gender"][17] = 3                     # out of range
    bad["age"][200] = -7                      # below -1
    bad["gender"][250] = -1
    bad["age"][250] = -1                      # names no head
    with _generic(generic):
        z, hist, (_, stop, prob) = _run(hot, N, target, 0, {}, steps)
        zb, hb, (_, sb, pb) = _run(hot, N, bad, 0, {}, steps)
    badrows = [17, 200, 250]
    keep = torch.ones(N, dtype=torch.bool, device=DEV)
    keep[badrows] = False
    assert torch.equal(zb[keep], z[keep]) and torch.equal(hb[:, keep], hist[:, keep])
    assert torch.equal(sb[keep], stop[keep]) and torch.equal(pb[keep], prob[keep])
    for r in badrows:
        assert torch.isnan(zb[r]).all() and torch.isnan(hb[:, r]).all() and torch.isnan(pb[r]), (case, r)
    with pytest.raises(IndexError):
        _P().conditional_synthesis(m, N, bad, num_steps=1, device=DEV)


def test_mix_offsets():
    m = _model("lin")
    hot = m.hot_path
    hot.seed = 3
    mix = [({"gender": 0}, 1.0), ({"gender": 1}, 1.0), ({"gender": 2}, 1.0)]
    entries, thr = hot.target_mix_for(mix)
    N, steps = 4099, 5
    hot.offset = 0
    _, _, _, t1 = hot.langevin(N, None, 0.01, steps, 1.0, target_mix=mix)
    assert hot.offset == steps + 2
    _, _, _, t2 = hot.langevin(N, None, 0.01, steps, 1.0, target_mix=mix)
    assert hot.offset == 2 * (steps + 2)
    for t, off in ((t1, 0), (t2, steps + 2)):
        want = _expected_targets(hot, entries, thr, N, off, steps, 0)
        assert torch.equal(t["gender"].cpu(), want["gender"])
    assert not torch.equal(t1["gender"], t2["gender"])
    # an eager shared-target call after a mix call starts at offset + num_steps + 2
    hot.offset = 0
    hot.langevin(N, None, 0.01, steps, 1.0, target_mix=mix)
    z_after, _, _ = hot.langevin(N, {"gender": 1}, 0.01, steps, 1.0)
    hot.offset = steps + 2
    z_ref, _, _ = hot.langevin(N, {"gender": 1}, 0.01, steps, 1.0)
    assert torch.equal(z_after, z_ref)
