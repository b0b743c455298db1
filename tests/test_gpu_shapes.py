"""Shape-matrix parity tests (-m gpu): model shapes off the L = 64 / 2 x 512 path, each routed by the host code to a different kernel
(latent widths 4..256, 1 to 7 hidden layers, hidden widths that tile by 64 / 128 / 256 columns, ragged output tiles, linear heads with
and without the fused classifier pass, MLP trunks), against

  * the fp64 oracle (oracle/ps_vae_oracle.py) in fp32 mode: forward and losses at FP32_TOL, gradients at FP32_FLIP_TOL from 1000 rows
    (FP32_TOL below that), and the classifier and last-layer gradients -- the tensors the shape-specific kernels write -- at FP32_TOL;
  * the bf16-emulating twin (oracle/bf16_twin.py) in tensor-core mode, in fast and deterministic mode, at BF16_TWIN_TOL,
    BF16_TWIN_FWD_TOL and BF16_TWIN_LOSS_TOL.

Each case names the kernels it exists for; one step per case runs under torch.profiler (CUDA activity tracing only) and asserts that
those kernels ran and their alternatives did not, so that a later change of the dispatch cannot silently move a case off its route.
Decode (given z, the in-kernel Philox draw, the row-chunk loop and its ragged tail, sharding by row0) and the Langevin loops (fast
thread-per-sample kernel and generic tile kernel, conditional synthesis and latent transformation) are covered on the same shapes.
"""
import contextlib
import functools
import re

import numpy as np
import pytest
import torch

from oracle import bf16_twin as T
from oracle import philox_ref as PR
from oracle import ps_vae_oracle as O
from tests.golden_util import rel_err

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
FP32_FLIP_TOL = 2e-3        # B >= 1000, fp32: one flipped ReLU unit out of B rows (tests/test_gpu_parity.py)
BF16_TWIN_TOL = 1e-3        # gradients against the bf16 twin (tests/test_gpu_round2.py)
BF16_TWIN_LOSS_TOL = 2e-5
BF16_TWIN_FWD_TOL = 2e-4
TOUCHED_OPTIONS = ("deterministic", "clf_grad_in_bwd", "decode_chunk", "langevin_generic")


def _gu():
    from tests import gpu_util

    return gpu_util


@pytest.fixture(scope="module", autouse=True)
def _restore_options():
    """Every option a test here changes is put back to what it was before the module ran."""
    L = _gu().L
    saved = {k: L.get_option(k) for k in TOUCHED_OPTIONS}
    yield
    for k, v in saved.items():
        L.set_option(k, v)


@contextlib.contextmanager
def _options(**kw):
    L = _gu().L
    prev = {k: L.get_option(k) for k in kw}
    try:
        for k, v in kw.items():
            L.set_option(k, v)
        yield
    finally:
        for k, v in prev.items():
            L.set_option(k, v)


# ------------------------------------------------------------------------------------------------
# the shapes and the kernels each one exists for
# ------------------------------------------------------------------------------------------------
def _clf(nc, layers=1, hidden=128, act="relu"):
    return dict(num_classes=nc, num_layers=layers, hidden_dim=hidden, activation=act)


# The route entries name kernels (the function name, without namespace or template arguments) that must run in one step of the mode:
#   fp32       fp32 mode (sgemm engine; never a tcgen05 kernel)
#   bf16       tensor-core mode, default (fast) options
#   bf16_det   tensor-core mode, deterministic = 1
#   bf16_cgib  tensor-core mode, clf_grad_in_bwd = 1 (only where that changes the route)
# "EpiLatent": a gemm_tc_kernel with the fused encoder-head epilogue; "multi>1": more than one merged-wgrad launch (gemm_tc_multi_kernel),
# i.e. the ping-pong flushes in the middle of the backward pass.  The alternatives of a named kernel (the other latent backward kernels,
# fused vs unfused classifier, the fused head) must be absent.
CS, GEN, CLF8, CLFK = "latent_bwd_cs_kernel", "latent_bwd_kernel", "latent_bwd_clf8_kernel", "latent_bwd_clf_kernel"
FUSED, UNFUSED = "clf_fused_kernel", "ce_kernel"
TRAIN_CASES = {
    # sgemm everywhere; latent_bwd_cs at L = 4 (one quad per row); the unfused classifier with N = 2, K = 4
    # grad_tol: at B = 1000 one layer-0 pre-activation of encoder_sigma is 2.7e-8 in fp64 and takes the other sign in fp32 (a ReLU flip):
    # measured 2.8e-3 on model.encoder_sigma.0.weight, every other tensor <= 1.8e-4
    "l4_fp32": dict(D=100, L=4, H=100, nh=2, clf=_clf(2), prec=("fp32",), routes=dict(fp32=(CS, UNFUSED)), grad_tol=dict(fp32=4e-3)),
    # generic latent_bwd_kernel (3 quads per row); one hidden layer; two heads on the unfused classifier
    "l12_fp32": dict(D=68, L=12, H=36, nh=1, clf=_clf({"a": 3, "b": 2}), prec=("fp32",), routes=dict(fp32=(GEN, UNFUSED))),
    # the reference's own smoke shape (VAEModel(784, 20)), with the backward pass and a 2 x 96 tanh trunk
    "l20_fp32": dict(D=784, L=20, H=512, nh=2, clf=_clf(2, 3, 96, "tanh"), prec=("fp32",), routes=dict(fp32=(GEN, UNFUSED))),
    # per-encoder head GEMMs with N = 8 and dgrad K = 8; unfused classifier; latent_bwd_cs
    "l8": dict(D=64, L=8, H=64, nh=2, clf=_clf(3), prec=("fp32", "bf16"),
               routes=dict(fp32=(CS, UNFUSED), bf16=(CS, UNFUSED), bf16_det=(CS, UNFUSED))),
    # clf_fused_kernel<16>; no hidden-to-hidden layer; BN = 64 tiles (H = 192)
    "l16_nh1": dict(D=128, L=16, H=192, nh=1, clf=_clf(2), prec=("fp32", "bf16"),
                    routes=dict(fp32=(FUSED, CS), bf16=(FUSED, CS), bf16_det=(FUSED, CS), bf16_cgib=(FUSED, CLF8))),
    # generic latent_bwd_kernel (6 quads per row); D = 200: ragged last N tile; three hidden layers: merged-wgrad flushes before a
    # ping-pong gradient buffer is overwritten
    # grad_tol: four ReLU layers deep, an activation one bf16 ulp from the twin's (fp32 vs fp64 accumulation on a rounding boundary) can flip
    # a ReLU unit of the next layer, which moves a layer-0 weight gradient by one row's contribution: measured 3.0e-3 on
    # model.encoder_sigma.0.weight at B = 77 (no layer-0 pre-activation is within fp32 accumulation error of 0 there), 1.9e-3 on
    # model.decoder.0.weight at B = 1000, 7.6e-4 at B = 8269; the same in fast and deterministic mode
    "l24_nh3": dict(D=200, L=24, H=320, nh=3, clf=_clf(2), prec=("fp32", "bf16"), big=True, grad_tol=dict(bf16=5e-3),
                    routes=dict(fp32=(GEN, UNFUSED), bf16=(GEN, UNFUSED, "multi>1"), bf16_det=(GEN, UNFUSED))),
    # clf_fused_kernel<32> with 5 classes over two heads (not latent8_ok); BN = 128 tiles (H = 384)
    "l32_mh": dict(D=256, L=32, H=384, nh=2, clf=_clf({"age": 3, "gender": 2}), prec=("fp32", "bf16"),
                   routes=dict(fp32=(FUSED, CS), bf16=(FUSED, CS), bf16_det=(FUSED, CS), bf16_cgib=(FUSED, CLFK))),
    # clf_fused_kernel<128> at the total x L = 512 boundary; latent8_ok with clf_grad_in_bwd = 1
    "l128_c4": dict(D=512, L=128, H=256, nh=2, clf=_clf(4), prec=("fp32", "bf16"), big=True,
                    routes=dict(fp32=(FUSED, CS), bf16=(FUSED, CS), bf16_det=(FUSED, CS), bf16_cgib=(FUSED, CLF8))),
    # just past the boundary (5 x 128 > 512): the unfused classifier at L = 128
    "l128_c5": dict(D=256, L=128, H=256, nh=2, clf=_clf(5), prec=("fp32", "bf16"),
                    routes=dict(fp32=(UNFUSED, CS), bf16=(UNFUSED, CS), bf16_det=(UNFUSED, CS))),
    # latent_cs_ok is false (2 L > 256): generic backward, head bias gradients from colsum; grouped head launch with L = 256
    # grad_tol: at B = 1000 three layer-0 pre-activations of encoder_mu lie within fp32 accumulation error of 0 (ReLU flips against the
    # twin's fp64 sums): measured 1.07e-3 on model.encoder_mu.0.weight, <= 3.1e-4 elsewhere, in fast and deterministic mode
    "l256": dict(D=256, L=256, H=512, nh=2, clf=None, prec=("fp32", "bf16"), routes=dict(fp32=(GEN,), bf16=(GEN,), bf16_det=(GEN,)),
                 grad_tol=dict(bf16=2e-3)),
    "l256_c2": dict(D=256, L=256, H=512, nh=2, clf=_clf(2), prec=("fp32", "bf16"),
                    routes=dict(fp32=(GEN, UNFUSED), bf16=(GEN, UNFUSED), bf16_det=(GEN, UNFUSED))),
    # the fused encoder head with the deepest model PSVAE_MAX_LAYERS allows; many merged-wgrad flushes
    # grad_tol: eight Linear layers per MLP: the twin's error grows smoothly with depth (measured at B = 1000 from 1e-5 on the last encoder
    # layers to 8e-5 on layer 1 and 4.4e-3 on model.encoder_mu.0.weight; 1.4e-3 at B = 8269; the same in fast and deterministic mode), the
    # bf16 rounding-boundary flips of l24_nh3 compounded
    "l64_nh7": dict(D=256, L=64, H=128, nh=7, clf=_clf(2), prec=("fp32", "bf16"), big=True, grad_tol=dict(bf16=5e-3),
                    routes=dict(fp32=(FUSED, CS), bf16=("EpiLatent", CLF8, "multi>1"), bf16_det=(FUSED, CS))),
    # the fused encoder head with H % 128 != 0
    "l64_h192": dict(D=192, L=64, H=192, nh=2, clf=_clf(3), prec=("fp32", "bf16"),
                     routes=dict(fp32=(FUSED, CS), bf16=("EpiLatent", CLF8), bf16_det=(FUSED, CS))),
}
LATENT_KERNELS = (CS, GEN, CLF8, CLFK)
CLF_KERNELS = (FUSED, UNFUSED)
CGIB_CASES = ("l16_nh1", "l32_mh", "l128_c4")
BIG_B = 8192 + 77


def _cfg(cid, **over):
    c = dict(TRAIN_CASES.get(cid, {}), **over)
    cfg = dict(D=c["D"], L=c["L"], H=c["H"], nh=c["nh"], wseed=c.get("wseed", 17))
    if c.get("clf"):
        cfg["clf"] = dict(c["clf"], input_dim=c["L"])
    return cfg


def _params(cfg):
    shapes = O.vae_param_shapes(cfg["D"], cfg["L"], cfg["H"], cfg["nh"])
    if cfg.get("clf"):
        c = cfg["clf"]
        shapes += O.classifier_param_shapes(cfg["L"], c["num_classes"], c["num_layers"], c["hidden_dim"])
    return {k: v.astype(np.float32) for k, v in O.synth_params(shapes, seed=cfg["wseed"], dtype=np.float64).items()}


def _act(cfg):
    return cfg["clf"]["activation"] if cfg.get("clf") else "relu"


@functools.lru_cache(maxsize=None)
def _batch(cid, B):
    cfg = _cfg(cid)
    nc = cfg["clf"]["num_classes"] if cfg.get("clf") else 2
    return O.synth_batch(B, cfg["D"], cfg["L"], nc, seed=1000 + B)


@functools.lru_cache(maxsize=None)
def _reference(cid, B, precision):
    """(scalars, outputs, grads) of the fp64 oracle (fp32 mode) or of the bf16 twin (tensor-core mode) on the case's batch."""
    cfg = _cfg(cid)
    p = _params(cfg)
    x, y, eps = _batch(cid, B)
    if precision == "fp32":
        return O.train_loss_and_grads({k: v.astype(np.float64) for k, v in p.items()}, x.astype(np.float64), y, eps.astype(np.float64),
                                      classifier_activation=_act(cfg))
    return T.train_loss_and_grads_bf16(p, x, y, eps, classifier_activation=_act(cfg))


# ------------------------------------------------------------------------------------------------
# kernel routes from torch.profiler
# ------------------------------------------------------------------------------------------------
def _kernel_counts(fn):
    """{kernel full name: launches} of the CUDA kernels ``fn`` ran (CUDA activity tracing only)."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and not ev.key.startswith(("Memcpy", "Memset")):
            out[ev.key] = out.get(ev.key, 0) + ev.count
    assert out, "torch.profiler recorded no CUDA kernel events on this machine: the kernel routes cannot be checked"
    return out


def _base(name):
    s = name[5:] if name.startswith("void ") else name
    m = re.match(r"[\w:]+", s)
    return m.group(0).split("::")[-1] if m else s


def _check_routes(tag, counts, want, precision):
    bases = {}
    for k, n in counts.items():
        bases[_base(k)] = bases.get(_base(k), 0) + n
    epi_latent = any(_base(k) == "gemm_tc_kernel" and "EpiLatent" in k for k in counts)
    got = sorted(bases)
    for w in want:
        if w == "EpiLatent":
            assert epi_latent, (tag, "no gemm_tc_kernel<EpiLatent>", got)
        elif w == "multi>1":
            assert bases.get("gemm_tc_multi_kernel", 0) > 1, (tag, "expected more than one merged-wgrad launch", bases.get("gemm_tc_multi_kernel", 0))
        else:
            assert w in bases, (tag, f"{w} did not run", got)
    for group in (LATENT_KERNELS, CLF_KERNELS):
        named = [w for w in want if w in group]
        for alt in group:
            if named and alt not in named:
                assert alt not in bases, (tag, f"{alt} ran instead of {named}", got)
    if "EpiLatent" not in want:
        assert not epi_latent, (tag, "the fused encoder head ran", got)
    else:       # the fused head computes the classifier forward itself
        assert not any(k in bases for k in CLF_KERNELS), (tag, got)
    if precision == "fp32":
        assert "sgemm_kernel" in bases and not any(b.startswith("gemm_tc") for b in bases), (tag, got)
    print(f"route {tag}: {', '.join(w for w in want)} -- ran {got}")


# ------------------------------------------------------------------------------------------------
# train step: losses, outputs and every gradient tensor
# ------------------------------------------------------------------------------------------------
def _modes(cid, precision):
    if precision == "fp32":
        return [("fp32", {})]
    modes = [("bf16", dict(deterministic=0, clf_grad_in_bwd=0)), ("bf16_det", dict(deterministic=1, clf_grad_in_bwd=0))]
    if cid in CGIB_CASES:
        modes.append(("bf16_cgib", dict(deterministic=0, clf_grad_in_bwd=1)))
    return modes


def _last_layer(k, nh):
    return f".{2 * nh}." in k and k.startswith("model.")


TRAIN_PARAMS = [(cid, p) for cid, c in TRAIN_CASES.items() for p in c["prec"]]


@pytest.mark.parametrize("cid,precision", TRAIN_PARAMS, ids=[f"{c}-{p}" for c, p in TRAIN_PARAMS])
def test_train_step_shape_matrix(cid, precision):
    G = _gu()
    case = TRAIN_CASES[cid]
    cfg = _cfg(cid)
    params = _params(cfg)
    has_clf = bool(cfg.get("clf"))
    failures = []
    batches = (77, 1000) + ((BIG_B,) if case.get("big") else ())
    for mode, opts in _modes(cid, precision):
        with _options(**opts):
            module = G.module_from_cfg(cfg, precision, params=params)
            hot = module.hot_path
            for i, B in enumerate(batches):
                x, y, eps = _batch(cid, B)
                scal, out, grads = _reference(cid, B, precision)
                xt, et = torch.from_numpy(x).to(G.DEV), torch.from_numpy(eps).to(G.DEV)
                yt = G.labels_to_torch(y) if has_clf else None
                g = torch.empty(hot.arena.numel, device=G.DEV)
                res = {}

                def run():
                    res["r"] = hot.step(xt, yt, et, grads=g, want_outputs=True)

                if i == 0:
                    _check_routes(f"{cid} {mode}", _kernel_counts(run), case["routes"][mode], precision)
                else:
                    run()
                losses, _, outs = res["r"]
                torch.cuda.synchronize()
                lt = losses.cpu().numpy()
                gd = G.flat_to_dict(module, g)
                errs = {k: rel_err(gd[k], grads[k]) for k in grads}
                ferrs = {k: rel_err(t.cpu().numpy(), out[k]) for t, k in zip(outs, ("x_hat", "mu", "log_sigma"))}
                slots = ((0, "loss"), (1, "recon_loss"), (2, "kl_loss")) + (((3, "classifier_loss"),) if has_clf else ())
                lerrs = {k: abs(float(lt[s]) - float(scal[k])) / max(1.0, abs(float(scal[k]))) for s, k in slots}
                clf_last = {k: v for k, v in errs.items() if k.startswith("classifier.") or _last_layer(k, cfg["nh"])}
                if precision == "fp32":
                    tf, tl, tg = FP32_TOL, FP32_TOL, (FP32_FLIP_TOL if B >= 1000 else FP32_TOL)
                else:
                    tf, tl, tg = BF16_TWIN_FWD_TOL, BF16_TWIN_LOSS_TOL, BF16_TWIN_TOL
                tg = max(tg, case.get("grad_tol", {}).get(precision, 0.0))
                worst = max(errs, key=errs.get)
                print(f"shape {cid} {mode} B={B}: fwd {max(ferrs.values()):.1e} loss {max(lerrs.values()):.1e} grad {errs[worst]:.1e} ({worst})"
                      f" clf+last {max(clf_last.values()):.1e}")
                report = (cid, mode, B, {k: f"{v:.1e}" for k, v in ferrs.items()}, {k: f"{v:.1e}" for k, v in lerrs.items()},
                          {k: f"{v:.1e}" for k, v in errs.items()})
                # every batch and mode runs before the verdict, so that one run reports all the measured values
                if not (all(v <= tl for v in lerrs.values()) and all(v <= tf for v in ferrs.values()) and max(errs.values()) <= tg
                        and (precision != "fp32" or all(v <= FP32_TOL for v in clf_last.values()))):
                    failures.append(report)
    assert not failures, failures


# ------------------------------------------------------------------------------------------------
# classifier-only scope (freeze_vae): the classifier's gradients, and nothing else in the buffer changes
# ------------------------------------------------------------------------------------------------
SCOPE_PARAMS = [(cid, p) for cid in ("l8", "l16_nh1", "l128_c4", "l128_c5") for p in ("fp32", "bf16")]


@pytest.mark.parametrize("cid,precision", SCOPE_PARAMS, ids=[f"{c}-{p}" for c, p in SCOPE_PARAMS])
def test_classifier_scope_shape_matrix(cid, precision):
    G = _gu()
    cfg = _cfg(cid)
    module = G.module_from_cfg(cfg, precision, params=_params(cfg))
    hot = module.hot_path
    B = 1000
    x, y, eps = _batch(cid, B)
    _, _, grads = _reference(cid, B, precision)
    a, b = hot.classifier_span()
    gen = torch.Generator(device=G.DEV).manual_seed(3)
    R = torch.randn(hot.arena.numel, device=G.DEV, generator=gen)
    buf = R.clone()
    hot.step(torch.from_numpy(x).to(G.DEV), G.labels_to_torch(y), torch.from_numpy(eps).to(G.DEV), grads=buf, grad_scope="classifier")
    torch.cuda.synchronize()
    outside = torch.ones(hot.arena.numel, dtype=torch.bool, device=G.DEV)
    outside[a:b] = False
    assert torch.equal(buf[outside], R[outside]), (cid, precision, "the classifier scope wrote outside the classifier span")
    gd = G.flat_to_dict(module, buf)
    errs = {k: rel_err(gd[k], grads[k]) for k in grads if k.startswith("classifier.")}
    print(f"classifier scope {cid} {precision}: worst classifier gradient {max(errs.values()):.1e}")
    assert max(errs.values()) <= (FP32_TOL if precision == "fp32" else BF16_TWIN_TOL), (cid, precision, {k: f"{v:.1e}" for k, v in errs.items()})


# ------------------------------------------------------------------------------------------------
# decode: given z, the Philox draw, the row-chunk loop (ragged tail) and sharding by row0
# ------------------------------------------------------------------------------------------------
DECODE_MODELS = {cid: dict(D=c["D"], L=c["L"], H=c["H"], nh=c["nh"], prec=c["prec"]) for cid, c in TRAIN_CASES.items() if cid != "l256_c2"}
DECODE_MODELS.update({
    "d272": dict(D=272, L=64, H=512, nh=2, prec=("fp32", "bf16")),      # D > 256: not chain-eligible
    "h640": dict(D=256, L=64, H=640, nh=2, prec=("fp32", "bf16")),      # H > 512: not chain-eligible
    "chain": dict(D=192, L=64, H=256, nh=2, prec=("fp32", "bf16")),     # decoder_chain_kernel in bf16
})
DECODE_PARAMS = [(cid, p) for cid, c in DECODE_MODELS.items() for p in c["prec"]]


def _chain_ok(c):
    """decoder_chain_ok (csrc/decoder_chain.cuh): two hidden layers of 128..512 (a multiple of 128), latent 64, D % 16 == 0, D <= 256."""
    return c["nh"] == 2 and c["L"] == 64 and c["H"] % 128 == 0 and 128 <= c["H"] <= 512 and c["D"] % 16 == 0 and c["D"] <= 256


@pytest.mark.parametrize("cid,precision", DECODE_PARAMS, ids=[f"{c}-{p}" for c, p in DECODE_PARAMS])
def test_decode_shape_matrix(cid, precision):
    G = _gu()
    c = DECODE_MODELS[cid]
    cfg = dict(D=c["D"], L=c["L"], H=c["H"], nh=c["nh"], wseed=23)
    params = _params(cfg)
    p64 = {k: v.astype(np.float64) for k, v in params.items()}
    module = G.module_from_cfg(cfg, precision, params=params)
    hot = module.hot_path
    chained = precision == "bf16" and _chain_ok(c)

    def want(z):
        if precision == "fp32":
            return O.decode(p64, z.astype(np.float64)), FP32_TOL
        return T._mlp_fwd(p64, "model.decoder", T.bf16_round(z))[0], BF16_TWIN_FWD_TOL

    z = np.random.default_rng(5).standard_normal((1000, c["L"])).astype(np.float32)
    counts = _kernel_counts(lambda: hot.decode(torch.from_numpy(z).to(G.DEV)))
    ran = {_base(k) for k in counts}
    assert ("decoder_chain_kernel" in ran) == chained, (cid, precision, sorted(ran))
    xz = hot.decode(torch.from_numpy(z).to(G.DEV)).cpu().numpy()
    ref, tol = want(z)
    errs = {"given z": rel_err(xz, ref)}
    if not chained:
        N = 2531
        with _options(decode_chunk=1000):          # chunks of 1000, 1000 and 531 rows
            z2 = np.random.default_rng(6).standard_normal((N, c["L"])).astype(np.float32)
            x2 = hot.decode(torch.from_numpy(z2).to(G.DEV)).cpu().numpy()
            ref2, _ = want(z2)
            errs["chunked z"] = rel_err(x2, ref2)
            errs["chunked z, last row"] = rel_err(x2[-1:], ref2[-1:])
            hot.manual_seed(11, 0)
            xd, zd = hot.decode(None, num_samples=N, return_z=True)
            zd = zd.cpu().numpy()
            zerr = np.abs(zd - PR.philox_normal(N, c["L"], 11, 0, 0))        # as test_unconditional_synthesis_distribution_and_api
            assert zerr.mean() < 4e-7 and np.quantile(zerr, 0.999) < 3e-6 and zerr.max() < 3e-4, (cid, precision, zerr.max())
            refd, _ = want(zd)
            errs["philox z"] = rel_err(xd.cpu().numpy(), refd)
            hot.manual_seed(11, 0)
            full = hot.decode(None, num_samples=N)
            parts = []
            for r0, r1 in ((0, 1200), (1200, 1201), (1201, N)):
                hot.manual_seed(11, 0)
                parts.append(hot.decode(None, num_samples=r1 - r0, row0=r0))
            assert torch.equal(torch.cat(parts), full), (cid, precision, "row0 shards differ from the single call")
    print(f"decode {cid} {precision}{' (chained)' if chained else ''}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert all(v <= tol for v in errs.values()), (cid, precision, errs)


# ------------------------------------------------------------------------------------------------
# Langevin: conditional synthesis and latent transformation, fast and generic kernel
# ------------------------------------------------------------------------------------------------
LANGEVIN_CASES = {
    # fast path (thread per sample): no trunk, L in {16, 32, 64}, <= 8 targeted classes
    "l16_c2": dict(L=16, clf=_clf(2), target=1, fast=True, thr=0.66),
    "l16_c332": dict(L=16, clf=_clf({"a": 3, "b": 3, "c": 2}), target={"a": 2, "b": 0, "c": 1}, fast=True, thr=0.13),
    "l32_c2": dict(L=32, clf=_clf(2), target=0, fast=True, thr=0.56),
    "l32_c332": dict(L=32, clf=_clf({"a": 3, "b": 3, "c": 2}), target={"a": 1, "b": 2, "c": 0}, fast=True, thr=0.1),
    # generic tile kernel
    "l12_c2": dict(L=12, clf=_clf(2), target=1, fast=False, thr=0.65),
    "l24_c2": dict(L=24, clf=_clf(2), target=1, fast=False, thr=0.59),
    "l128_c2": dict(L=128, clf=_clf(2), target=0, fast=False, thr=0.63),
    "l32_c54": dict(L=32, clf=_clf({"a": 5, "b": 4}), target={"a": 3, "b": 1}, fast=False, thr=0.07),        # 9 targeted classes
    "l16_trunk": dict(L=16, clf=_clf(3, 3, 64, "tanh"), target=2, fast=False, thr=0.3),                     # a 2-layer tanh trunk
}


def _langevin_model(lid):
    G = _gu()
    c = LANGEVIN_CASES[lid]
    cfg = dict(D=64, L=c["L"], H=64, nh=2, wseed=29, clf=dict(c["clf"], input_dim=c["L"]))
    params = _params(cfg)
    return G.module_from_cfg(cfg, "fp32", params=params), {k: v.astype(np.float64) for k, v in params.items()}, cfg, c


@pytest.mark.parametrize("lid", list(LANGEVIN_CASES))
def test_conditional_synthesis_shape_matrix(lid):
    G = _gu()
    import pseudo_speaker_vae_b200 as P

    module, p64, cfg, c = _langevin_model(lid)
    N, steps, step_size, nw = 300, 6, 0.5, 0.7
    rng = np.random.default_rng(8)
    z0 = rng.standard_normal((N, c["L"])).astype(np.float32)
    noises = rng.standard_normal((steps, N, c["L"])).astype(np.float32)
    z0t, nt = torch.from_numpy(z0).to(G.DEV), torch.from_numpy(noises).to(G.DEV)
    res = {}
    counts = _kernel_counts(lambda: res.setdefault("r", P.conditional_synthesis(module, N, c["target"], step_size, steps, nw, True, G.DEV,
                                                                                 z0=z0t, noise=nt)))
    ran = {_base(k) for k in counts}
    want, alt = ("langevin_fast_kernel", "langevin_kernel") if c["fast"] else ("langevin_kernel", "langevin_fast_kernel")
    assert want in ran and alt not in ran, (lid, sorted(ran))
    xc, hist = res["r"]
    xr, hr = O.conditional_synthesis(p64, z0.astype(np.float64), list(noises.astype(np.float64)), c["target"], step_size, nw,
                                     activation=_act(cfg), return_history=True)
    e_hist, e_x = rel_err(np.stack(hist), np.stack(hr)), rel_err(xc.numpy(), xr)
    msg = f"langevin {lid} ({want}): history {e_hist:.1e} x_hat {e_x:.1e}"
    if c["fast"]:
        # the generic kernel on the same Philox counters (no injected draws): within 2e-6 of the fast one
        hot = module.hot_path
        outs = []
        for generic in (1, 0):
            with _options(langevin_generic=generic):
                hot.manual_seed(4242, 3)
                z, h, _ = hot.langevin(1000, c["target"], 0.3, 5, 0.8, return_history=True)
                outs.append((z.cpu().numpy(), h.cpu().numpy()))
        e_gz, e_gh = rel_err(outs[1][0], outs[0][0]), rel_err(outs[1][1], outs[0][1])
        msg += f"; fast vs generic z {e_gz:.1e} history {e_gh:.1e}"
        assert e_gz <= 2e-6 and e_gh <= 2e-6, (lid, e_gz, e_gh)
    print(msg)
    assert e_hist <= FP32_TOL and e_x <= FP32_TOL, (lid, e_hist, e_x)


@pytest.mark.parametrize("lid", list(LANGEVIN_CASES))
def test_latent_transformation_shape_matrix(lid):
    G = _gu()
    import pseudo_speaker_vae_b200 as P

    module, p64, cfg, c = _langevin_model(lid)
    N, steps = 256, 8
    x, _, _ = O.synth_batch(N, cfg["D"], c["L"], 2, seed=41)
    noises = np.random.default_rng(9).standard_normal((steps, N, c["L"])).astype(np.float32)
    kw = dict(step_size=0.6, max_steps=steps, noise_weight=0.3, prior_weight=0.5, threshold=c["thr"])
    outs = {}
    for generic in ((0, 1) if c["fast"] else (0,)):
        with _options(langevin_generic=generic):
            x_hat, zf, stop, prob = P.latent_transformation(module, torch.from_numpy(x).to(G.DEV), c["target"], noise=torch.from_numpy(noises).to(G.DEV), **kw)
        outs[generic] = (x_hat.numpy(), zf.numpy(), stop.numpy().astype(np.int64), prob.numpy())
    zs = O.vae_forward(p64, x.astype(np.float64), np.zeros((N, c["L"])))[1]
    args = ([n for n in noises.astype(np.float64)], c["target"], kw["step_size"], kw["noise_weight"], kw["prior_weight"], kw["threshold"], _act(cfg))
    zr, sr, pr = O.latent_transformation(p64, zs, *args)
    _, sr32, _ = O.latent_transformation({k: v.astype(np.float32) for k, v in p64.items()}, zs.astype(np.float32),
                                         [n.astype(np.float32) for n in args[0]], *args[1:])
    for generic, (xh, zf, stop, prob) in outs.items():
        e_z, e_x, e_p = rel_err(zf, zr), rel_err(xh, O.decode(p64, zr)), float(np.abs(prob - pr).max())
        print(f"latent transformation {lid} generic={generic}: z {e_z:.1e} x_hat {e_x:.1e} prob {e_p:.1e}, "
              f"{int((stop < steps).sum())} of {N} stopped")
        # the stop step is a comparison with the threshold: exact against the fp64 loop, or the fp32 one where a probability sits on it
        assert np.array_equal(stop, sr) or np.array_equal(stop, sr32), (lid, generic, np.nonzero(stop != sr)[0][:8])
        assert e_z <= FP32_TOL and e_x <= FP32_TOL and e_p <= 1e-5, (lid, generic, e_z, e_x, e_p)
    assert 0 < int((sr < steps).sum()) < N, (lid, "the threshold should stop some samples and not others")
