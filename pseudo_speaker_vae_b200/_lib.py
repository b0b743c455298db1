"""ctypes binding of include/psvae_b200.h -- the only door between the Python host code and the CUDA kernels.

Every compute entry point of this package goes through ``lib()``; if ``libpsvae_b200.so`` has not been built
(``python -m pseudo_speaker_vae_b200.build``) that is a hard error -- there is no eager/PyTorch/CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

HERE = os.path.dirname(os.path.abspath(__file__))
# PSVAE_B200_LIB: load another build of the same ABI instead (A/B timing of two kernel versions in one process tree; tools only)
LIB_PATH = os.environ.get("PSVAE_B200_LIB") or os.path.join(HERE, "libpsvae_b200.so")

PSVAE_ABI_VERSION = 5
MAX_LAYERS = 8
MAX_CLF_TRUNK = 4
MAX_CLF_HEADS = 4
NUM_LOSSES = 16
FP32, BF16 = 0, 1
X_F32, X_BF16 = 0, 1
MODE_TRAIN, MODE_FORWARD, MODE_DECODE, MODE_TRAIN_CLASSIFIER = 0, 1, 2, 3
#: psvae_train_fwd_bwd_scoped: which parameters get gradients
GRAD_ALL, GRAD_CLASSIFIER = 0, 1
ACTIVATIONS = {"relu": 0, "tanh": 1, "sigmoid": 2, "leaky_relu": 3}
LOSS_TOTAL, LOSS_RECON, LOSS_KL, LOSS_CLF, LOSS_CLF_HEAD0, LOSS_ACC_HEAD0 = 0, 1, 2, 3, 4, 8
LOSS_CONS, LOSS_CONS_ACC = 12, 13

#: every symbol include/psvae_b200.h declares (tests check the library exports exactly these)
EXPORTS = [
    "psvae_abi_version", "psvae_last_error_string", "psvae_model_desc_init", "psvae_workspace_bytes", "psvae_shadow_bytes",
    "psvae_flops_per_sample", "psvae_set_option", "psvae_get_option", "psvae_adam_step", "psvae_adam_step_ex", "psvae_philox_uint32", "psvae_philox_normal",
    "psvae_refresh_shadow", "psvae_forward", "psvae_decode", "psvae_train_fwd_bwd", "psvae_langevin", "psvae_gemm_bf16",
    "psvae_gemm_fp32", "psvae_gemm_probe", "psvae_launch_count", "psvae_consistency_desc_init", "psvae_consistency_workspace_bytes",
    "psvae_consistency_forward", "psvae_train_fwd_bwd_consistency", "psvae_vae_backward", "psvae_gather_rows",
    "psvae_embedding_classifier_workspace_bytes", "psvae_embedding_classifier_step", "psvae_train_fwd_bwd_dc", "psvae_adam_step_dc",
    "psvae_step_counters_advance", "psvae_train_fwd_bwd_acc", "psvae_grad_norm", "psvae_adam_step_clip", "psvae_step_counters_advance_by",
    "psvae_train_fwd_bwd_scoped", "psvae_langevin_rows", "psvae_cosine_topk_workspace_bytes", "psvae_cosine_topk",
]

#: int64 slots of ``psvae_step_counters`` (a device tensor of COUNTER_SLOTS int64)
COUNTER_RNG_OFFSET, COUNTER_ADAM_STEP, COUNTER_SLOTS = 0, 1, 4
#: psvae_adam_step_clip modes and the psvae_grad_norm limits
CLIP_NONE, CLIP_NORM, CLIP_VALUE = 0, 1, 2
GRAD_NORM_MAX_SPANS, GRAD_NORM_SCRATCH_BYTES = 16, 4096
#: psvae_langevin_rows: entries of a target mix
MAX_TARGET_MIX = 64
#: psvae_cosine_topk flags and limits
TOPK_SMALLEST, TOPK_EXCLUDE_SELF = 1, 2
TOPK_MAX_K, TOPK_MAX_DIM = 16, 512


class ModelDesc(C.Structure):
    """Mirror of ``psvae_model_desc``."""

    _fields_ = [
        ("input_dim", C.c_int32), ("latent_dim", C.c_int32), ("hidden_dim", C.c_int32), ("num_hidden", C.c_int32),
        ("normalize_decoder", C.c_int32), ("clf_num_trunk", C.c_int32), ("clf_hidden", C.c_int32), ("clf_activation", C.c_int32),
        ("clf_num_heads", C.c_int32), ("clf_single_label", C.c_int32), ("clf_head_classes", C.c_int32 * MAX_CLF_HEADS),
        ("reserved_", C.c_int32 * 2),
        ("enc_w", C.c_int64 * MAX_LAYERS), ("enc_b", C.c_int64 * MAX_LAYERS), ("dec_w", C.c_int64 * MAX_LAYERS), ("dec_b", C.c_int64 * MAX_LAYERS),
        ("clf_trunk_w", C.c_int64 * MAX_CLF_TRUNK), ("clf_trunk_b", C.c_int64 * MAX_CLF_TRUNK),
        ("clf_head_w", C.c_int64 * MAX_CLF_HEADS), ("clf_head_b", C.c_int64 * MAX_CLF_HEADS),
        ("vae_numel", C.c_int64), ("total_numel", C.c_int64),
    ]


class ConsistencyDesc(C.Structure):
    """Mirror of ``psvae_consistency_desc``."""

    _fields_ = [("input_dim", C.c_int32), ("hidden_dim", C.c_int32), ("num_classes", C.c_int32), ("reserved_", C.c_int32),
                ("w", C.c_int64 * 3), ("b", C.c_int64 * 3), ("total_numel", C.c_int64)]


_lib: Optional[C.CDLL] = None


def _declare(l: C.CDLL) -> None:
    P, I32, I64, U64, F, VP, DBL = C.POINTER, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_void_p, C.c_double
    D = P(ModelDesc)
    l.psvae_abi_version.restype = C.c_int
    l.psvae_abi_version.argtypes = []
    l.psvae_last_error_string.restype = C.c_char_p
    l.psvae_last_error_string.argtypes = []
    l.psvae_launch_count.restype = I64
    l.psvae_launch_count.argtypes = []
    l.psvae_set_option.restype = C.c_int
    l.psvae_set_option.argtypes = [C.c_char_p, I64]
    l.psvae_get_option.restype = I64
    l.psvae_get_option.argtypes = [C.c_char_p]
    l.psvae_model_desc_init.restype = C.c_int
    l.psvae_model_desc_init.argtypes = [D, I32, I32, I32, I32, I32, I32, I32, I32, I32, I32, P(I32)]
    l.psvae_workspace_bytes.restype = I64
    l.psvae_workspace_bytes.argtypes = [D, I64, I32, I32]
    l.psvae_shadow_bytes.restype = I64
    l.psvae_shadow_bytes.argtypes = [D]
    l.psvae_flops_per_sample.restype = I64
    l.psvae_flops_per_sample.argtypes = [D, I32]
    l.psvae_adam_step.restype = C.c_int
    l.psvae_adam_step.argtypes = [VP, VP, VP, VP, I64, DBL, DBL, DBL, DBL, DBL, I64, DBL, VP, VP]
    l.psvae_adam_step_ex.restype = C.c_int
    l.psvae_adam_step_ex.argtypes = [VP, VP, VP, VP, VP, I64, DBL, DBL, DBL, DBL, DBL, I64, DBL, C.c_int32, C.c_int32, VP, VP]
    l.psvae_philox_uint32.restype = C.c_int
    l.psvae_philox_uint32.argtypes = [VP, I64, U64, U64, I64, VP]
    l.psvae_philox_normal.restype = C.c_int
    l.psvae_philox_normal.argtypes = [VP, I64, I32, U64, U64, I64, VP]
    l.psvae_gather_rows.restype = C.c_int
    l.psvae_gather_rows.argtypes = [VP, I64, I64, VP, I64, VP, VP]
    l.psvae_refresh_shadow.restype = C.c_int
    l.psvae_refresh_shadow.argtypes = [D, VP, VP, VP]
    l.psvae_forward.restype = C.c_int
    l.psvae_forward.argtypes = [D, VP, VP, VP, I32, VP, U64, U64, I64, I64, I32, VP, VP, VP, VP, I64, VP]
    l.psvae_decode.restype = C.c_int
    l.psvae_decode.argtypes = [D, VP, VP, VP, U64, U64, I64, I64, I32, VP, VP, VP, I64, VP]
    l.psvae_train_fwd_bwd.restype = C.c_int
    l.psvae_train_fwd_bwd.argtypes = [D, VP, VP, VP, VP, I32, VP, VP, U64, U64, I64, I64, F, F, I32, I32, I32, VP, VP, VP, VP, VP, I64, VP]
    l.psvae_vae_backward.restype = C.c_int
    l.psvae_vae_backward.argtypes = [D, VP, VP, VP, VP, I32, VP, U64, U64, I64, I64, I32, VP, VP, VP, VP, I64, VP]
    CD = P(ConsistencyDesc)
    l.psvae_consistency_desc_init.restype = C.c_int
    l.psvae_consistency_desc_init.argtypes = [CD, I32, I32, I32]
    l.psvae_consistency_workspace_bytes.restype = I64
    l.psvae_consistency_workspace_bytes.argtypes = [CD, I64, I32]
    l.psvae_consistency_forward.restype = C.c_int
    l.psvae_consistency_forward.argtypes = [CD, VP, VP, I64, VP, VP, I64, VP]
    l.psvae_embedding_classifier_workspace_bytes.restype = I64
    l.psvae_embedding_classifier_workspace_bytes.argtypes = [CD, I64]
    l.psvae_embedding_classifier_step.restype = C.c_int
    l.psvae_embedding_classifier_step.argtypes = [CD, VP, VP, VP, VP, I64, I32, VP, VP, VP, I64, VP]
    l.psvae_train_fwd_bwd_consistency.restype = C.c_int
    l.psvae_train_fwd_bwd_consistency.argtypes = l.psvae_train_fwd_bwd.argtypes + [CD, VP, VP, F]
    l.psvae_train_fwd_bwd_dc.restype = C.c_int
    l.psvae_train_fwd_bwd_dc.argtypes = l.psvae_train_fwd_bwd_consistency.argtypes + [VP]
    l.psvae_adam_step_dc.restype = C.c_int
    l.psvae_adam_step_dc.argtypes = [VP, VP, VP, VP, VP, I64, VP, VP, DBL, DBL, DBL, DBL, DBL, C.c_int32, C.c_int32, VP, VP]
    l.psvae_step_counters_advance.restype = C.c_int
    l.psvae_step_counters_advance.argtypes = [VP, VP]
    # additive to ABI 5: an earlier ABI-5 build without them (loaded through PSVAE_B200_LIB for A/B timing) still loads
    if hasattr(l, "psvae_train_fwd_bwd_acc"):
        l.psvae_train_fwd_bwd_acc.restype = C.c_int
        l.psvae_train_fwd_bwd_acc.argtypes = l.psvae_train_fwd_bwd_dc.argtypes + [I32, VP]
        l.psvae_grad_norm.restype = C.c_int
        l.psvae_grad_norm.argtypes = [VP, P(I64), I32, DBL, DBL, VP, VP, VP, I64, VP]
        l.psvae_adam_step_clip.restype = C.c_int
        l.psvae_adam_step_clip.argtypes = [VP, VP, VP, VP, VP, I64, DBL, I64, VP, VP, DBL, DBL, DBL, DBL, DBL, C.c_int32, C.c_int32, C.c_int32, VP,
                                           DBL, VP, VP]
        l.psvae_step_counters_advance_by.restype = C.c_int
        l.psvae_step_counters_advance_by.argtypes = [VP, U64, I64, VP]
    if hasattr(l, "psvae_train_fwd_bwd_scoped"):
        l.psvae_train_fwd_bwd_scoped.restype = C.c_int
        l.psvae_train_fwd_bwd_scoped.argtypes = l.psvae_train_fwd_bwd_acc.argtypes + [I32]
    l.psvae_langevin.restype = C.c_int
    l.psvae_langevin.argtypes = [D, VP, VP, I64, P(I32), F, I32, F, U64, U64, I64, I32, VP, VP, VP, F, F, VP, VP, VP]
    if hasattr(l, "psvae_langevin_rows"):
        l.psvae_langevin_rows.restype = C.c_int
        l.psvae_langevin_rows.argtypes = [D, VP, VP, I64, VP, I32, P(I32), P(C.c_uint32), VP, F, I32, F, U64, U64, I64, I32, VP, VP, VP, F, F, VP, VP,
                                          VP]
    if hasattr(l, "psvae_cosine_topk"):
        l.psvae_cosine_topk_workspace_bytes.restype = I64
        l.psvae_cosine_topk_workspace_bytes.argtypes = [I64, I64, I32, I32]
        l.psvae_cosine_topk.restype = C.c_int
        l.psvae_cosine_topk.argtypes = [VP, I32, I64, I64, VP, I32, I64, I64, I32, I32, I32, VP, VP, VP, I64, VP]
    l.psvae_gemm_bf16.restype = C.c_int
    l.psvae_gemm_bf16.argtypes = [VP, VP, VP, VP, I64, I32, I64, I32, I32, I32, I32, VP, I64, VP]
    l.psvae_gemm_probe.restype = C.c_int
    l.psvae_gemm_probe.argtypes = [VP, VP, VP, VP, VP, VP, I64, I32, I64, I32, VP]
    l.psvae_gemm_fp32.restype = C.c_int
    l.psvae_gemm_fp32.argtypes = [VP, VP, VP, VP, I64, I32, I64, I32, I32, I32, VP]


def lib() -> C.CDLL:
    """The loaded library.  Raises if it was never built: this package has no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built (python -m pseudo_speaker_vae_b200.build). "
                "pseudo_speaker_vae_b200 has no PyTorch/CPU fallback.")
        l = C.CDLL(LIB_PATH)
        _declare(l)
        v = l.psvae_abi_version()
        if v != PSVAE_ABI_VERSION:
            raise RuntimeError(f"ABI mismatch: library {v}, binding {PSVAE_ABI_VERSION}; rebuild the extension")
        for key, val in os.environ.items():          # PSVAE_OPT_<NAME>=<int>: tuning options without touching code
            if key.startswith("PSVAE_OPT_"):
                if l.psvae_set_option(key[len("PSVAE_OPT_"):].lower().encode(), int(val)) != 0:
                    raise ValueError(f"{key}: {l.psvae_last_error_string().decode()}")
        _lib = l
    return _lib


def last_error() -> str:
    return lib().psvae_last_error_string().decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    """Map the C-ABI return convention onto Python exceptions (include/psvae_b200.h: 0 ok, <0 argument, >0 cudaError_t)."""
    if rc == 0:
        return
    msg = f"{what}: {last_error()}" if what else last_error()
    if rc in (-1, -2):
        raise ValueError(msg)
    if rc == -4:
        raise RuntimeError(msg + " [no sm_100 device: this package has no CPU fallback]")
    raise RuntimeError(f"{msg} (code {rc})")


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


#: bumped by every set_option(): cached workspace sizes (engine.HotPath._workspace) depend on the tuning options
OPTIONS_EPOCH = 0


def set_option(name: str, value: int) -> None:
    global OPTIONS_EPOCH
    check(lib().psvae_set_option(name.encode(), int(value)), "psvae_set_option")
    OPTIONS_EPOCH += 1


def get_option(name: str) -> int:
    return int(lib().psvae_get_option(name.encode()))


def make_consistency_desc(input_dim: int, hidden_dim: int, num_classes: int) -> ConsistencyDesc:
    d = ConsistencyDesc()
    check(lib().psvae_consistency_desc_init(C.byref(d), int(input_dim), int(hidden_dim), int(num_classes)), "psvae_consistency_desc_init")
    return d


def make_desc(input_dim: int, latent_dim: int, hidden_dim: int = 512, num_hidden: int = 2, normalize_decoder: bool = False,
              clf_num_trunk: int = 0, clf_hidden: int = 0, clf_activation: str = "relu", clf_head_classes=(), clf_single_label: bool = True) -> ModelDesc:
    if clf_activation not in ACTIVATIONS:
        raise ValueError(f"Unsupported activation: {clf_activation}")
    d = ModelDesc()
    heads = list(clf_head_classes)
    if len(heads) > MAX_CLF_HEADS:
        raise ValueError(f"at most {MAX_CLF_HEADS} classifier heads are supported, got {len(heads)}")
    arr = (C.c_int32 * max(1, len(heads)))(*heads) if heads else None
    rc = lib().psvae_model_desc_init(C.byref(d), input_dim, latent_dim, hidden_dim, num_hidden, int(bool(normalize_decoder)), clf_num_trunk,
                                     clf_hidden, ACTIVATIONS[clf_activation], len(heads), int(bool(clf_single_label)), arr)
    check(rc, "psvae_model_desc_init")
    return d
