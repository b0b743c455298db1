"""CPU checks of the trainer options (accumulate_grad_batches, gradient_clip_val / gradient_clip_algorithm): argument validation, the
new library symbols, and the accumulation schedule -- which micro-batch writes the gradient, which adds to it, and which one runs the
all-reduce and Adam -- with the device calls replaced by recorders."""

import pytest
import torch

import pseudo_speaker_vae_b200 as P
from pseudo_speaker_vae_b200 import _lib as L


def _module():
    return P.PseudoSpeakerVAE(model=dict(input_dim=64, latent_dim=8, hidden_dim=64), classifier=dict(input_dim=8, num_classes=2),
                              optimizer=dict(lr=1e-3), scheduler=dict(T_max=10))


@pytest.mark.parametrize("kw", [dict(accumulate_grad_batches=0), dict(accumulate_grad_batches=2.0), dict(accumulate_grad_batches=True),
                                dict(gradient_clip_val=-1.0), dict(gradient_clip_algorithm="l1"), dict(gradient_clip_algorithm="NORM")])
def test_invalid_options_raise(kw):
    with pytest.raises(ValueError):
        P.DataParallelTrainer(_module(), local_only=True, **kw)


@pytest.mark.parametrize("val", [None, 0, 0.0])
def test_clip_val_none_or_zero_is_off(val):
    tr = P.DataParallelTrainer(_module(), local_only=True, gradient_clip_val=val)
    assert tr.gradient_clip_val is None and tr.optimizer.clip_mode == "none"


def test_options_reach_the_optimizer():
    tr = P.DataParallelTrainer(_module(), local_only=True, accumulate_grad_batches=4, gradient_clip_val=0.5, gradient_clip_algorithm="value")
    assert tr.optimizer.grad_scale == 0.25
    assert (tr.optimizer.clip_mode, tr.optimizer.clip_value) == ("value", 0.5)
    tr = P.DataParallelTrainer(_module(), local_only=True, gradient_clip_val=1.0, gradient_clip_algorithm=None)   # Lightning: None means "norm"
    assert tr.optimizer.clip_mode == "norm"
    tr = P.DataParallelTrainer(_module(), local_only=True)
    assert tr.optimizer.grad_scale == 1.0 and tr.optimizer.clip_mode == "none"


def test_new_symbols_are_exported_and_checked():
    lib = L.lib()
    for name in ("psvae_train_fwd_bwd_acc", "psvae_grad_norm", "psvae_adam_step_clip", "psvae_step_counters_advance_by"):
        assert name in L.EXPORTS and hasattr(lib, name)
    assert L.PSVAE_ABI_VERSION == 5 == lib.psvae_abi_version()
    assert lib.psvae_step_counters_advance_by(None, 1, 0, None) != 0       # NULL block or no device: an error code, never a crash
    assert lib.psvae_grad_norm(None, None, 0, 1.0, 1.0, None, None, None, 0, None) != 0


def _recording_trainer(k, monkeypatch, **kw):
    tr = P.DataParallelTrainer(_module(), local_only=True, accumulate_grad_batches=k, **kw)
    gflat = torch.zeros(tr.hot.arena.numel)
    calls = []

    def fwd_bwd(x, y=None, eps=None, counters=None, accumulate=False):
        calls.append(("fwd_bwd", accumulate))
        return torch.zeros(L.NUM_LOSSES), gflat

    monkeypatch.setattr(tr, "_fwd_bwd", fwd_bwd)
    monkeypatch.setattr(tr, "_all_reduce", lambda g, kind=None: calls.append(("all_reduce",)))
    monkeypatch.setattr(tr, "_clip_norm", lambda g: calls.append(("clip_norm",)))
    monkeypatch.setattr(tr.optimizer, "_update", lambda *a, **k: calls.append(("adam",)))
    return tr, calls


@pytest.mark.parametrize("k", [1, 3])
def test_accumulation_schedule(k, monkeypatch):
    tr, calls = _recording_trainer(k, monkeypatch, gradient_clip_val=1.0)
    x = torch.zeros(4, 64)
    for _ in range(2 * k):
        tr.train_step(x, torch.zeros(4, dtype=torch.int64))
    window = [("fwd_bwd", False)] + [("fwd_bwd", True)] * (k - 1) + [("all_reduce",), ("clip_norm",), ("adam",)]
    assert calls == window * 2                       # one fwd+bwd (one Philox offset) per call; all-reduce, norm and Adam once per k calls
    assert tr._micro == 0


def test_flush_ends_a_partial_window(monkeypatch):
    tr, calls = _recording_trainer(4, monkeypatch)
    x = torch.zeros(4, 64)
    tr.train_step(x)
    tr.train_step(x, flush=True)
    tr.train_step(x)
    assert calls == [("fwd_bwd", False), ("fwd_bwd", True), ("all_reduce",), ("clip_norm",), ("adam",), ("fwd_bwd", False)]
    assert tr._micro == 1
    assert tr.optimizer.grad_scale == 0.25          # Lightning's fixed loss / k, also for the flushed partial window
