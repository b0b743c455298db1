"""CPU checks of the classifier-only train step (frozen VAE, ``freeze_vae``): the scope the requires_grad flags select, the new library
symbol and workspace mode, and the argument errors the library reports before it looks for a device."""

import ctypes as C

import pytest

import pseudo_speaker_vae_b200 as P
from pseudo_speaker_vae_b200 import _lib as L


def _module(**kw):
    return P.PseudoSpeakerVAE(model=dict(input_dim=64, latent_dim=8, hidden_dim=64), classifier=dict(input_dim=8, num_classes=2),
                              optimizer=dict(lr=1e-3), scheduler=dict(T_max=10), **kw)


def _set(params, flag):
    for p in params:
        p.requires_grad = flag


def test_scope_follows_requires_grad():
    m = _module()
    hot = m.hot_path
    assert hot.train_scope() == "all"                          # everything trainable
    _set(m.model.parameters(), False)
    assert hot.train_scope() == "classifier"                   # freeze_vae
    _set(list(m.classifier.parameters())[:1], False)
    assert hot.train_scope() == "all"                          # a partly frozen classifier: the full step
    _set(m.classifier.parameters(), False)
    assert hot.train_scope() == "all"                          # nothing trainable
    _set(m.model.parameters(), True)
    assert hot.train_scope() == "all"                          # a frozen classifier only
    _set(m.classifier.parameters(), True)
    _set(list(m.model.parameters())[:2], False)
    assert hot.train_scope() == "all"                          # a partly frozen VAE


def test_freeze_vae_hparam_selects_the_classifier_scope():
    assert _module(freeze_vae=True).hot_path.train_scope() == "classifier"
    m = P.PseudoSpeakerVAE(model=dict(input_dim=64, latent_dim=8, hidden_dim=64), optimizer=dict(lr=1e-3), scheduler=dict(T_max=10),
                           freeze_vae=True)
    assert m.hot_path.train_scope() == "all"                   # no classifier: nothing for the scope to train


def test_classifier_span_is_the_arena_tail():
    hot = _module().hot_path
    a, b = hot.classifier_span()
    assert (a, b) == (int(hot.desc.vae_numel), int(hot.desc.total_numel)) and a % 8 == 0
    clf = [(p, o) for p, o in hot.arena.entries if o >= a]
    assert len(clf) == 2 and all(a <= o and o + p.numel() <= b for p, o in clf)
    assert all(o + p.numel() <= a for p, o in hot.vae_entries())


def test_scoped_entry_point_is_exported():
    lib = L.lib()
    assert "psvae_train_fwd_bwd_scoped" in L.EXPORTS and hasattr(lib, "psvae_train_fwd_bwd_scoped")
    assert L.PSVAE_ABI_VERSION == 5 == lib.psvae_abi_version()


@pytest.mark.parametrize("precision", [L.FP32, L.BF16])
@pytest.mark.parametrize("rows", [2048, 65536])
def test_classifier_workspace_is_far_below_the_train_workspace(precision, rows):
    lib = L.lib()
    for heads, trunk in (([2], 0), ([3, 2], 0), ([3], 2)):
        d = L.make_desc(256, 64, 512, 2, False, trunk, 128 if trunk else 0, "relu", heads, len(heads) == 1)
        train = lib.psvae_workspace_bytes(C.byref(d), rows, precision, L.MODE_TRAIN)
        fwd = lib.psvae_workspace_bytes(C.byref(d), rows, precision, L.MODE_FORWARD)
        clf = lib.psvae_workspace_bytes(C.byref(d), rows, precision, L.MODE_TRAIN_CLASSIFIER)
        assert 0 < fwd <= clf < train
        assert clf < 0.6 * train
    assert lib.psvae_workspace_bytes(C.byref(d), rows, precision, 4) < 0


def _scoped(desc, scope, compute_grads=1):
    # every pointer NULL: the argument checks must answer before the library looks for a device
    return L.lib().psvae_train_fwd_bwd_scoped(C.byref(desc), None, None, None, None, L.X_F32, None, None, 0, 0, 0, 16, 1.0, 1.0, 0,
                                             compute_grads, L.FP32, None, None, None, None, None, 0, None, None, None, None, 0.0, None, 0, None,
                                             scope)


def test_classifier_scope_without_a_classifier_is_an_argument_error():
    d = L.make_desc(64, 8, 64, 2)
    assert _scoped(d, L.GRAD_CLASSIFIER) < 0
    assert "no latent classifier" in L.last_error()
    assert _scoped(d, L.GRAD_CLASSIFIER, compute_grads=0) < 0


def test_unknown_scope_is_an_argument_error():
    d = L.make_desc(64, 8, 64, 2, clf_head_classes=[2])
    assert _scoped(d, 2) < 0 and "grad_scope" in L.last_error()
    assert _scoped(d, -1) < 0


def test_step_rejects_a_bad_scope_before_touching_the_device():
    m = _module()
    x = __import__("torch").zeros(4, 64)
    with pytest.raises(ValueError, match="grad_scope"):
        m.hot_path.step(x, None, grad_scope="vae")
    noclf = P.PseudoSpeakerVAE(model=dict(input_dim=64, latent_dim=8, hidden_dim=64), optimizer=dict(lr=1e-3), scheduler=dict(T_max=10))
    with pytest.raises(ValueError, match="latent classifier"):
        noclf.hot_path.step(x, None, grad_scope="classifier")
