"""CPU checks of per-row classifier targets and target mixes: the exact thresholds a mix becomes, the parsing of per-row targets, the
argument errors psvae_langevin_rows reports before it looks for a device, the export, and the ``--target_mix`` flag of the CLI."""

import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

import pseudo_speaker_vae_b200 as P
from oracle import philox_ref
from oracle import row_targets as RT
from pseudo_speaker_vae_b200 import _lib as L
from pseudo_speaker_vae_b200 import inference
from pseudo_speaker_vae_b200.utils import mix_thresholds, parse_target_mix


# ---- thresholds -------------------------------------------------------------------------------
def test_thresholds_are_exact_integers():
    kept, thr = mix_thresholds([0.3, 0.7])
    assert kept == [0, 1] and thr == [math.floor(Fraction(0.3) * 2 ** 32 / (Fraction(0.3) + Fraction(0.7)))]
    kept, thr = mix_thresholds([1, 1, 1, 1])
    assert thr == [2 ** 30, 2 ** 31, 3 * 2 ** 30]
    kept, thr = mix_thresholds([1, 2])
    assert thr == [(2 ** 32) // 3] and all(isinstance(t, int) for t in thr)


def test_thresholds_are_monotone_and_fit_uint32():
    rng = np.random.default_rng(0)
    for n in (2, 7, 64):
        w = rng.random(n).tolist()
        kept, thr = mix_thresholds(w)
        assert kept == list(range(n)) and len(thr) == n - 1
        assert all(0 <= a <= b < 2 ** 32 for a, b in zip(thr, thr[1:] + [2 ** 32 - 1]))
    # tiny weights next to huge ones: equal thresholds are allowed (the entry is then never drawn)
    _, thr = mix_thresholds([1e-30, 1.0, 1e-30])
    assert thr == [0, 2 ** 32 - 1]


def test_zero_weights_are_dropped_and_one_entry_has_no_threshold():
    assert mix_thresholds([0.0, 2.0, 0, 2.0]) == ([1, 3], [2 ** 31])
    assert mix_thresholds([5]) == ([0], [])
    assert mix_thresholds([0, 0.5, 0]) == ([1], [])


@pytest.mark.parametrize("weights,exc", [([], ValueError), ([0, 0], ValueError), ([1, -0.5], ValueError), ([1, float("nan")], ValueError),
                                         ([1, float("inf")], ValueError), ([1] * 65, ValueError), (["a"], TypeError), ([True], TypeError)])
def test_threshold_errors(weights, exc):
    with pytest.raises(exc):
        mix_thresholds(weights)


def test_more_than_64_entries_count_after_dropping_zero_weights():
    assert len(mix_thresholds([1] * 64 + [0] * 10)[0]) == 64


def test_draw_target_mix_reference():
    thr = mix_thresholds([1, 2, 1])[1]
    for row0 in (0, 5):
        k = RT.draw_target_mix(thr, 37, seed=11, offset=9, row0=row0)
        u = philox_ref.philox_uint32(37, 11, 9, first_elem=row0)
        want = np.array([next((j for j, t in enumerate(thr) if x < t), len(thr)) for x in u.tolist()])
        assert np.array_equal(k, want)
    # shards of the row range draw what one call draws
    full = RT.draw_target_mix(thr, 100, 3, 4)
    assert np.array_equal(np.concatenate([RT.draw_target_mix(thr, 33, 3, 4, 0), RT.draw_target_mix(thr, 67, 3, 4, 33)]), full)


# ---- per-row target parsing -------------------------------------------------------------------
def _single():
    return P.PseudoSpeakerVAE(model=dict(input_dim=64, latent_dim=16, hidden_dim=64), classifier=dict(input_dim=16, num_classes=3),
                              optimizer={}, scheduler=dict(T_max=1)).hot_path


def _multi():
    return P.PseudoSpeakerVAE(model=dict(input_dim=64, latent_dim=16, hidden_dim=64),
                              classifier=dict(input_dim=16, num_classes={"gender": 3, "age": 3}), optimizer={}, scheduler=dict(T_max=1)).hot_path


def test_shared_forms_keep_the_shared_path():
    hot, mhot = _single(), _multi()
    assert hot.row_targets_for(1, 5, "cpu") is None
    assert hot.row_targets_for(torch.tensor(2), 5, "cpu") is None               # 0-d tensor: shared
    assert mhot.row_targets_for({"gender": 1}, 5, "cpu") is None
    assert mhot.row_targets_for({"gender": torch.tensor(1)}, 5, "cpu") is None


def test_single_label_rows():
    hot = _single()
    t = hot.row_targets_for(torch.tensor([0, 2, 1, 1]), 4, "cpu", check=True)
    assert t.dtype == torch.int32 and t.tolist() == [[0, 2, 1, 1]]
    assert hot.row_targets_for(np.array([2, 0], dtype=np.int64), 2, "cpu").tolist() == [[2, 0]]
    # unchecked: out-of-range values stay out of range (no wrap into a valid class) for the kernel's NaN rule
    assert hot.row_targets_for(torch.tensor([2 ** 32, -2 ** 32, 5]), 3, "cpu").tolist() == [[127, -2, 5]]


def test_multi_label_rows_broadcast_and_fill():
    hot = _multi()
    t = hot.row_targets_for({"gender": torch.tensor([0, 1, -1]), "age": 2}, 3, "cpu", check=True)
    assert t.tolist() == [[0, 1, -1], [2, 2, 2]]
    t = hot.row_targets_for({"age": np.array([1, 0, 2])}, 3, "cpu", check=True)
    assert t.tolist() == [[-1, -1, -1], [1, 0, 2]]


@pytest.mark.parametrize("target,exc", [
    (torch.tensor([0, 1, 2]), ValueError),                     # length 3 for 4 rows
    (torch.tensor([[0, 1], [1, 0]]), ValueError),              # 2-D
    (torch.tensor([0.0, 1.0, 1.0, 0.0]), TypeError),           # not an integer tensor
    (torch.tensor([True, False, True, False]), TypeError),
    (torch.tensor([0, 3, 1, 1]), IndexError),                  # checked: out of range
    (torch.tensor([0, -1, 1, 1]), ValueError),                 # checked: a row that names no head
    ({"gender": torch.tensor([0, 1, 0, 1])}, ValueError),      # dict for a single-label classifier
])
def test_single_label_row_errors(target, exc):
    with pytest.raises(exc):
        _single().row_targets_for(target, 4, "cpu", check=True)


@pytest.mark.parametrize("target,exc", [
    (torch.tensor([0, 1, 1]), ValueError),                                    # tensor for a multi-label classifier
    ({"gender": torch.tensor([0, 1])}, ValueError),                           # length
    ({"gender": torch.tensor([0, 1, 1]), "age": 3}, IndexError),              # broadcast int out of range
    ({"gender": torch.tensor([0, 1, 1]), "accent": 0}, KeyError),             # unknown label
    ({"gender": torch.tensor([0, -1, 1])}, ValueError),                       # checked: row 1 names no head
    ({"gender": torch.tensor([0, -2, 1]), "age": 1}, IndexError),             # checked: below -1
    ({"gender": torch.tensor([0, 1, 1]), "age": torch.tensor([0, 1, 3])}, IndexError),
])
def test_multi_label_row_errors(target, exc):
    with pytest.raises(exc):
        _multi().row_targets_for(target, 3, "cpu", check=True)


def test_target_mix_entries():
    hot = _multi()
    entries, thr = hot.target_mix_for([({"gender": 0, "age": 1}, 0.3), ({"gender": 1}, 0.0), ({"age": 2}, 0.7)])
    assert entries == [[0, 1], [-1, 2]] and thr == mix_thresholds([0.3, 0.7])[1]
    with pytest.raises(IndexError):
        hot.target_mix_for([({"gender": 3}, 1.0)])
    with pytest.raises(ValueError):
        hot.target_mix_for([])
    with pytest.raises(ValueError):
        hot.target_mix_for([({"gender": 0}, 1.0, 2)])
    with pytest.raises(ValueError):
        hot.target_mix_for([({"gender": 0}, -1.0)])
    assert _single().target_mix_for([(2, 1), (0, 3)]) == ([[2], [0]], [2 ** 30])


# ---- the C-ABI ----------------------------------------------------------------------------------
def test_rows_entry_point_is_exported():
    lib = L.lib()
    assert "psvae_langevin_rows" in L.EXPORTS and hasattr(lib, "psvae_langevin_rows")
    assert L.PSVAE_ABI_VERSION == 5 == lib.psvae_abi_version()
    assert L.MAX_TARGET_MIX == 64


def _rows_call(desc, row_targets=None, mix=(), thr=(), targets_out=True, n_mix=None):
    # no device pointers beyond opaque placeholders: the argument checks must answer before the library looks for a device
    n = len(mix) if n_mix is None else n_mix
    marr = (C.c_int32 * max(1, len(mix) * L.MAX_CLF_HEADS))(*[t for e in mix for t in list(e) + [-1] * (L.MAX_CLF_HEADS - len(e))])
    tarr = (C.c_uint32 * max(1, len(thr)))(*thr)
    rc = L.lib().psvae_langevin_rows(C.byref(desc), None, None, 16, row_targets, n, marr if mix else None, tarr if thr else None,
                                     0x1000 if targets_out else None, 0.01, 5, 1.0, 0, 0, 0, 1, None, None, None, 1.0, 0.0, None, None, None)
    return rc, L.last_error()


def _desc(heads=(3, 3), single=False):
    return L.make_desc(64, 16, 64, 2, False, 0, 0, "relu", list(heads), single)


@pytest.mark.parametrize("case", ["no_classifier", "neither", "both", "too_many", "negative_n", "no_head", "class_high", "class_low",
                                  "head_beyond", "decreasing", "no_out"])
def test_rows_argument_errors_need_no_device(case):
    d = _desc()
    kw = dict(mix=[(0, 1), (1, -1)], thr=[2 ** 31])
    if case == "no_classifier":
        d = L.make_desc(64, 16, 64, 2, False, 0, 0, "relu", [], True)
    elif case == "neither":
        kw = dict()
    elif case == "both":
        kw["row_targets"] = 0x1000
    elif case == "too_many":
        kw = dict(mix=[(0, 0)] * 65, thr=list(range(64)))
    elif case == "negative_n":
        kw = dict(mix=[(0, 0)], n_mix=-1)
    elif case == "no_head":
        kw = dict(mix=[(0, 1), (-1, -1)], thr=[5])
    elif case == "class_high":
        kw = dict(mix=[(0, 3)], thr=[])
    elif case == "class_low":
        kw = dict(mix=[(-2, 0)], thr=[])
    elif case == "head_beyond":
        kw = dict(mix=[(0, 1, 0)], thr=[])
    elif case == "decreasing":
        kw = dict(mix=[(0, 1), (1, 1), (2, 2)], thr=[10, 9])
    elif case == "no_out":
        kw["targets_out"] = False
    rc, msg = _rows_call(d, **kw)
    assert rc in (-1, -2), (case, rc, msg)
    assert "device" not in msg.lower(), msg


def test_valid_rows_arguments_reach_the_device_check():
    # the same calls with valid arguments get as far as the device check (or, on a GPU box, the NULL-pointer check)
    for kw in (dict(mix=[(0, 1), (1, -1)], thr=[2 ** 31]), dict(row_targets=0x1000), dict(mix=[(-1, 2)], thr=[]),
               dict(mix=[(0, 0), (1, 1)], thr=[7, 7][:1])):
        rc, msg = _rows_call(_desc(), **kw)
        assert rc != 0 and ("device" in msg.lower() or "sm_100" in msg.lower() or "must not be null" in msg.lower()), (kw, rc, msg)


# ---- the CLI ------------------------------------------------------------------------------------
def test_parse_target_mix():
    mix = parse_target_mix('[[{"gender": 0, "age": 1}, 0.3], [1, 2]]')
    assert mix == [({"gender": 0, "age": 1}, 0.3), (1, 2.0)]
    for bad in ("[]", "{}", "[[0]]", "[[0, 1, 2]]", '[["a", 1]]', '[[0, "w"]]', "[[0, true]]", "not json"):
        with pytest.raises(ValueError):
            parse_target_mix(bad)


@pytest.mark.parametrize("extra", [["--synthesis_type", "conditional", "--classifier_target", "1", "--target_mix", "[[0, 1]]"],
                                   ["--synthesis_type", "unconditional", "--target_mix", "[[0, 1]]"],
                                   ["--synthesis_type", "conditional", "--target_mix", "[[0, -1]]x"]])
def test_cli_target_mix_conflicts(extra, tmp_path):
    # rejected while parsing, before the checkpoint (which does not exist) is opened
    with pytest.raises(SystemExit) as e:
        inference.main(["--vae_ckpt_path", str(tmp_path / "missing.ckpt"), "--save_dir", str(tmp_path)] + extra)
    assert e.value.code == 2
