"""CPU-side tests of the cosine top-k search: argument errors before any device work (Python and C-ABI), the workspace-size function,
the fp64 reference's ordering / NaN / exclude-self rules on hand-built cases, and the inference CLI's --nearest_store / --nearest_k."""
import ctypes as C
import json

import numpy as np
import pytest
import torch

import pseudo_speaker_vae_b200 as P
from oracle import cosine_topk as R
from pseudo_speaker_vae_b200 import _lib as L
from pseudo_speaker_vae_b200 import inference


# ---- the Python entry point ---------------------------------------------------------------------
@pytest.mark.parametrize("case", ["k0", "k17", "dim12", "dim520", "dim_mismatch", "dtype", "k_gt_nk", "k_gt_nk_excl", "devices", "rank",
                                  "row0"])
def test_argument_errors_before_device_work(case):
    q, x, kw = torch.zeros(4, 16), torch.zeros(5, 16), dict(k=1)
    if case == "k0":
        kw["k"] = 0
    elif case == "k17":
        kw["k"] = 17
    elif case == "dim12":
        q, x = torch.zeros(4, 12), torch.zeros(5, 12)
    elif case == "dim520":
        q, x = torch.zeros(4, 520), torch.zeros(5, 520)
    elif case == "dim_mismatch":
        x = torch.zeros(5, 24)
    elif case == "dtype":
        q = torch.zeros(4, 16, dtype=torch.float16)
    elif case == "k_gt_nk":
        kw["k"] = 6
    elif case == "k_gt_nk_excl":
        kw.update(k=5, exclude_self=True)
    elif case == "devices":
        x = torch.zeros(5, 16, device="meta")
    elif case == "rank":
        q = torch.zeros(4, 2, 8)
    elif case == "row0":
        kw["query_row0"] = -1
    with pytest.raises(ValueError):
        P.cosine_topk(q, x, **kw)


def test_valid_cpu_arguments_are_refused_as_no_device():
    with pytest.raises(RuntimeError, match="CUDA"):
        P.cosine_topk(torch.zeros(4, 16), torch.zeros(5, 16), 5)


# ---- the C-ABI ----------------------------------------------------------------------------------
def test_entry_points_are_exported():
    lib = L.lib()
    for name in ("psvae_cosine_topk", "psvae_cosine_topk_workspace_bytes"):
        assert name in L.EXPORTS and hasattr(lib, name)
    assert L.get_option("topk_key_splits") == 0


def _abi_call(nq=300, nk=1000, dim=256, k=4, flags=0, q_dtype=L.X_F32, k_dtype=L.X_F32, ws_bytes=None, q_row0=0, q=0x1000):
    # opaque placeholders instead of device pointers: the argument checks must answer before the library looks for a device
    if ws_bytes is None:
        ws_bytes = 1 << 40
    rc = L.lib().psvae_cosine_topk(q, q_dtype, nq, q_row0, 0x2000, k_dtype, nk, 0, dim, k, flags, 0x3000, 0x4000, 0x5000, ws_bytes, None)
    return rc, L.last_error()


@pytest.mark.parametrize("case", ["k0", "k17", "dim0", "dim12", "dim520", "q_dtype", "k_dtype", "flags", "k_gt_nk", "k_gt_nk_excl", "nq0",
                                  "nk0", "row0", "workspace"])
def test_abi_argument_errors_need_no_device(case):
    kw = {"k0": dict(k=0), "k17": dict(k=17), "dim0": dict(dim=0), "dim12": dict(dim=12), "dim520": dict(dim=520), "q_dtype": dict(q_dtype=2),
          "k_dtype": dict(k_dtype=-1), "flags": dict(flags=4), "k_gt_nk": dict(nk=3), "k_gt_nk_excl": dict(nk=4, flags=L.TOPK_EXCLUDE_SELF),
          "nq0": dict(nq=0), "nk0": dict(nk=0), "row0": dict(q_row0=-5), "workspace": dict(ws_bytes=1024)}[case]
    rc, msg = _abi_call(**kw)
    assert rc in (-1, -2), (case, rc, msg)
    assert "device" not in msg.lower(), msg


def test_valid_abi_arguments_reach_the_device_check():
    # a NULL query pointer: valid arguments get as far as the device check, or on a GPU box to the NULL-pointer check, and launch nothing
    L.lib().psvae_set_option(b"no_such_option", 0)        # clears a stale message of an earlier call
    for kw in (dict(), dict(flags=L.TOPK_SMALLEST | L.TOPK_EXCLUDE_SELF, nk=5), dict(q_dtype=L.X_BF16), dict(dim=8, k=16, nk=16)):
        rc, msg = _abi_call(q=None, **kw)
        assert rc != 0 and ("device" in msg.lower() or "sm_100" in msg.lower() or "must not be null" in msg.lower()), (kw, rc, msg)


def test_workspace_bytes():
    ws = L.lib().psvae_cosine_topk_workspace_bytes
    big = ws(1 << 20, 674068, 256, 16)
    # unit bf16 copies + inverse norms of both sets + one key range of 32 candidates per query row (8 bytes each)
    assert big >= (1 << 20) * 256 * 2 + 674068 * 256 * 2 + 4 * ((1 << 20) + 674068) + (1 << 20) * 32 * 8
    assert big < 2 * ((1 << 20) * 256 * 2 + 674068 * 256 * 2 + (1 << 20) * 32 * 8)
    assert ws(300, 1000, 256, 1) < ws(300, 1000, 256, 16) < ws(300, 1000, 512, 16)
    assert ws(0, 10, 64, 1) == -1 and "nq" in L.last_error()
    assert ws(10, 10, 60, 1) == -1 and "dim" in L.last_error()
    assert ws(10, 10, 64, 0) == -1 and "k" in L.last_error()
    # few queries: the key range is split for the grid, more candidate lists, more workspace; a forced split count changes the size
    base = ws(1000, 100000, 256, 4)
    try:
        L.set_option("topk_key_splits", 1)
        one = ws(1000, 100000, 256, 4)
        L.set_option("topk_key_splits", 7)
        seven = ws(1000, 100000, 256, 4)
    finally:
        L.set_option("topk_key_splits", 0)
    assert one < seven and one < base
    assert seven - one == 6 * 8 * 128 * 8 * 8          # 6 more key ranges x 8 query tiles x 128 rows x 8 candidates x 8 bytes


# ---- the fp64 reference -------------------------------------------------------------------------
def test_oracle_ties_go_to_the_lower_index():
    q = np.array([[1.0, 0.0]])
    x = np.array([[0.0, 1.0], [2.0, 0.0], [1.0, 0.0], [-1.0, 0.0], [3.0, 0.0]])
    s, i = R.cosine_topk(q, x, 4)
    assert i.tolist() == [[1, 2, 4, 0]] and np.allclose(s, [[1, 1, 1, 0]])
    s, i = R.cosine_topk(q, x, 2, largest=False)
    assert i.tolist() == [[3, 0]] and np.allclose(s, [[-1, 0]])
    s, i = R.cosine_topk(q, x, 2, key_row0=100)
    assert i.tolist() == [[101, 102]]


def test_oracle_zero_rows_score_zero_and_nan_is_never_chosen():
    q = np.array([[1.0, 1.0], [0.0, 0.0]])
    x = np.array([[np.nan, 1.0], [-1.0, -1.0], [0.0, 0.0], [1.0, 0.5]])
    s, i = R.cosine_topk(q, x, 3)
    assert i[0].tolist() == [3, 2, 1]
    assert s[0, 1] == 0.0
    assert i[1].tolist() == [1, 2, 3] and s[1].tolist() == [0.0, 0.0, 0.0]         # a zero query scores 0 against everything
    s, i = R.cosine_topk(q, x, 4)                     # the NaN key is never chosen: its slot stays empty
    assert i[:, 3].tolist() == [-1, -1] and np.isnan(s[:, 3]).all()
    s, i = R.cosine_topk(np.array([[np.nan, 0.0]]), x, 2)
    assert i.tolist() == [[-1, -1]] and np.isnan(s).all()


def test_oracle_exclude_self_and_sharding():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((50, 16))
    x[7] = x[3]                                           # a duplicate: with the diagonal removed, 3 and 7 find each other
    s, i = R.cosine_topk(x, x, 3, exclude_self=True)
    assert (i != np.arange(50)[:, None]).all()
    assert i[3, 0] == 7 and i[7, 0] == 3 and np.isclose(s[3, 0], 1.0)
    full = R.cosine_sim(x, x)
    np.fill_diagonal(full, np.nan)
    assert np.allclose(s[:, 0], np.nanmax(full, axis=1))
    parts = [R.cosine_topk(x[a:b], x, 3, exclude_self=True, query_row0=a) for a, b in ((0, 17), (17, 18), (18, 50))]
    assert np.array_equal(np.concatenate([p[1] for p in parts]), i)
    s2, i2 = R.cosine_topk(x, x, 3, exclude_self=True, chunk=7)
    assert np.array_equal(i2, i) and np.array_equal(s2, s)


# ---- the CLI ------------------------------------------------------------------------------------
def test_cli_nearest_flags_parse(tmp_path, monkeypatch):
    base = ["--vae_ckpt_path", str(tmp_path / "missing.ckpt"), "--save_dir", str(tmp_path), "--synthesis_type", "unconditional"]
    for extra in (["--nearest_store", str(tmp_path / "nostore")], ["--nearest_store", str(tmp_path), "--nearest_k", "0"],
                  ["--nearest_store", str(tmp_path), "--nearest_k", "17"]):
        with pytest.raises(SystemExit) as e:            # rejected while parsing, before the checkpoint (which does not exist) is opened
            inference.main(base + extra)
        assert e.value.code == 2
    store = tmp_path / "store"
    P.PackedEmbeddingStore.from_arrays(str(store), np.zeros((3, 16), np.float32))
    assert json.load(open(store / "index.json"))["n"] == 3
    seen = {}

    def fake_load(path):
        seen["path"] = path
        raise FileNotFoundError(path)

    monkeypatch.setattr(P.PseudoSpeakerVAE, "load_from_checkpoint", staticmethod(fake_load))
    with pytest.raises(FileNotFoundError):              # valid flags get as far as loading the checkpoint
        inference.main(base + ["--nearest_store", str(store), "--nearest_k", "16"])
    assert seen["path"].endswith("missing.ckpt")
