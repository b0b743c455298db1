"""Cosine top-k search on the GPU (-m gpu) against the fp64 reference (oracle/cosine_topk.py).

Every returned similarity is within 1e-6 of the fp64 value of its pair.  The candidates come from bf16 unit vectors, whose score error
is at most 2^-8 * sum_i |u_i v_i| <= 2^-8 plus the fp32 accumulation (BF16_BOUND); so the index set must equal the reference's on every
row whose rank-k and rank-(2k+1) similarities are more than twice that apart (and whose rank k and k+1 are not an fp32 tie).  Results
are bit-identical across runs, query shards and key-range splits."""
import numpy as np
import pytest
import torch

from oracle import cosine_topk as R

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SIM_TOL = 1e-6
BF16_BOUND = 2.0 ** -8 + 2.0 ** -16 + 512 * 2.0 ** -24


def _P():
    import pseudo_speaker_vae_b200 as P

    return P


def _data(n, d, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, d, generator=g)
    return x.to(dtype)


def _check_against_oracle(q, x, k, largest=True, exclude_self=False, min_share=0.5):
    sim, idx = _P().cosine_topk(q.to(DEV), x.to(DEV), k, largest=largest, exclude_self=exclude_self)
    sim, idx = sim.cpu().numpy(), idx.cpu().numpy()
    qn, xn = q.double().numpy(), x.double().numpy()
    nk = x.shape[0]
    kk = min(2 * k + 1, nk - (1 if exclude_self else 0))
    rs, ri = R.cosine_topk(qn, xn, kk, largest=largest, exclude_self=exclude_self)
    assert (idx >= 0).all()
    # every returned similarity is that pair's fp64 similarity
    uq, ux = R.unit_rows(qn), R.unit_rows(xn)
    pair = np.einsum("ij,ikj->ik", uq, ux[idx])
    assert np.abs(sim - pair).max() <= SIM_TOL
    sgn = 1.0 if largest else -1.0
    assert (np.diff(sgn * sim, axis=1) <= SIM_TOL).all()           # in order
    if exclude_self:
        assert (idx != np.arange(q.shape[0])[:, None]).all()
    # rows where the bf16 selection cannot have missed a member of the true top k
    sep = np.ones(q.shape[0], bool)
    if kk > k:
        sep &= sgn * (rs[:, k - 1] - rs[:, kk - 1]) > 2 * BF16_BOUND
        sep &= sgn * (rs[:, k - 1] - rs[:, k]) > 4 * SIM_TOL
    got = np.sort(idx, axis=1)
    want = np.sort(ri[:, :k], axis=1)
    assert np.array_equal(got[sep], want[sep])
    assert sep.mean() >= min_share, sep.mean()
    return sim, idx


@pytest.mark.parametrize("d", [64, 192, 256, 512])
@pytest.mark.parametrize("k", [1, 5, 16])
def test_against_the_oracle(d, k):
    q = _data(1000, d, seed=d + k)
    x = _data(4099, d, seed=1000 + d + k)
    for largest in (True, False):
        _check_against_oracle(q, x, k, largest=largest)


@pytest.mark.parametrize("nq,nk", [(1, 127), (127, 129), (129, 1), (4099, 300007)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ragged_shapes_and_dtypes(nq, nk, dtype):
    k = min(5, nk)
    q = _data(nq, 256, seed=nq, dtype=dtype)
    x = _data(nk, 256, seed=nk + 1, dtype=dtype)
    if nk > 100000:
        q = q[:257]
    _check_against_oracle(q, x, k, min_share=0.3 if nk > 100000 else 0.5)


def test_mixed_dtypes():
    q = _data(300, 192, seed=3)
    x = _data(2000, 192, seed=4, dtype=torch.bfloat16)
    _check_against_oracle(q, x, 3)
    _check_against_oracle(q.to(torch.bfloat16), x.float(), 3)


def test_planted_duplicates_are_found():
    x = _data(5000, 256, seed=5)
    plant = [3, 1234, 4990, 4999]                         # the last two in the last, partial key tile (5000 = 19 * 256 + 136)
    q = _data(64, 256, seed=6)
    for j, p in enumerate(plant):
        q[j] = x[p] * (j + 1.5)                            # a scaled copy: similarity 1
        q[10 + j] = x[p] + 1e-4 * torch.randn(256, generator=torch.Generator().manual_seed(j))
    sim, idx = _P().cosine_topk(q.to(DEV), x.to(DEV), 2)
    sim, idx = sim.cpu(), idx.cpu()
    for j, p in enumerate(plant):
        assert idx[j, 0] == p and sim[j, 0] >= 1 - 1e-6
        assert idx[10 + j, 0] == p and sim[10 + j, 0] >= 1 - 1e-6


def test_exclude_self_and_duplicate_keys():
    x = _data(3000, 128, seed=7)
    x[2500] = x[17]
    x[2999] = x[17]
    sim, idx = _check_against_oracle(x, x, 4, exclude_self=True)
    assert idx[17, 0] == 2500 and idx[17, 1] == 2999 and idx[2500, 0] == 17 and idx[2999, :2].tolist() == [17, 2500]
    # without exclude_self a row finds itself, and duplicate keys resolve to the lower index
    sim, idx = _P().cosine_topk(x.to(DEV), x.to(DEV), 2)
    idx = idx.cpu()
    assert (idx[:, 0] == torch.arange(3000)).sum() >= 2998
    assert idx[2500].tolist() == [17, 2500] and idx[2999].tolist() == [17, 2500]


def test_zero_and_nan_rows():
    x = _data(600, 64, seed=8)
    x[5] = 0.0
    x[300, 7] = float("nan")
    q = _data(40, 64, seed=9)
    q[0] = 0.0
    q[1, 3] = float("nan")
    sim, idx = _P().cosine_topk(q.to(DEV), x.to(DEV), 16)
    sim, idx = sim.cpu(), idx.cpu()
    assert (idx != 300).all()                             # NaN key never preferred
    assert (idx[1] == -1).all() and torch.isnan(sim[1]).all()      # a NaN query has no candidate: -1 / NaN slots
    assert (sim[0] == 0).all() and idx[0].tolist() == [j for j in range(17) if j != 300][:16]     # zero query: all score 0, lowest indices
    lo, li = _P().cosine_topk(q.to(DEV), x.to(DEV), 1, largest=False)
    assert (li.cpu() != 300).all()
    # the zero key scores 0
    s0, i0 = _P().cosine_topk(x[5:6].to(DEV), x.to(DEV), 1)
    assert s0.item() == 0.0 and i0.item() == 0
    # unfillable slots: a NaN key among 3 keys with k = 3
    s, i = _P().cosine_topk(q[:4].to(DEV), x[299:302].to(DEV), 3, key_row0=299)
    assert (i[:, 2].cpu() == -1).all() and torch.isnan(s[:, 2].cpu()).all()
    assert set(i[2, :2].cpu().tolist()) == {299, 301}


def test_bit_identical_across_runs_shards_and_splits():
    from pseudo_speaker_vae_b200 import _lib as L

    P = _P()
    q = _data(3001, 256, seed=10).to(DEV)
    x = _data(20000, 256, seed=11).to(DEV)
    ref = P.cosine_topk(q, x, 7)
    again = P.cosine_topk(q, x, 7)
    assert torch.equal(ref[0], again[0]) and torch.equal(ref[1], again[1])
    for shards in (2, 3, 8):
        parts = []
        for r in range(shards):
            a, n = P.shard_rows(q.shape[0], r, shards)
            parts.append(P.cosine_topk(q[a:a + n], x, 7, query_row0=a))
        assert torch.equal(torch.cat([p[0] for p in parts]), ref[0]) and torch.equal(torch.cat([p[1] for p in parts]), ref[1])
    try:
        for splits in (1, 2, 7):
            L.set_option("topk_key_splits", splits)
            got = P.cosine_topk(q, x, 7)
            assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), splits
            got = P.cosine_topk(q[:300], x, 7, largest=False, exclude_self=True)
            if splits == 1:
                small = got
            else:
                assert torch.equal(got[0], small[0]) and torch.equal(got[1], small[1]), splits
    finally:
        L.set_option("topk_key_splits", 0)
    auto = P.cosine_topk(q[:300], x, 7, largest=False, exclude_self=True)
    assert torch.equal(auto[0], small[0]) and torch.equal(auto[1], small[1])
    # sharded self-search with exclude_self
    ex = P.cosine_topk(x, x, 3, exclude_self=True)
    a, n = P.shard_rows(x.shape[0], 1, 3)
    part = P.cosine_topk(x[a:a + n], x, 3, exclude_self=True, query_row0=a)
    assert torch.equal(part[1], ex[1][a:a + n]) and torch.equal(part[0], ex[0][a:a + n])


def test_side_stream_without_host_sync():
    P = _P()
    q = _data(2000, 256, seed=12).to(DEV)
    x = _data(9000, 256, seed=13).to(DEV)
    ref = P.cosine_topk(q, x, 4)
    s = torch.cuda.Stream(DEV)
    s.wait_stream(torch.cuda.current_stream(DEV))
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.cuda.stream(s):
            got = P.cosine_topk(q, x, 4)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.current_stream(DEV).wait_stream(s)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])


def test_cli_nearest_store(tmp_path):
    P = _P()
    from pseudo_speaker_vae_b200 import inference

    torch.manual_seed(0)
    m = P.PseudoSpeakerVAE(model=dict(input_dim=256, latent_dim=64), optimizer={}, scheduler=dict(T_max=1))
    ckpt = str(tmp_path / "m.ckpt")
    torch.save({"state_dict": m.state_dict(), "hyper_parameters": dict(m.hparams)}, ckpt)
    store = P.PackedEmbeddingStore.from_arrays(str(tmp_path / "store"), _data(5000, 256, seed=14), dtype="bf16")
    out = tmp_path / "out"
    inference.main(["--vae_ckpt_path", ckpt, "--save_dir", str(out), "--synthesis_type", "unconditional", "--n_samples", "300",
                    "--nearest_store", store.root, "--nearest_k", "3", "--device", DEV])
    near = torch.load(out / "nearest.pt")
    assert near["index"].dtype == torch.int64 and near["index"].shape == (300, 3) and near["similarity"].dtype == torch.float32
    x_hat = torch.stack([torch.load(out / P.sample_filename(i)) for i in range(300)])
    sim, idx = P.cosine_topk(x_hat.to(DEV), store.to_device(DEV)[0], 3)
    assert torch.equal(near["index"], idx.cpu()) and torch.equal(near["similarity"], sim.cpu())
