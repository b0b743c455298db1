"""fp64 reference of ``psvae_cosine_topk`` / ``pseudo_speaker_vae_b200.cosine_topk`` (numpy, chunked over the queries).

sim(q, x) = q.x / (max(|q|, 1e-8) * max(|x|, 1e-8)), torch's ``F.cosine_similarity``.  For every query row the k best keys: descending
similarity (ascending with ``largest=False``), equal similarities to the lower key index, NaN similarities and (with ``exclude_self``) the
pairs ``query_row0 + i == key_row0 + j`` never chosen, slots without a candidate -1 / NaN.  Indices are global (``key_row0 + j``)."""
from __future__ import annotations

import numpy as np


def unit_rows(x) -> np.ndarray:
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        n = np.sqrt((x * x).sum(axis=1, keepdims=True))
        return x / np.where(np.isnan(n), n, np.maximum(n, 1e-8))


def cosine_sim(q, x) -> np.ndarray:
    """fp64 [Nq, Nk] similarity matrix."""
    with np.errstate(invalid="ignore", over="ignore"):
        return unit_rows(q) @ unit_rows(x).T


def cosine_topk(q, keys, k: int = 1, largest: bool = True, exclude_self: bool = False, query_row0: int = 0, key_row0: int = 0,
                chunk: int = 4096):
    """(similarity fp64 [Nq, k], index int64 [Nq, k]) by the ordering rules above."""
    uq, uk = unit_rows(q), unit_rows(keys)
    nq, nk = uq.shape[0], uk.shape[0]
    sim = np.full((nq, k), np.nan)
    idx = np.full((nq, k), -1, dtype=np.int64)
    cols = np.arange(nk)
    for a in range(0, nq, chunk):
        b = min(nq, a + chunk)
        with np.errstate(invalid="ignore", over="ignore"):
            s = uq[a:b] @ uk.T
        bad = np.isnan(s)
        if exclude_self:
            bad |= (query_row0 + np.arange(a, b))[:, None] == (key_row0 + cols)[None, :]
        key = np.where(bad, np.inf, -s if largest else s)
        order = np.argsort(key, axis=1, kind="stable")[:, :k]          # stable: equal scores keep the lower index first
        take = np.take_along_axis(key, order, axis=1)
        ok = np.isfinite(take)
        sim[a:b] = np.where(ok, np.take_along_axis(s, order, axis=1), np.nan)
        idx[a:b] = np.where(ok, key_row0 + order, -1)
    return sim, idx
