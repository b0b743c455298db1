"""Cosine top-k search between two embedding sets on the device (``psvae_cosine_topk``).

Two questions users ask of a pseudo-speaker population are cosine searches: which real training speaker is closest to each
pseudo-speaker (a memorisation / privacy check), and which pool entries are the most or least similar to a source speaker (selection
and evaluation).  ``cosine_topk`` answers both without materialising the similarity matrix: candidates are selected on the tensor
cores from bf16 unit vectors, the best 2k per row are re-scored in fp32 from the inputs, and the best k are returned.

Ordering rules: descending similarity (ascending with ``largest=False``), equal similarities to the lower key index, a NaN similarity
never chosen, a slot without any candidate ``-1`` / NaN.  A zero vector scores 0 (``F.cosine_similarity``'s definition).  The result is
bit-identical from run to run and for any sharding of the queries (``shard_rows`` + ``query_row0``).
"""
from __future__ import annotations

from typing import Tuple

import torch
from torch import Tensor

from . import _lib as L

#: queries per library call: bounds the workspace (unit bf16 copies, inverse norms and candidate lists of one chunk)
CHUNK_ROWS = 1 << 20

_DTYPES = {torch.float32: L.X_F32, torch.bfloat16: L.X_BF16}


def _check(queries: Tensor, keys: Tensor, k: int, exclude_self: bool, query_row0: int, key_row0: int) -> None:
    for name, t in (("queries", queries), ("keys", keys)):
        if not isinstance(t, Tensor):
            raise TypeError(f"{name} must be a torch.Tensor")
        if t.dim() != 2:
            raise ValueError(f"{name} must be [N, D], got shape {tuple(t.shape)}")
        if t.dtype not in _DTYPES:
            raise ValueError(f"{name} must be float32 or bfloat16, got {t.dtype}")
    nq, d = queries.shape
    nk, dk = keys.shape
    if d != dk:
        raise ValueError(f"queries have D={d}, keys D={dk}")
    if d <= 0 or d % 8 != 0 or d > L.TOPK_MAX_DIM:
        raise ValueError(f"D={d}: must be a positive multiple of 8, at most {L.TOPK_MAX_DIM}")
    if not 1 <= int(k) <= L.TOPK_MAX_K:
        raise ValueError(f"k={k} out of range [1, {L.TOPK_MAX_K}]")
    avail = nk - (1 if exclude_self else 0)
    if int(k) > avail:
        raise ValueError(f"k={k} exceeds the {avail} keys available" + (" (exclude_self)" if exclude_self else ""))
    if nq == 0:
        raise ValueError("queries must have at least one row")
    if query_row0 < 0 or key_row0 < 0:
        raise ValueError("query_row0 and key_row0 must be >= 0")
    if queries.device != keys.device:
        raise ValueError(f"queries on {queries.device}, keys on {keys.device}: both must be on the same CUDA device")
    if queries.device.type != "cuda":
        raise RuntimeError(f"cosine_topk runs on a CUDA (B200) device only; the inputs are on {queries.device}")


def cosine_topk(queries: Tensor, keys: Tensor, k: int = 1, *, largest: bool = True, exclude_self: bool = False, query_row0: int = 0,
                key_row0: int = 0) -> Tuple[Tensor, Tensor]:
    """The ``k`` keys of highest (``largest=False``: lowest) cosine similarity to every query row.

    ``queries`` [Nq, D] and ``keys`` [Nk, D] are float32 or bfloat16 tensors on one CUDA device (they may be the same tensor); D is a
    multiple of 8 up to 512 and 1 <= k <= 16.  Returns device tensors ``(similarity float32 [Nq, k], index int64 [Nq, k])``; indices are
    global, ``key_row0 + j``.  With ``exclude_self`` the pairs whose global indices ``query_row0 + i`` and ``key_row0 + j`` are equal are
    skipped, so a set can search itself, also when its queries are sharded.  Runs on the current stream without a host synchronisation."""
    _check(queries, keys, k, exclude_self, query_row0, key_row0)
    k = int(k)
    queries = queries.contiguous()
    keys = keys.contiguous()
    nq, d = queries.shape
    nk = keys.shape[0]
    dev = queries.device
    sim = torch.empty(nq, k, dtype=torch.float32, device=dev)
    idx = torch.empty(nq, k, dtype=torch.int64, device=dev)
    flags = (L.TOPK_SMALLEST if not largest else 0) | (L.TOPK_EXCLUDE_SELF if exclude_self else 0)
    lib = L.lib()
    chunk = min(nq, CHUNK_ROWS)
    # the split of the key range, and with it the candidate-list area, depends on the chunk's rows: size for the full and the last chunk
    sizes = [int(lib.psvae_cosine_topk_workspace_bytes(n, nk, d, k)) for n in {chunk, nq - (nq - 1) // chunk * chunk}]
    if min(sizes) < 0:
        raise ValueError(L.last_error())
    ws_bytes = max(sizes)
    with torch.cuda.device(dev):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        for a in range(0, nq, chunk):
            b = min(nq, a + chunk)
            L.check(lib.psvae_cosine_topk(queries[a:b].data_ptr(), _DTYPES[queries.dtype], b - a, int(query_row0) + a, keys.data_ptr(),
                                          _DTYPES[keys.dtype], nk, int(key_row0), d, k, flags, sim[a:b].data_ptr(), idx[a:b].data_ptr(),
                                          ws.data_ptr(), ws_bytes, stream), "psvae_cosine_topk")
    return sim, idx
