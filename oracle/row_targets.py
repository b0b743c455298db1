"""TEST INFRASTRUCTURE ONLY -- fp64 reference for per-row classifier targets and in-kernel target mixes.

The reference samples with one classifier target per call.  A per-row call is, row for row, that loop run on the group of rows that
share a target, so the reference here groups rows by target and runs ``ps_vae_oracle.langevin`` / ``latent_transformation`` per group.
A target mix draws each row's entry from one uint32 Philox word (``philox_ref.philox_uint32``) compared against integer thresholds.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import numpy as np

from oracle import philox_ref
from oracle import ps_vae_oracle as O


def _target_key(t):
    return tuple(sorted(t.items())) if isinstance(t, dict) else int(t)


def langevin_rows(params, z0: np.ndarray, noises: Sequence[np.ndarray], targets: Sequence, step_size: float = 0.01, noise_weight: float = 1.0,
                  activation: str = "relu", return_history: bool = False, transform: Optional[dict] = None):
    """Per-row targets: ``targets[i]`` is row i's target (an int, or a dict of label -> class naming the heads it uses).  Rows are grouped by
    target and each group runs ``langevin`` (or, with ``transform = dict(prior_weight=, threshold=)``, ``latent_transformation``) on its rows
    of ``z0`` and of every noise.  Returns what those return, reassembled in row order: ``z`` (and the history), or ``(z, stop, prob)``."""
    N = z0.shape[0]
    groups: Dict = {}
    for i, t in enumerate(targets):
        groups.setdefault(_target_key(t), (t, []))[1].append(i)
    z = np.empty_like(z0)
    hist = [np.empty_like(z0) for _ in noises] if return_history else None
    stop = np.empty(N, dtype=np.int64)
    prob = np.empty(N, dtype=z0.dtype)
    for t, rows in groups.values():
        idx = np.asarray(rows)
        sub = [n[idx] for n in noises]
        if transform is not None:
            z[idx], stop[idx], prob[idx] = O.latent_transformation(params, z0[idx], sub, t, step_size, noise_weight, activation=activation, **transform)
            continue
        out = O.langevin(params, z0[idx], sub, t, step_size, noise_weight, activation, return_history)
        if return_history:
            z[idx] = out[0]
            for h, g in zip(hist, out[1]):
                h[idx] = g
        else:
            z[idx] = out
    if transform is not None:
        return z, stop, prob
    return (z, hist) if return_history else z


def draw_target_mix(thresholds: Sequence[int], n: int, seed: int, offset: int, row0: int = 0) -> np.ndarray:
    """The mix entry each of rows row0 .. row0 + n - 1 draws: u = word row0 + r of the uint32 Philox stream at ``offset``, entry = the first
    k < len(thresholds) with u < thresholds[k], else len(thresholds).  Integer comparisons only, so it matches the kernel bit for bit."""
    u = philox_ref.philox_uint32(n, seed, offset, first_elem=row0).astype(np.uint64)
    return np.searchsorted(np.asarray(thresholds, dtype=np.uint64), u, side="right").astype(np.int64)
