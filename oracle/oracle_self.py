"""CPU oracle of the self filter (``ffr_filter_self``): each row's best match among the OTHER rows of the same set.  TEST
INFRASTRUCTURE ONLY, like ``oracle.py``: a blocked NumPy restatement of ``oracle.filter_cosine`` / ``oracle.filter_euclid``
on the masked score matrix.  Neither the reference nor the gallery filter defines this question; the masking rule is the one
``include/ffr.h`` documents."""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .oracle import METRIC_COSINE

SELF_OTHERS = 0
SELF_EARLIER = 1


def filter_self(x: np.ndarray, thr: float, metric="cosine", mode="others", rows=None, block: int = 2048,
                dtype=np.float32) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Self filter: every row j of ``x`` (or of ``rows``, global row indices) against the OTHER rows of ``x`` -- all i != j
    (``mode="others"``) or i < j (``"earlier"``) -- with ``filter_cosine`` / ``filter_euclid``'s arithmetic on the masked
    score matrix: first arg-best, ``keep = best >= thr`` (cosine) / ``<= thr`` (Euclid).  A row with no eligible reference
    gets keep 0, index -1 and -inf (cosine) / +inf (Euclid).  Returns (keep u8, best_idx i32, best f32) per row of ``rows``;
    ``dtype=np.float64`` gives the fp64 shadow."""
    cos = metric in ("cosine", METRIC_COSINE)
    earlier = mode in ("earlier", SELF_EARLIER)
    x = np.asarray(x, dtype=dtype)
    n = x.shape[0]
    rows = np.arange(n) if rows is None else np.asarray(rows, dtype=np.int64)
    m = len(rows)
    best = np.empty(m, dtype=dtype)
    idx = np.empty(m, dtype=np.int32)
    if cos:
        xn = x / np.sqrt(np.einsum("ij,ij->i", x, x, dtype=dtype))[:, None].astype(dtype)
        step = block
    else:
        step = max(1, (block << 12) // (n * x.shape[1]))       # [step, N, D] differences: ~8 M elements per block
    bad = np.inf if not cos else -np.inf
    for s in range(0, m, step):
        g = rows[s:s + step]
        if cos:
            sc = xn[g] @ xn.T                                      # [b, N]
        else:
            diff = x[g][:, None, :] - x[None, :, :]                # [b, N, D]: direct differences
            sc = np.sqrt(np.einsum("bnd,bnd->bn", diff, diff, dtype=dtype))
        col = np.arange(n)[None, :]
        masked = (col >= g[:, None]) if earlier else (col == g[:, None])
        sc = np.where(masked, bad, sc)
        i = np.argmax(sc, axis=1) if cos else np.argmin(sc, axis=1)     # first occurrence
        none = masked.all(axis=1)
        idx[s:s + step] = np.where(none, -1, i)
        best[s:s + step] = np.where(none, bad, sc[np.arange(len(g)), i])
    keep = ((best >= dtype(thr)) if cos else (best <= dtype(thr))) & (idx >= 0)
    return keep.astype(np.uint8), idx, best.astype(dtype)
