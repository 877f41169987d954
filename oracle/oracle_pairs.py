"""CPU oracle of the match lists (``ffr_match_pairs`` / ``ffr_match_pairs_self``): every (candidate, reference) pair on the
matching side of the threshold.  TEST INFRASTRUCTURE ONLY, like ``oracle.py``: a blocked NumPy restatement with
``oracle.filter_cosine`` / ``oracle.filter_euclid``'s arithmetic -- normalised rows and a matmul for cosine (as ``oracle_self``),
direct differences for Euclid -- that keeps every pair instead of each candidate's best."""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .oracle import METRIC_COSINE


def _normalise(x: np.ndarray, dtype) -> np.ndarray:
    with np.errstate(divide="ignore", invalid="ignore"):       # zero rows: NaN similarities, never a cosine pair
        return x / np.sqrt(np.einsum("ij,ij->i", x, x, dtype=dtype))[:, None].astype(dtype)


def _pairs(ref, cand, thr, metric, ref_end, block, dtype) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    cos = metric in ("cosine", METRIC_COSINE)
    ref = np.asarray(ref, dtype=dtype)
    cand = np.asarray(cand, dtype=dtype)
    n, m = ref.shape[0], cand.shape[0]
    rn = _normalise(ref, dtype) if cos else None
    step = block if cos else max(1, (block << 12) // max(1, n * ref.shape[1]))   # Euclid: [step, N, D] differences per block
    out_c, out_r, out_v = [], [], []
    for s in range(0, m, step):
        c = cand[s:s + step]
        if cos:
            val = _normalise(c, dtype) @ rn.T                               # [b, N]
            with np.errstate(invalid="ignore"):
                hit = val >= dtype(thr)
        else:
            diff = c[:, None, :] - ref[None, :, :]                          # [b, N, D]: direct differences
            val = np.sqrt(np.einsum("bnd,bnd->bn", diff, diff, dtype=dtype))
            hit = val <= dtype(thr)
        if ref_end is not None:                                             # self: references i < the candidate's row only
            hit &= np.arange(n)[None, :] < ref_end[s:s + step, None]
        ci, ri = np.nonzero(hit)                                            # row-major: sorted by (cand, ref)
        out_c.append(ci + s)
        out_r.append(ri)
        out_v.append(val[ci, ri])
    if not out_c:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, dtype)
    return (np.concatenate(out_c).astype(np.int64), np.concatenate(out_r).astype(np.int64),
            np.concatenate(out_v).astype(dtype))


def match_pairs(ref: np.ndarray, cand: np.ndarray, thr: float, metric="cosine", ref_index_base: int = 0, block: int = 2048,
                dtype=np.float32) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Gallery form: every pair with ``(r.c)/(|r||c|) >= thr`` (cosine) / ``|c - r| <= thr`` (Euclid).  Returns (cand i64[P],
    ref i64[P] + ref_index_base, value[P]) sorted by (cand, ref); ``dtype=np.float64`` gives the fp64 shadow."""
    c, r, v = _pairs(ref, cand, thr, metric, None, block, dtype)
    return c, r + ref_index_base, v


def self_pairs(x: np.ndarray, thr: float, metric="cosine", rows=None, block: int = 2048,
               dtype=np.float32) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Self form: candidate rows ``rows`` (global indices, default all) of ``x`` against the rows i < j of ``x``.  Returns
    (position in ``rows`` i64[P], global reference row i64[P], value[P]) sorted by (cand, ref)."""
    x = np.asarray(x)
    rows = np.arange(x.shape[0]) if rows is None else np.asarray(rows, dtype=np.int64)
    return _pairs(x, x[rows], thr, metric, rows, block, dtype)
