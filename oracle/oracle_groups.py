"""CPU oracle of the near-duplicate groups (``ffr_self_groups``): the connected components of the graph whose edges are
``oracle_pairs.self_pairs``, each row labelled with the smallest row of its component.  TEST INFRASTRUCTURE ONLY, like
``oracle.py``; NumPy alone (no graph library)."""
from __future__ import annotations

from typing import Tuple

import numpy as np

from .oracle_pairs import self_pairs


def components(n: int, a, b) -> np.ndarray:
    """Min-index component labels of the graph on rows [0, n) with edges (a[k], b[k]): int64 [n].  A vectorised union-find: every
    round hooks the larger root of each edge whose endpoints lie in different trees under the smaller one, then compresses the
    paths fully.  A parent is never larger than its child, so each root is its tree's minimum."""
    lab = np.arange(n, dtype=np.int64)
    a = np.asarray(a, dtype=np.int64)
    b = np.asarray(b, dtype=np.int64)
    while True:
        ra, rb = lab[a], lab[b]
        cross = ra != rb
        if not cross.any():
            return lab
        lo, hi = np.minimum(ra[cross], rb[cross]), np.maximum(ra[cross], rb[cross])
        np.minimum.at(lab, hi, lo)
        while True:                                          # full path compression
            nxt = lab[lab]
            if np.array_equal(nxt, lab):
                break
            lab = nxt


def self_groups(x: np.ndarray, thr: float, metric="cosine", block: int = 2048, dtype=np.float32) -> Tuple[np.ndarray, int]:
    """Groups of the rows of ``x``: (labels int64 [n], number of groups).  ``dtype=np.float64`` gives the fp64 shadow."""
    x = np.asarray(x)
    c, r, _ = self_pairs(x, thr, metric, block=block, dtype=dtype)
    lab = components(x.shape[0], c, r)
    return lab, int((lab == np.arange(x.shape[0])).sum())
