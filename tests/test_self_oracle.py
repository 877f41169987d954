"""oracle_self.filter_self against a brute-force masked argmax / argmin, and the self-mode workspace query (no GPU needed)."""
import numpy as np
import pytest

from oracle.oracle_self import filter_self


def _brute(x, thr, metric, mode, rows):
    x64 = x.astype(np.float64)
    keep, idx, best = [], [], []
    for j in rows:
        cand = [i for i in range(len(x)) if (i < j if mode == "earlier" else i != j)]
        if not cand:
            keep.append(0), idx.append(-1), best.append(-np.inf if metric == "cosine" else np.inf)
            continue
        if metric == "cosine":
            s = [x64[i] @ x64[j] / (np.linalg.norm(x64[i]) * np.linalg.norm(x64[j])) for i in cand]
            k = int(np.argmax(s))
            keep.append(int(s[k] >= thr))
        else:
            s = [np.linalg.norm(x64[i] - x64[j]) for i in cand]
            k = int(np.argmin(s))
            keep.append(int(s[k] <= thr))
        idx.append(cand[k]), best.append(s[k])
    return np.array(keep), np.array(idx), np.array(best)


@pytest.mark.parametrize("metric,thr", [("cosine", 0.5), ("euclid", 1.0)])
@pytest.mark.parametrize("mode", ["others", "earlier"])
@pytest.mark.parametrize("n", [1, 2, 7, 40])
def test_filter_self_matches_brute_force(n, mode, metric, thr):
    rng = np.random.default_rng(n)
    x = rng.standard_normal((n, 16)).astype(np.float32)
    if n > 4:
        x[n - 1] = x[1]                                   # a bit-identical copy is found, not folded
        x[n - 2] = x[0] + 0.01 * rng.standard_normal(16).astype(np.float32)
    rows = np.arange(n)
    k, i, b = filter_self(x, thr, metric, mode)
    kb, ib, bb = _brute(x, thr, metric, mode, rows)
    assert np.array_equal(i, ib)
    assert np.array_equal(k, kb)
    fin = np.isfinite(bb)
    assert np.array_equal(np.isinf(b), ~fin)
    assert np.allclose(b[fin], bb[fin], rtol=1e-5, atol=1e-6)
    if n > 4 and mode == "earlier":
        assert i[n - 1] == 1 and i[n - 2] == 0
    # a row subset gives the same rows' answers
    sub = np.array([n - 1, 0, n // 2])
    ks, is_, _ = filter_self(x, thr, metric, mode, rows=sub)
    assert np.array_equal(is_, i[sub]) and np.array_equal(ks, k[sub])


def test_filter_self_fp64_shadow():
    x = np.random.default_rng(3).standard_normal((30, 8)).astype(np.float32)
    _, i32, b32 = filter_self(x, 0.5, "cosine", "others")
    _, i64, b64 = filter_self(x, 0.5, "cosine", "others", dtype=np.float64)
    assert b64.dtype == np.float64 and np.array_equal(i32, i64) and np.allclose(b32, b64, atol=1e-6)


def test_self_workspace_query(ffr_lib):
    ws = ffr_lib.ffr_filter_self_workspace_bytes
    assert ws(0, 0, 128, 0) == 0 and ws(10, -1, 128, 0) == 0 and ws(10, 10, 0, 0) == 0
    # <= 8 rows or dim > 512: the CUDA-core kernel, header only
    assert ws(8, 8, 128, 0) == 256 and ws(1000, 1000, 640, 1) == 256
    # tcgen05: cosine needs no fp16 copy of the candidates (they are a slice of x's), Euclid does (its A operand differs)
    cos, euc = ws(1000, 1000, 128, 0), ws(1000, 1000, 128, 1)
    assert cos >= 256 + 1000 * 128 * 2 and euc >= cos + 1000 * 128 * 2
    assert ws(1000, 10, 128, 0) < cos                       # per-candidate lists scale with the row range
    # smaller than the gallery call of the same shape, which also sizes the duplicate fold and the candidates' fp16 rows
    assert cos <= ffr_lib.ffr_filter_workspace_bytes(1000, 1000, 128, 0, 0)
