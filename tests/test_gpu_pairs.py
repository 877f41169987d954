"""Match lists on the GPU (ffr_match_pairs / ffr_match_pairs_self): the tensor-core path against the exact kernel (same pairs, same
bits), against the fp64 oracle, against the one-answer calls, overflow and retry, self mode's row splits, and the errors."""
import ctypes as C

import numpy as np
import pytest
import torch

from face_detection_and_recognition_b200 import _lib, ops
from face_detection_and_recognition_b200._lib import FLAG_FORCE_FP32, FLAG_FORCE_MMA, FLAG_NO_RECHECK, FfrError
from oracle import oracle_pairs

pytestmark = pytest.mark.gpu

THR = {"cosine": 0.5, "euclid": 2.0}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _unit(rng, n, dim):
    x = rng.standard_normal((n, dim))
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def _planted(rng, r, thr, metric, eps):
    """A candidate whose fp64 value against reference r is thr + eps (cosine) / thr * (1 + eps) (Euclid)."""
    u = rng.standard_normal(r.shape)
    rn = r / max(np.linalg.norm(r), 1e-30)
    u -= (u @ rn) * rn
    u /= np.linalg.norm(u)
    if metric == "cosine":
        t = thr + eps
        return np.linalg.norm(r) * (t * rn + np.sqrt(1 - t * t) * u)
    return r + thr * (1 + eps) * u


def _data(n_ref, n_cand, dim, metric, seed):
    """Unit rows (cosine) or rows scaled by 0.5..12 (Euclid); noisy copies; planted pairs at thr +- 2e-3 and +- 1e-5; groups of
    bit-identical references; a zero row among the references and among the candidates."""
    rng = np.random.default_rng(seed)
    thr = THR[metric]
    ref = _unit(rng, n_ref, dim)
    if metric == "euclid":
        ref *= rng.uniform(0.5, 12.0, (n_ref, 1))
    if n_ref >= 6:
        ref[n_ref - 3:] = ref[2]                              # three more copies of reference 2
    cand = _unit(rng, n_cand, dim) * (rng.uniform(0.5, 12.0, (n_cand, 1)) if metric == "euclid" else 1.0)
    k = rng.integers(0, n_ref, n_cand)
    noisy = rng.random(n_cand) < 0.4
    scale = 0.05 if metric == "euclid" else 0.03
    cand[noisy] = ref[k[noisy]] + scale * np.linalg.norm(ref[k[noisy]], axis=1, keepdims=True) * rng.standard_normal((noisy.sum(), dim))
    for j, eps in zip(range(1, min(n_cand, 41)), [2e-3, -2e-3, 1e-5, -1e-5] * 10):
        cand[j] = _planted(rng, ref[k[j]], thr, metric, eps)
    if n_ref >= 3:
        ref[1] = 0.0
    cand[0] = 0.0
    return ref.astype(np.float32), cand.astype(np.float32)


def _pairs_set(res):
    return set(zip(res.cand.tolist(), res.ref.tolist()))


def _value64(ref, cand, c, r, metric):
    a, b = cand[c].astype(np.float64), ref[r].astype(np.float64)
    if metric == "cosine":
        return a @ b / (np.linalg.norm(a) * np.linalg.norm(b))
    return np.linalg.norm(a - b)


def _band(v64, thr, metric, tol=1e-6):
    return abs(v64 - thr) <= (tol if metric == "cosine" else tol * thr)


def _check_oracle(res, ref, cand, thr, metric, rows=None, base=0):
    """Equal to the fp64 oracle's pair set except pairs within 1e-6 of thr (Euclid: relative); values within 1e-5."""
    if rows is None:
        oc, orf, ov = oracle_pairs.match_pairs(ref, cand, thr, metric, ref_index_base=base, dtype=np.float64)
        cands = cand
    else:
        oc, orf, ov = oracle_pairs.self_pairs(ref, thr, metric, rows=rows, dtype=np.float64)
        cands = ref[rows]
    got = _pairs_set(res)
    want = set(zip(oc.tolist(), orf.tolist()))
    for c, r in got ^ want:
        assert _band(_value64(ref, cands, c, r - base, metric), thr, metric), (c, r, c in got)
    o = dict(zip(zip(oc.tolist(), orf.tolist()), ov.tolist()))
    v = res.val.cpu().numpy().astype(np.float64)
    for (c, r), x in zip(zip(res.cand.tolist(), res.ref.tolist()), v):
        if (c, r) in o:
            assert abs(x - o[(c, r)]) <= (1e-5 if metric == "cosine" else 1e-5 * max(1.0, o[(c, r)])), (c, r, x, o[(c, r)])
    return got


def _check_one_answer(pairs, res, keep, idx, best, ref, cands, thr, metric):
    """A kept row has its (cand, best_idx) pair, a discarded row none -- outside the band; Euclid: that pair's value is best_val."""
    keep, idx, best = keep.cpu().numpy(), idx.cpu().numpy(), best.cpu().numpy()
    per_row = {}
    for (c, r), v in zip(zip(res.cand.tolist(), res.ref.tolist()), res.val.cpu().numpy()):
        per_row.setdefault(c, {})[r] = v
    for j in range(len(keep)):
        if idx[j] < 0:
            assert j not in per_row
            continue
        if _band(_value64(ref, cands, j, idx[j], metric), thr, metric, 1e-5):
            continue
        if keep[j]:
            assert (j, int(idx[j])) in pairs, j
            if metric == "euclid":
                assert per_row[j][int(idx[j])] == best[j]
        else:
            assert j not in per_row, j


SHAPES = [(1, 100, 128), (8, 300, 128), (9, 200, 130), (255, 300, 512), (256, 129, 128), (257, 600, 128), (300, 200, 640),
          (4100, 150, 512)]


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
@pytest.mark.parametrize("n_ref,n_cand,dim", SHAPES)
def test_match_pairs(dev, n_ref, n_cand, dim, metric):
    ref, cand = _data(n_ref, n_cand, dim, metric, seed=n_ref + dim)
    thr = THR[metric]
    r_t, c_t = torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev)
    res = ops.match_pairs(r_t, c_t, thr, metric, want_stats=True)
    exact = ops.match_pairs(r_t, c_t, thr, metric, flags=FLAG_FORCE_FP32, want_stats=True)
    mma = n_ref > 8 and dim <= 512
    assert res.stats["path"] == ("tcgen05" if mma else "fp32") and exact.stats["path"] == "fp32"
    assert torch.equal(res.cand, exact.cand) and torch.equal(res.ref, exact.ref)
    assert torch.equal(res.val.view(torch.int32), exact.val.view(torch.int32))         # bit for bit
    pairs = _check_oracle(res, ref, cand, thr, metric)
    assert len(pairs) > 0
    if mma:
        assert res.stats["raw_pairs"] >= len(pairs) - (n_ref if metric == "euclid" else 0)
    # every copy of a duplicated reference is listed; zero rows: no cosine pairs
    if n_ref >= 6:
        for c, r in pairs:
            if r == 2:
                assert all((c, d) in pairs for d in range(n_ref - 3, n_ref))
    if metric == "cosine":
        assert not any(c == 0 or (r == 1 and n_ref >= 3) for c, r in pairs)
    f = ops.face_filter(r_t, c_t, thr, metric)
    _check_one_answer(pairs, res, f.keep, f.best_idx, f.best_val, ref, cand, thr, metric)
    # reference indices carry ref_index_base
    shifted = ops.match_pairs(r_t, c_t, thr, metric, ref_index_base=1000)
    assert torch.equal(shifted.ref, res.ref + 1000) and torch.equal(shifted.val, res.val)


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
@pytest.mark.parametrize("n,rows", [(2, None), (9, None), (300, (37, 300)), (5000, (300, 4700))])
def test_self_pairs(dev, n, rows, metric):
    x, _ = _data(n, 1, 128, metric, seed=n)
    rng = np.random.default_rng(n)
    near = rng.choice(n, n // 3, replace=False)
    src = rng.integers(0, n, n // 3)
    if len(near):
        x[near] = x[src] + 0.03 * np.abs(x[src]).max() * rng.standard_normal((len(near), 128)).astype(np.float32)
    x[n // 2] = x[0]                                         # a bit-identical pair
    thr = THR[metric]
    x_t = torch.from_numpy(x).to(dev)
    res = ops.self_pairs(x_t, thr, metric, rows=rows, want_stats=True)
    exact = ops.self_pairs(x_t, thr, metric, rows=rows, flags=FLAG_FORCE_FP32)
    assert res.stats["path"] == ("tcgen05" if n > 8 else "fp32")
    assert torch.equal(res.cand, exact.cand) and torch.equal(res.ref, exact.ref)
    assert torch.equal(res.val.view(torch.int32), exact.val.view(torch.int32))
    b, e = (0, n) if rows is None else rows
    rr = np.arange(b, e)
    pairs = _check_oracle(res, x, None, thr, metric, rows=rr)
    assert all(r < b + c for c, r in pairs)
    if n <= 9:                                               # tiny sets: exact, not just outside the band
        oc, orf, _ = oracle_pairs.self_pairs(x, thr, metric, rows=rr, dtype=np.float64)
        assert pairs == set(zip(oc.tolist(), orf.tolist()))
    f = ops.self_filter(x_t, thr, metric, mode="earlier", rows=rows)
    _check_one_answer(pairs, res, f.keep, f.best_idx, f.best_val, x, x[rr], thr, metric)
    # the union over a split of the row range is the whole call
    mid = b + (e - b) // 2 + 3 if e - b > 8 else b + 1
    lo = ops.self_pairs(x_t, thr, metric, rows=(b, mid))
    hi = ops.self_pairs(x_t, thr, metric, rows=(mid, e))
    union = _pairs_set(lo) | {(c + mid - b, r) for c, r in _pairs_set(hi)}
    assert union == pairs


def _c_pairs(lib, ref, cand, thr, metric, cap, ws_extra=0, flags=0, base=0):
    dev = cand.device
    m = _lib.METRIC_EUCLID if metric == "euclid" else _lib.METRIC_COSINE
    n_ref, dim = ref.shape
    need = int(lib.ffr_match_pairs_workspace_bytes(n_ref, cand.shape[0], dim, m, cap))
    ws = torch.empty(need + ws_extra + 256, dtype=torch.uint8, device=dev)
    pc, pr = torch.empty(max(cap, 1), dtype=torch.int32, device=dev), torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    pv, cnt = torch.empty(max(cap, 1), dtype=torch.float32, device=dev), torch.full((1,), -7, dtype=torch.int64, device=dev)
    rc = lib.ffr_match_pairs(ref.data_ptr(), n_ref, cand.data_ptr(), cand.shape[0], dim, m, float(thr), base, pc.data_ptr(),
                             pr.data_ptr(), pv.data_ptr(), cap, cnt.data_ptr(), flags, ws.data_ptr(), need + ws_extra,
                             torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    return rc, int(cnt.item()), pc, pr, pv


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
def test_overflow_and_retry(dev, metric):
    lib = _lib.load()
    ref, cand = _data(700, 500, 256, metric, seed=7)
    thr = THR[metric] * (0.2 if metric == "cosine" else 4.0)          # many pairs
    r_t, c_t = torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev)
    full = ops.match_pairs(r_t, c_t, thr, metric, cap=10 ** 6)
    total = len(full.cand)
    assert total > 1000
    rc, cnt, *_ = _c_pairs(lib, r_t, c_t, thr, metric, 0)                 # cap 0: counts only
    assert rc == 0 and cnt >= total
    rc, cnt, *_ = _c_pairs(lib, r_t, c_t, thr, metric, 100)
    assert rc == 0 and cnt > 100
    rc, cnt2, pc, pr, pv = _c_pairs(lib, r_t, c_t, thr, metric, cnt)
    assert rc == 0 and cnt2 == total
    got = sorted(zip(pc[:cnt2].tolist(), pr[:cnt2].tolist(), pv[:cnt2].view(torch.int32).tolist()))
    assert got == list(zip(full.cand.tolist(), full.ref.tolist(), full.val.view(torch.int32).tolist()))
    small = ops.match_pairs(r_t, c_t, thr, metric, cap=50)                # the wrapper retries by itself
    assert torch.equal(small.cand, full.cand) and torch.equal(small.ref, full.ref) and torch.equal(small.val, full.val)


def test_threshold_that_matches_everything(dev):
    rng = np.random.default_rng(11)
    ref, cand = _unit(rng, 40, 64).astype(np.float32), _unit(rng, 70, 64).astype(np.float32)
    res = ops.match_pairs(torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), -1.0, cap=16, want_stats=True)
    assert res.stats["path"] == "tcgen05" and len(res.cand) == 40 * 70
    assert torch.equal(res.cand, torch.arange(70, device=dev).repeat_interleave(40))
    assert torch.equal(res.ref, torch.arange(40, device=dev).repeat(70))


def test_pairs_errors(dev):
    lib = _lib.load()
    rng = np.random.default_rng(12)
    ref = torch.from_numpy(_unit(rng, 64, 128).astype(np.float32)).to(dev)
    cand = torch.from_numpy(_unit(rng, 32, 128).astype(np.float32)).to(dev)
    with pytest.raises(FfrError) as e:
        ops.match_pairs(ref, cand, 0.5, flags=FLAG_NO_RECHECK)
    assert e.value.code == -4
    with pytest.raises(FfrError) as e:
        ops.self_pairs(ref, 0.5, flags=FLAG_NO_RECHECK)
    assert e.value.code == -4
    with pytest.raises(FfrError) as e:
        ops.match_pairs(ref[:8], cand, 0.5, flags=FLAG_FORCE_MMA)
    assert e.value.code == -4
    with pytest.raises(FfrError) as e:
        ops.self_pairs(ref[:8], 0.5, flags=FLAG_FORCE_MMA)
    assert e.value.code == -4
    assert ops.match_pairs(ref, cand, 0.5, flags=FLAG_FORCE_MMA, want_stats=True).stats["path"] == "tcgen05"
    for metric in ("cosine", "euclid"):
        rc, *_ = _c_pairs(lib, ref, cand, 0.5, metric, 100, ws_extra=-1)   # one byte short
        assert rc == -3
        rc, *_ = _c_pairs(lib, ref, cand, 0.5, metric, 100, base=2 ** 31 - 64)
        assert rc == -1
