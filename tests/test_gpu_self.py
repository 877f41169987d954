"""Self mode: each row's best match among the OTHER rows of the same set (ffr_filter_self / ops.self_filter).

Bars (DESIGN.md section 5, applied to the masked problem): cosine best_val within 1e-3 of oracle_self.filter_self, best_idx equal
except where the two leading fp64 scores differ by < 1e-6, keep equal except |best64 - thr| < 1e-6.  Euclid: best_idx equal to the
FFR_FLAG_FORCE_FP32 self result (K2s) except on fp32 ties (two smallest fp64 distances within 1e-6 relative), keep and best_val
bit-identical to it wherever best_idx agrees, and the oracle bars with distances within 1e-3 relative.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle.oracle_self import filter_self

pytestmark = pytest.mark.gpu

TIE = 1e-6
THR = {"cosine": 0.8, "euclid": 0.9}


@pytest.fixture(scope="module")
def ops(ffr_lib, cuda_dev):
    from face_detection_and_recognition_b200 import ops as _ops
    return _ops


def make_set(n, dim, metric, seed, n_near=None, n_copy=None):
    """Unit-norm random rows; some rows are noisy copies of an EARLIER row within +-2e-3 of the threshold (cosine: the score,
    Euclid: the distance), some are bit-identical copies of an earlier row."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    if n < 3:
        return x
    n_near = n // 8 if n_near is None else n_near
    n_copy = n // 16 if n_copy is None else n_copy
    js = rng.choice(np.arange(1, n), min(n - 1, n_near + n_copy), replace=False)
    for t, j in enumerate(js):
        k = int(rng.integers(0, j))
        if t >= n_near:
            x[j] = x[k]
            continue
        g = rng.standard_normal(dim)
        g -= (g @ x[k]) * x[k]
        g /= np.linalg.norm(g)
        u = rng.uniform(-2e-3, 2e-3)
        if metric == "cosine":
            c = THR["cosine"] + u
            x[j] = c * x[k] + np.sqrt(1 - c * c) * g
        else:
            x[j] = x[k] + g * THR["euclid"] * (1 + u)
    return x.astype(np.float32)


def top2_64(x, rows, metric, mode):
    """fp64 shadow of the two leading masked scores per row (cosine: largest, Euclid: smallest distance)."""
    x64 = x.astype(np.float64)
    n = len(x)
    out1, out2 = np.empty(len(rows)), np.empty(len(rows))
    nrm = np.sqrt(np.einsum("ij,ij->i", x64, x64))
    for s in range(0, len(rows), 1024):
        g = rows[s:s + 1024]
        dots = x64[g] @ x64.T
        if metric == "cosine":
            sc = -(dots / (nrm[g][:, None] * nrm[None, :]))
        else:
            sc = np.sqrt(np.maximum(nrm[g][:, None] ** 2 + nrm[None, :] ** 2 - 2 * dots, 0.0))
        col = np.arange(n)[None, :]
        sc[(col >= g[:, None]) if mode == "earlier" else (col == g[:, None])] = np.inf
        if n >= 3:
            p = np.partition(sc, 1, axis=1)
            a, b = p[:, 0], p[:, 1]
        else:
            a, b = sc.min(axis=1), np.full(len(g), np.inf)
        out1[s:s + 1024], out2[s:s + 1024] = (-a, -b) if metric == "cosine" else (a, b)
    return out1, out2


def run(ops, x, metric, mode, rows=None, flags=0, band_tol=1e-3):
    res = ops.self_filter(torch.from_numpy(x).cuda(), THR[metric], metric=metric, mode=mode, rows=rows, flags=flags,
                          band_tol=band_tol, want_stats=True)
    torch.cuda.synchronize()
    return res


def check(ops, x, metric, mode, rows=None, sample=None):
    """The tcgen05 / default result against the oracle on ``sample`` (global rows inside ``rows``), and (Euclid) against the
    FORCE_FP32 self result on every row of the range."""
    n = len(x)
    b, e = (0, n) if rows is None else rows
    res = run(ops, x, metric, mode, rows)
    assert res.stats["path"] == ("tcgen05" if n > 8 and x.shape[1] <= 512 else "fp32"), res.stats
    keep, idx, val = res.keep.cpu().numpy(), res.best_idx.cpu().numpy(), res.best_val.cpu().numpy()
    thr = THR[metric]
    g = np.arange(b, e) if sample is None else np.asarray(sample)
    loc = g - b
    ko, io, so = filter_self(x, thr, metric, mode, rows=g)
    b1, b2 = top2_64(x, g, metric, mode)
    none = io < 0
    assert np.array_equal(idx[loc][none], io[none]) and not keep[loc][none].any()
    assert np.all(val[loc][none] == (-np.inf if metric == "cosine" else np.inf))
    with np.errstate(invalid="ignore"):              # (rows without an eligible reference: inf - inf)
        tie = np.abs(b1 - b2) <= TIE * (np.maximum(np.abs(b1), 1.0) if metric == "euclid" else 1.0)
    bad = np.flatnonzero((idx[loc] != io) & ~tie & ~none)
    assert bad.size == 0, (bad.size, g[bad[:5]], idx[loc][bad[:5]], io[bad[:5]], res.stats)
    near = np.abs(b1 - thr) <= TIE * max(1.0, thr)
    bad = np.flatnonzero((keep[loc] != ko) & ~near)
    assert bad.size == 0, (bad.size, g[bad[:5]], b1[bad[:5]])
    fin = ~none
    tol = 1e-3 * (np.maximum(1.0, so[fin]) if metric == "euclid" else 1.0)
    assert np.all(np.abs(val[loc][fin] - so[fin]) <= tol)
    if res.band_rows is not None:                    # the band is exact: rows within 1e-3 of thr by their returned score
        want = np.flatnonzero(np.abs(val - np.float32(thr)) <= np.float32(1e-3))
        assert np.array_equal(np.sort(res.band_rows.cpu().numpy()), want)
    if metric == "euclid":
        ex = run(ops, x, metric, mode, rows, flags=ops.FLAG_FORCE_FP32)
        assert ex.stats["path"] == "fp32"
        ke, ie, ve = ex.keep.cpu().numpy(), ex.best_idx.cpu().numpy(), ex.best_val.cpu().numpy()
        same = idx == ie
        assert np.mean(same) > 0.999
        assert np.array_equal(keep[same], ke[same]) and np.array_equal(val[same].view(np.uint32), ve[same].view(np.uint32))
        diff = np.flatnonzero(~same[loc])
        assert np.all(tie[diff]), (g[diff[:5]], idx[loc][diff[:5]], ie[loc][diff[:5]])
    return res


SMALL_N = [1, 2, 8, 9, 255, 256, 257, 1000]


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
@pytest.mark.parametrize("mode", ["others", "earlier"])
@pytest.mark.parametrize("dim", [64, 128, 256, 512])
@pytest.mark.parametrize("n", SMALL_N)
def test_self_small(ops, n, dim, mode, metric):
    check(ops, make_set(n, dim, metric, seed=n * 7 + dim), metric, mode)


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
@pytest.mark.parametrize("mode", ["others", "earlier"])
@pytest.mark.parametrize("n,dim", [(4097, 128), (4097, 512), (20_000, 64), (20_000, 256)])
def test_self_large(ops, n, dim, mode, metric):
    x = make_set(n, dim, metric, seed=n + dim)
    rng = np.random.default_rng(1)
    sample = np.unique(np.r_[np.arange(300), np.arange(n - 300, n), rng.choice(n, 1500, replace=False)])
    check(ops, x, metric, mode, sample=sample)


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
@pytest.mark.parametrize("mode", ["others", "earlier"])
def test_self_row_range_unaligned(ops, mode, metric):
    """A row_begin that is not a multiple of 128 / 256 and a ragged n_rows: a CTA pair's rows straddle two reference tiles."""
    x = make_set(3000, 128, metric, seed=5)
    check(ops, x, metric, mode, rows=(389, 389 + 1003))
    full = run(ops, x, metric, mode)
    part = run(ops, x, metric, mode, rows=(389, 1392))
    assert np.array_equal(full.best_idx.cpu().numpy()[389:1392], part.best_idx.cpu().numpy())


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
def test_self_no_eligible_reference(ops, metric):
    x = make_set(300, 128, metric, seed=2)
    bad = -np.inf if metric == "cosine" else np.inf
    for rows in [None, (0, 1), (0, 257)]:
        r = run(ops, x, metric, "earlier", rows=rows, band_tol=10.0)
        assert r.best_idx[0].item() == -1 and r.keep[0].item() == 0 and r.best_val[0].item() == bad
        assert 0 not in r.band_rows.cpu().numpy().tolist()
    one = run(ops, x[:1], metric, "others")
    assert one.best_idx.item() == -1 and one.keep.item() == 0 and one.best_val.item() == bad
    assert run(ops, x[:2], metric, "earlier").best_idx.cpu().tolist() == [-1, 0]


def test_self_copies_found_at_fold_scale(ops):
    """50 k x 128 (a gallery call of this shape folds bit-identical references): every copy's earliest occurrence is found."""
    n, dim = 50_000, 128
    rng = np.random.default_rng(9)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    src = rng.choice(n // 2, 500, replace=False)
    dst = rng.choice(np.arange(n // 2, n), 500, replace=False)
    x[dst] = x[src]
    for metric in ("cosine", "euclid"):
        r = run(ops, x, metric, "earlier")
        assert r.stats["path"] == "tcgen05" and r.stats["refs_scanned"] == n, r.stats
        idx, keep = r.best_idx.cpu().numpy(), r.keep.cpu().numpy()
        assert np.array_equal(idx[dst], src) and keep[dst].all()
        rows = np.unique(np.r_[dst[:200], rng.choice(n, 800, replace=False)])
        _, io, _ = filter_self(x, THR[metric], metric, "earlier", rows=rows)
        assert np.array_equal(idx[rows], io)
        o = run(ops, x, "cosine", "others")
        oi = o.best_idx.cpu().numpy()
        assert np.array_equal(oi[src], dst) and np.array_equal(oi[dst], src)


def test_self_refusals(ops):
    from face_detection_and_recognition_b200._lib import FfrError
    x = torch.from_numpy(make_set(100, 128, "cosine", seed=3)).cuda()
    with pytest.raises(FfrError) as e:
        ops.self_filter(x.half(), 0.8)
    assert e.value.code == -4
    with pytest.raises(FfrError) as e:
        ops.self_filter(x, 0.8, flags=ops.FLAG_NO_RECHECK)
    assert e.value.code == -4
    for rows in [(-1, 10), (50, 101), (90, 200)]:
        with pytest.raises(FfrError) as e:
            ops.self_filter(x, 0.8, rows=rows)
        assert e.value.code == -1
    with pytest.raises(TypeError):
        ops.self_filter(x.cpu(), 0.8)
    assert ops.self_filter(x, 0.8, rows=(40, 40)).keep.numel() == 0


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from face_detection_and_recognition_b200.sharding import CandidateSharder
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    x = make_set(10_001, 128, "cosine", seed=13)
    sh = CandidateSharder(rank, world, device=rank, gather="nccl")
    keep, idx, _ = sh.self_filter(torch.from_numpy(x).cuda(), THR["cosine"], metric="cosine", mode="earlier")
    torch.cuda.synchronize()
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), keep=keep.cpu().numpy(), idx=idx.cpu().numpy())
    sh.close()
    dist.destroy_process_group()


def test_self_sharded_nccl(ops, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    one = run(ops, make_set(10_001, 128, "cosine", seed=13), "cosine", "earlier")
    for r in range(2):
        g = np.load(tmp_path / f"r{r}.npz")
        assert np.array_equal(g["keep"], one.keep.cpu().numpy()) and np.array_equal(g["idx"], one.best_idx.cpu().numpy())
