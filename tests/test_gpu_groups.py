"""Near-duplicate groups on the GPU (ffr_self_groups / ops.self_groups): the labels against the host union-find of the same call's
match list, the tensor-core path against the exact kernel, the fp64 oracle as a sandwich, union-find stress shapes (a permuted
chain, a star, a clique of bit-identical rows), overflow and retry, mode "earlier", CUDA-graph capture, the file layer and the
errors."""
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from face_detection_and_recognition_b200 import _lib, embeddings_io, ops
from face_detection_and_recognition_b200._lib import FLAG_FORCE_FP32, FLAG_FORCE_MMA, FLAG_NO_RECHECK, FfrError
from oracle import oracle_pairs
from oracle.oracle_groups import components

pytestmark = pytest.mark.gpu

THR = {"cosine": 0.85, "euclid": 2.0}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _unit(rng, n, dim):
    x = rng.standard_normal((n, dim))
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def _clustered(n, dim, metric, seed):
    """Groups of noisy copies of a base row (noise 0.2..0.6 of the base's norm: some copies match, some only through others),
    unrelated rows, one bit-identical pair and zero rows.  Euclid: rows scaled by 0.3..4."""
    rng = np.random.default_rng(seed)
    x = _unit(rng, n, dim)
    if metric == "euclid":
        x *= rng.uniform(0.3, 4.0, (n, 1))
    n_dup = n // 2
    src = rng.integers(0, max(n // 8, 1), n_dup)
    dst = rng.choice(n, n_dup, replace=False)
    s = rng.uniform(0.2, 0.6, (n_dup, 1))
    base = x[src]
    x[dst] = base + s * np.linalg.norm(base, axis=1, keepdims=True) * rng.standard_normal((n_dup, dim)) / np.sqrt(dim)
    if n >= 4:
        x[n - 1] = x[n // 3]
        x[n // 2] = 0.0
        x[1] = 0.0
    return x.astype(np.float32)


def _host_labels(pairs, n):
    return components(n, pairs.cand.cpu().numpy(), pairs.ref.cpu().numpy())


def _finer(fine, coarse):
    """Every group of `fine` lies inside one group of `coarse` (labels are member rows, so one lookup per row decides)."""
    return bool(np.array_equal(coarse, coarse[fine]))


def _check_sandwich(labels, x, thr, metric, tol=1e-6):
    """loose graph (fp64 edges outside the tol band) <= the library's partition <= full graph (fp64 edges and the band pairs)"""
    lo = thr - tol if metric == "cosine" else thr * (1 + tol)
    c, r, v = oracle_pairs.self_pairs(x, lo, metric, dtype=np.float64)
    inside = v > thr + tol if metric == "cosine" else v < thr * (1 - tol)
    full = components(len(x), c, r)
    loose = components(len(x), c[inside], r[inside])
    assert _finer(loose, labels) and _finer(labels, full)


def _check_against_pairs(dev, x_t, thr, metric, res=None):
    """The labels are the host union-find of self_pairs on the same input; the group and edge counts match it."""
    n = x_t.shape[0]
    res = res or ops.self_groups(x_t, thr, metric)
    pairs = ops.self_pairs(x_t, thr, metric)
    want = _host_labels(pairs, n)
    got = res.labels.cpu().numpy().astype(np.int64)
    assert res.labels.dtype == torch.int32 and res.labels.device == x_t.device
    assert np.array_equal(got, want)
    assert res.n_groups == int((want == np.arange(n)).sum()) and res.n_edges == len(pairs.cand)
    return got


SHAPES = [(1, 64), (5, 128), (8, 200), (9, 64), (300, 130), (2000, 256), (1500, 512), (400, 640)]


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
@pytest.mark.parametrize("n,dim", SHAPES)
def test_self_groups(dev, n, dim, metric):
    x = _clustered(n, dim, metric, seed=n + dim)
    thr = THR[metric]
    x_t = torch.from_numpy(x).to(dev)
    res = ops.self_groups(x_t, thr, metric, want_stats=True)
    mma = n > 8 and dim <= 512
    assert res.stats["path"] == ("tcgen05" if mma else "fp32")
    got = _check_against_pairs(dev, x_t, thr, metric, res)
    exact = ops.self_groups(x_t, thr, metric, flags=FLAG_FORCE_FP32, want_stats=True)
    assert exact.stats["path"] == "fp32"
    assert torch.equal(exact.labels, res.labels) and (exact.n_groups, exact.n_edges) == (res.n_groups, res.n_edges)
    _check_sandwich(got, x, thr, metric)
    assert (got <= np.arange(n)).all() and (got[got] == got).all()
    if n >= 300:
        assert 1 < res.n_groups < n - 10                     # the data has real groups
        assert got[n - 1] == got[n // 3]                     # the bit-identical pair
        if metric == "cosine":
            assert got[1] == 1 and got[n // 2] == n // 2     # zero rows are singletons
    if n == 1:
        assert got.tolist() == [0] and res.n_groups == 1 and res.n_edges == 0


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
def test_mode_earlier_flags_only_non_representatives(dev, metric):
    x = _clustered(3000, 128, metric, seed=31)
    thr = THR[metric]
    x_t = torch.from_numpy(x).to(dev)
    lab = ops.self_groups(x_t, thr, metric).labels.cpu().numpy()
    f = ops.self_filter(x_t, thr, metric, mode="earlier")
    keep, best = f.keep.cpu().numpy().astype(bool), f.best_val.cpu().numpy().astype(np.float64)
    band = np.abs(best - thr) <= (1e-6 if metric == "cosine" else 1e-6 * thr)
    j = np.arange(len(x))
    assert (lab[keep & ~band] < j[keep & ~band]).all()      # a row with an earlier match is never its group's representative
    rep = lab == j
    assert not (rep & keep & ~band).any()
    assert keep.sum() > 100


def test_permuted_chain(dev):
    """A random walk with consecutive rows at cosine 0.9 (rows two apart near 0.81), rows permuted: one component that is in
    essence a path over 20 000 rows.  Chance shortcuts above 0.85 change nothing."""
    rng = np.random.default_rng(41)
    n, dim = 20_000, 512
    w = np.empty((n, dim))
    w[0] = _unit(rng, 1, dim)[0]
    for k in range(1, n):
        u = rng.standard_normal(dim)
        u -= (u @ w[k - 1]) * w[k - 1]
        w[k] = 0.9 * w[k - 1] + np.sqrt(1 - 0.81) * u / np.linalg.norm(u)
    x = w[rng.permutation(n)].astype(np.float32)
    x_t = torch.from_numpy(x).to(dev)
    res = ops.self_groups(x_t, 0.85)
    assert res.n_groups == 1 and (res.labels == 0).all().item() and res.n_edges >= n - 1
    _check_against_pairs(dev, x_t, 0.85, "cosine", res)
    assert torch.equal(ops.self_groups(x_t, 0.85, flags=FLAG_FORCE_FP32).labels, res.labels)


def test_star(dev):
    """One hub and 4000 spokes at cosine 0.92 to it (about 0.846 to each other), among 2000 unrelated rows."""
    rng = np.random.default_rng(42)
    n_spokes, dim = 4000, 256
    hub = _unit(rng, 1, dim)[0]
    u = rng.standard_normal((n_spokes, dim))
    u -= (u @ hub)[:, None] * hub
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    spokes = 0.92 * hub + np.sqrt(1 - 0.92 ** 2) * u
    x = np.concatenate([_unit(rng, 2000, dim), spokes, hub[None]])
    perm = rng.permutation(len(x))
    x = x[perm].astype(np.float32)
    star = np.argsort(perm)[2000:]                           # positions of the spokes and the hub
    x_t = torch.from_numpy(x).to(dev)
    got = _check_against_pairs(dev, x_t, 0.85, "cosine")
    assert (got[star] == star.min()).all()
    assert (np.bincount(got, minlength=len(x))[star.min()] >= len(star))


def test_clique_of_identical_rows_overflows_and_retries(dev):
    """3000 bit-identical copies (4.5 M edges) among 3000 other rows: the default edge list overflows and the call retries."""
    rng = np.random.default_rng(43)
    n, dim = 6000, 128
    x = _unit(rng, n, dim).astype(np.float32)
    clique = np.sort(rng.choice(n, 3000, replace=False))
    x[clique] = x[clique[0]]
    x_t = torch.from_numpy(x).to(dev)
    res = ops.self_groups(x_t, 0.85, want_stats=True)
    assert res.n_edges >= 3000 * 2999 // 2 and res.n_edges > ops._default_pair_cap(n)
    lab = res.labels.cpu().numpy()
    assert (lab[clique] == clique[0]).all()
    rest = np.setdiff1d(np.arange(n), clique)
    assert res.n_groups == 1 + int((lab[rest] == rest).sum())
    assert torch.equal(ops.self_groups(x_t, 0.85, flags=FLAG_FORCE_FP32).labels, res.labels)


def test_make_set_data(dev):
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from bench_self import THR as SET_THR, make_set
    x, _ = make_set(20_000, 128, seed=5)
    x_t = torch.from_numpy(x).to(dev)
    res = _check_against_pairs(dev, x_t, SET_THR, "cosine")
    assert (res < np.arange(len(x))).sum() > 100
    assert torch.equal(ops.self_groups(x_t, SET_THR, flags=FLAG_FORCE_FP32).labels.cpu(), torch.from_numpy(res).int())


@pytest.mark.parametrize("metric,thr", [("cosine", 1.5), ("euclid", -1.0)])
def test_threshold_that_matches_nothing(dev, metric, thr):
    x_t = torch.from_numpy(_clustered(1000, 64, metric, seed=44)).to(dev)
    res = ops.self_groups(x_t, thr, metric)
    assert torch.equal(res.labels, torch.arange(1000, dtype=torch.int32, device=dev))
    assert res.n_groups == 1000 and res.n_edges == 0


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
def test_zero_rows(dev, metric):
    """Euclid: zero rows (1 / |c| not finite) go through the exact-row list and match each other and the short rows, so they
    join the group of the zero row 1 that _clustered plants; cosine: every zero row is its own group."""
    rng = np.random.default_rng(45)
    x = _clustered(700, 128, metric, seed=45)
    zeros = rng.choice(700, 12, replace=False)
    x[zeros] = 0.0
    x_t = torch.from_numpy(x).to(dev)
    got = _check_against_pairs(dev, x_t, THR[metric], metric)
    assert torch.equal(ops.self_groups(x_t, THR[metric], metric, flags=FLAG_FORCE_FP32).labels.cpu(), torch.from_numpy(got).int())
    _check_sandwich(got, x, THR[metric], metric)
    if metric == "cosine":
        assert (got[zeros] == zeros).all()
    else:
        assert (got[zeros] == got[1]).all() and got[1] <= 1


def _c_groups(lib, x_t, thr, metric, cap, flags=0, ws_extra=0, labels=None, n=None):
    dev = x_t.device
    m = _lib.METRIC_EUCLID if metric == "euclid" else _lib.METRIC_COSINE
    n = x_t.shape[0] if n is None else n
    dim = x_t.shape[1]
    need = int(lib.ffr_self_groups_workspace_bytes(x_t.shape[0], dim, m, cap))
    ws = torch.empty(need + 256, dtype=torch.uint8, device=dev)
    lab = torch.full((x_t.shape[0],), -7, dtype=torch.int32, device=dev)
    cnt = torch.full((2,), -7, dtype=torch.int64, device=dev)
    rc = lib.ffr_self_groups(x_t.data_ptr(), n, dim, m, float(thr), lab.data_ptr() if labels is None else labels, cnt.data_ptr(),
                             cap, cnt[1:].data_ptr(), flags, ws.data_ptr(), need + ws_extra,
                             torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize(dev)
    return rc, lab, int(cnt[0].item()), int(cnt[1].item())


@pytest.mark.parametrize("metric", ["cosine", "euclid"])
@pytest.mark.parametrize("flags", [0, FLAG_FORCE_FP32])
def test_overflow_at_the_c_level(dev, metric, flags):
    lib = _lib.load()
    x = _clustered(1200, 96, metric, seed=46)
    thr = 0.7 if metric == "cosine" else 3.0                 # many edges
    x_t = torch.from_numpy(x).to(dev)
    full = ops.self_groups(x_t, thr, metric, cap=10 ** 6)
    assert full.n_edges > 1000
    rc, lab, groups, cnt = _c_groups(lib, x_t, thr, metric, 0, flags)          # cap 0: counts only
    assert rc == 0 and cnt >= full.n_edges
    assert torch.equal(lab, torch.arange(1200, dtype=torch.int32, device=dev)) and groups == 1200
    rc, lab, groups, cnt = _c_groups(lib, x_t, thr, metric, 100, flags)
    assert rc == 0 and cnt > 100
    want = full.labels.cpu().numpy()
    part = lab.cpu().numpy()
    assert _finer(part, want) and groups == int((part == np.arange(1200)).sum()) and groups > full.n_groups
    rc, lab, groups, cnt2 = _c_groups(lib, x_t, thr, metric, cnt, flags)
    assert rc == 0 and cnt2 == full.n_edges and groups == full.n_groups
    assert torch.equal(lab, full.labels)
    one = ops.self_groups(x_t, thr, metric, cap=1, flags=flags)            # the wrapper retries by itself
    assert torch.equal(one.labels, full.labels) and (one.n_groups, one.n_edges) == (full.n_groups, full.n_edges)


def test_cuda_graph_capture(dev):
    """The C call has no host synchronisation and no allocation: captured once, a replay recomputes the labels of new data."""
    lib = _lib.load()
    n, dim, thr = 2000, 128, 0.85
    x = torch.from_numpy(_clustered(n, dim, "cosine", seed=47)).to(dev)
    cap = 1 << 16
    ws = torch.empty(int(lib.ffr_self_groups_workspace_bytes(n, dim, 0, cap)), dtype=torch.uint8, device=dev)
    lab = torch.empty(n, dtype=torch.int32, device=dev)
    cnt = torch.zeros(2, dtype=torch.int64, device=dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))

    def call():
        _lib.check(lib.ffr_self_groups(x.data_ptr(), n, dim, 0, thr, lab.data_ptr(), cnt.data_ptr(), cap, cnt[1:].data_ptr(), 0,
                                       ws.data_ptr(), ws.numel(), side.cuda_stream))

    with torch.cuda.stream(side):
        call()                                               # warm-up outside the capture
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        call()
    x.copy_(torch.from_numpy(_clustered(n, dim, "cosine", seed=48)).to(dev))
    lab.fill_(-1)
    g.replay()
    torch.cuda.synchronize(dev)
    want = ops.self_groups(x, thr)
    assert torch.equal(lab, want.labels) and cnt.tolist() == [want.n_groups, want.n_edges]


def test_group_embedding_files(dev, tmp_path):
    """Three .pkl files of four faces: img f holds faces f, f + 1, f + 2 of five people and one face of nobody else."""
    rng = np.random.default_rng(49)
    people = _unit(rng, 5, 128).astype(np.float32)
    files = []
    for f in range(3):
        faces = [{"det_score": 0.9, "normed_feature": people[f + k]} for k in range(3)]
        faces.append({"det_score": 0.8, "normed_feature": _unit(rng, 1, 128)[0].astype(np.float32)})
        p = tmp_path / f"img{f}.pkl"
        with open(p, "wb") as fh:
            pickle.dump(faces, fh)
        files.append(str(p))
    labels, n_groups, prov = embeddings_io.group_embedding_files(files, 0.9)
    x, prov2 = embeddings_io.load_embeddings(files)
    assert prov == prov2 and labels.dtype == np.int32 and len(labels) == 12
    want = ops.self_groups(torch.from_numpy(x).to(dev), 0.9)
    assert np.array_equal(labels, want.labels.cpu().numpy()) and n_groups == want.n_groups == 5 + 3
    for i in range(12):                                      # each face's group starts at its first occurrence
        assert labels[i] == min(j for j in range(12) if np.array_equal(x[j], x[i]))
    assert prov[labels[9]] == (files[1], 2)                  # person 3: face 2 of img1, face 1 of img2


def test_groups_errors(dev):
    lib = _lib.load()
    rng = np.random.default_rng(50)
    x = torch.from_numpy(_unit(rng, 64, 128).astype(np.float32)).to(dev)
    with pytest.raises(FfrError) as e:
        ops.self_groups(x, 0.5, flags=FLAG_NO_RECHECK)
    assert e.value.code == -4
    with pytest.raises(FfrError) as e:
        ops.self_groups(x[:8], 0.5, flags=FLAG_FORCE_MMA)
    assert e.value.code == -4
    with pytest.raises(FfrError) as e:
        ops.self_groups(torch.from_numpy(_unit(rng, 64, 640).astype(np.float32)).to(dev), 0.5, flags=FLAG_FORCE_MMA)
    assert e.value.code == -4
    assert ops.self_groups(x, 0.5, flags=FLAG_FORCE_MMA, want_stats=True).stats["path"] == "tcgen05"
    with pytest.raises(ValueError):
        ops.self_groups(x.reshape(64, 2, 64), 0.5)
    for metric in ("cosine", "euclid"):
        rc, *_ = _c_groups(lib, x, 0.5, metric, 100, ws_extra=-1)          # one byte short
        assert rc == -3
        rc, *_ = _c_groups(lib, x, 0.5, metric, 100, labels=C.c_void_p(0))  # null labels
        assert rc == -1
        rc, *_ = _c_groups(lib, x, 0.5, metric, 100, n=2 ** 31)
        assert rc == -1
        rc, *_ = _c_groups(lib, x, 0.5, metric, 100, n=0)
        assert rc == -1
