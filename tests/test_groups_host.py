"""Near-duplicate groups without a GPU: oracle_groups against a breadth-first search (and scipy when it imports), the workspace
query, argument errors and the wrappers' refusal of CPU and fp16 tensors."""
import ctypes as C
from collections import deque

import numpy as np
import pytest

from oracle.oracle_groups import components, self_groups
from oracle.oracle_pairs import self_pairs


def _bfs(n, a, b):
    adj = [[] for _ in range(n)]
    for u, v in zip(a, b):
        adj[u].append(v)
        adj[v].append(u)
    lab = [-1] * n
    for s in range(n):                                       # ascending start rows: each component is labelled by its minimum
        if lab[s] >= 0:
            continue
        lab[s] = s
        q = deque([s])
        while q:
            u = q.popleft()
            for v in adj[u]:
                if lab[v] < 0:
                    lab[v] = s
                    q.append(v)
    return np.array(lab, dtype=np.int64)


def _random_graph(n, m, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, n, m), rng.integers(0, n, m)


@pytest.mark.parametrize("n,m,seed", [(1, 0, 0), (7, 3, 1), (50, 30, 2), (200, 150, 3), (500, 2000, 4)])
def test_components_match_bfs(n, m, seed):
    a, b = _random_graph(n, m, seed)
    assert np.array_equal(components(n, a, b), _bfs(n, a, b))


def test_components_of_a_permuted_chain_and_a_star():
    rng = np.random.default_rng(5)
    perm = rng.permutation(3000)
    lab = components(3000, perm[:-1], perm[1:])
    assert (lab == 0).all()
    lab = components(1000, np.full(999, 617), np.arange(1000)[np.arange(1000) != 617])
    assert (lab == 0).all()
    lab = components(10, [], [])
    assert np.array_equal(lab, np.arange(10))


def test_components_match_scipy():
    sp = pytest.importorskip("scipy.sparse")
    csgraph = pytest.importorskip("scipy.sparse.csgraph")
    n = 2000
    a, b = _random_graph(n, 1500, 6)
    k, lab_sp = csgraph.connected_components(sp.coo_matrix((np.ones(len(a)), (a, b)), shape=(n, n)), directed=False)
    lab = components(n, a, b)
    assert len(np.unique(lab)) == k
    # the same partition: scipy's labels are a relabelling of the min-index ones
    first = {}
    for i, (x, y) in enumerate(zip(lab_sp.tolist(), lab.tolist())):
        assert first.setdefault(x, y) == y, i
    assert (lab <= np.arange(n)).all() and (lab[lab] == lab).all()


@pytest.mark.parametrize("metric,thr", [("cosine", 0.6), ("euclid", 2.5)])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_self_groups_oracle_is_components_of_the_pairs(metric, thr, dtype):
    rng = np.random.default_rng(7)
    x = rng.standard_normal((120, 16)).astype(np.float32)
    x[60:] = x[rng.integers(0, 60, 60)] + 0.25 * rng.standard_normal((60, 16)).astype(np.float32)
    x[100] = x[3]                                           # a bit-identical pair is an edge
    lab, k = self_groups(x, thr, metric, block=17, dtype=dtype)
    c, r, _ = self_pairs(x, thr, metric, dtype=dtype)
    assert np.array_equal(lab, _bfs(len(x), c, r))
    assert k == len(np.unique(lab)) and lab[100] == lab[3]
    assert 1 < k < len(x)


def test_groups_workspace_query(ffr_lib):
    q = ffr_lib.ffr_self_groups_workspace_bytes
    for metric in (0, 1):
        sizes = [q(5000, 128, metric, cap) for cap in (0, 1, 1000, 10 ** 6)]
        assert all(s > 0 for s in sizes) and sizes == sorted(sizes)
        assert sizes[-1] - sizes[0] >= 12 * 10 ** 6                      # the edge list: 12 bytes per entry
        assert q(5000, 128, metric, 1000) < q(50000, 128, metric, 1000)   # grows with n
        # at least the match list's buffers
        assert q(5000, 128, metric, 1000) >= ffr_lib.ffr_match_pairs_self_workspace_bytes(5000, 5000, 128, metric, 1000)
    # the exact path (n <= 8, dim > 512) still keeps the edge list
    assert q(8, 128, 0, 1000) - q(8, 128, 0, 0) >= 12000
    assert q(100, 640, 1, 1000) - q(100, 640, 1, 0) >= 12000
    for bad in ((0, 128, 0, 10), (-1, 128, 0, 10), (2 ** 31, 128, 0, 10), (100, 0, 0, 10), (100, 128, 7, 10), (100, 128, 0, -1)):
        assert q(*bad) == 0, bad


def test_groups_bad_arguments_and_no_gpu(ffr_lib):
    buf = (C.c_float * 1024)()
    lab = (C.c_int32 * 16)()
    cnt = (C.c_int64 * 2)()
    p = C.addressof(buf)
    ws = (C.c_uint8 * 4096)()
    # (x, n, dim, metric, thr, labels, group_count, edge_cap, edge_count, flags, ws, ws_bytes, stream)
    good = [p, 8, 8, 0, 0.5, C.addressof(lab), C.addressof(cnt), 16, C.addressof(cnt) + 8, 0, C.addressof(ws), 4096, None]
    bad = {0: None, 1: 0, 2: 0, 3: 5, 5: None, 6: None, 7: -1, 8: None}
    for k, v in bad.items():
        a = list(good)
        a[k] = v
        assert ffr_lib.ffr_self_groups(*a) == -1, k
    a = list(good)
    a[1] = 2 ** 31
    assert ffr_lib.ffr_self_groups(*a) == -1
    a = list(good)
    a[9] = 4                                                 # FFR_FLAG_NO_RECHECK
    assert ffr_lib.ffr_self_groups(*a) == -4
    if ffr_lib.ffr_device_count() == 0:
        assert ffr_lib.ffr_self_groups(*good) == -2 and b"no CUDA device" in ffr_lib.ffr_last_error()


def test_group_wrappers_refuse_cpu_fp16_and_bad_shapes(ffr_lib):
    import torch
    from face_detection_and_recognition_b200 import ops
    from face_detection_and_recognition_b200._lib import FfrError
    with pytest.raises(TypeError):
        ops.self_groups(torch.zeros(4, 128), 0.5)
    with pytest.raises(FfrError):
        ops.self_groups(torch.zeros(4, 128, dtype=torch.float16), 0.5)
    if torch.cuda.is_available():
        with pytest.raises(ValueError):
            ops.self_groups(torch.zeros(4, 2, 64, device="cuda"), 0.5)
