"""Match lists without a GPU: oracle_pairs against a brute-force loop and against oracle_self, the workspace queries, argument
errors and the wrappers' refusal of CPU tensors."""
import ctypes as C

import numpy as np
import pytest

from oracle.oracle_pairs import match_pairs, self_pairs
from oracle.oracle_self import filter_self


def _brute(ref, cand, thr, metric, earlier_rows=None):
    r64, c64 = ref.astype(np.float64), cand.astype(np.float64)
    out = []
    for j, c in enumerate(c64):
        for i, r in enumerate(r64):
            if earlier_rows is not None and i >= earlier_rows[j]:
                continue
            if metric == "cosine":
                v = r @ c / (np.linalg.norm(r) * np.linalg.norm(c))
                ok = v >= thr
            else:
                v = np.linalg.norm(c - r)
                ok = v <= thr
            if ok:
                out.append((j, i, v))
    return out


def _data(n, m, dim, seed):
    rng = np.random.default_rng(seed)
    ref = rng.standard_normal((n, dim)).astype(np.float32)
    cand = rng.standard_normal((m, dim)).astype(np.float32)
    cand[: m // 2] = ref[rng.integers(0, n, m // 2)] + 0.3 * rng.standard_normal((m // 2, dim)).astype(np.float32)
    ref[n - 1] = ref[0]                                     # a bit-identical copy: both are pairs
    return ref, cand


@pytest.mark.parametrize("metric,thr", [("cosine", 0.5), ("euclid", 3.0)])
def test_gallery_oracle_matches_brute_force(metric, thr):
    ref, cand = _data(23, 31, 12, 1)
    c, r, v = match_pairs(ref, cand, thr, metric, ref_index_base=100, block=7)
    want = _brute(ref, cand, thr, metric)
    assert [(a, b - 100) for a, b in zip(c.tolist(), r.tolist())] == [(a, b) for a, b, _ in want]
    assert np.allclose(v, [x for _, _, x in want], rtol=1e-5, atol=1e-6)
    assert len(want) > 10


@pytest.mark.parametrize("metric,thr", [("cosine", 0.5), ("euclid", 3.0)])
def test_self_oracle_matches_brute_force(metric, thr):
    x, _ = _data(29, 1, 12, 2)
    x[20:] = x[:9] + 0.2 * np.random.default_rng(3).standard_normal((9, 12)).astype(np.float32)
    rows = np.array([28, 3, 0, 17, 20])
    c, r, v = self_pairs(x, thr, metric, rows=rows, block=2)
    want = _brute(x, x[rows], thr, metric, earlier_rows=rows)
    assert list(zip(c.tolist(), r.tolist())) == [(a, b) for a, b, _ in want]
    assert np.allclose(v, [x_ for _, _, x_ in want], rtol=1e-5, atol=1e-6)
    assert (r < rows[c]).all() and len(want) >= 2


def test_zero_rows_give_no_cosine_pairs_and_their_euclid_pairs():
    ref, cand = _data(10, 6, 8, 4)
    ref[3] = 0.0
    cand[2] = 0.0
    c, r, _ = match_pairs(ref, cand, -1.0, "cosine")
    assert not np.isin(r, [3]).any() and not np.isin(c, [2]).any()
    c, r, v = match_pairs(ref, cand, 1e9, "euclid")
    assert len(c) == 60 and np.allclose(v[(c == 2)], np.linalg.norm(ref, axis=1))


@pytest.mark.parametrize("metric,thr", [("cosine", 0.3), ("euclid", 4.0)])
def test_self_oracle_best_pair_is_filter_self_best_match(metric, thr):
    x, _ = _data(60, 1, 10, 5)
    c, r, v = self_pairs(x, thr, metric, dtype=np.float64)
    keep, idx, best = filter_self(x, thr, metric, "earlier", dtype=np.float64)
    for j in range(len(x)):
        sel = c == j
        assert sel.any() == bool(keep[j])
        if sel.any():
            k = np.argmax(v[sel]) if metric == "cosine" else np.argmin(v[sel])
            assert r[sel][k] == idx[j] and v[sel][k] == best[j]


def test_pairs_workspace_queries_are_monotone_in_cap(ffr_lib):
    for q, a in ((ffr_lib.ffr_match_pairs_workspace_bytes, (1000, 5000, 512)),
                 (ffr_lib.ffr_match_pairs_self_workspace_bytes, (5000, 3000, 128))):
        for metric in (0, 1):
            sizes = [q(*a, metric, cap) for cap in (0, 1, 1000, 10 ** 6, 10 ** 8)]
            assert all(s > 0 for s in sizes) and sizes == sorted(sizes)
            assert sizes[-1] - sizes[0] >= 8 * 10 ** 8
        assert q(*a, 0, -1) == 0
    assert ffr_lib.ffr_match_pairs_workspace_bytes(0, 10, 128, 0, 10) == 0
    # the exact path (<= 8 references, dim > 512) keeps no raw list
    assert ffr_lib.ffr_match_pairs_workspace_bytes(8, 10, 128, 0, 0) == ffr_lib.ffr_match_pairs_workspace_bytes(8, 10, 128, 0, 10 ** 6)
    assert ffr_lib.ffr_match_pairs_workspace_bytes(100, 10, 640, 1, 0) == ffr_lib.ffr_match_pairs_workspace_bytes(100, 10, 640, 1, 99)


def test_pairs_bad_arguments_and_no_gpu(ffr_lib):
    buf = (C.c_float * 1024)()
    cnt = C.c_int64()
    p = C.addressof(buf)
    ws = (C.c_uint8 * 4096)()
    # (ref, n_ref, cand, n_cand, dim, metric, thr, base, pc, pr, pv, cap, count, flags, ws, ws_bytes, stream)
    good = [p, 4, p, 4, 8, 0, 0.5, 0, p, p, p, 16, C.addressof(cnt), 0, C.addressof(ws), 4096, None]
    bad = {1: 0, 3: -1, 4: 0, 5: 7, 0: None, 7: -1, 11: -1, 12: None}
    for k, v in bad.items():
        a = list(good)
        a[k] = v
        assert ffr_lib.ffr_match_pairs(*a) == -1, k
    a = list(good)
    a[7] = 2 ** 31 - 4                                       # ref_index_base + n_ref == 2^31
    assert ffr_lib.ffr_match_pairs(*a) == -1 and b"int32" in ffr_lib.ffr_last_error()
    a = list(good)
    a[8] = None                                              # cap > 0 without the output arrays
    assert ffr_lib.ffr_match_pairs(*a) == -1
    # self: (x, n, row_begin, n_rows, dim, metric, thr, pc, pr, pv, cap, count, flags, ws, ws_bytes, stream)
    sgood = [p, 8, 2, 4, 8, 0, 0.5, p, p, p, 16, C.addressof(cnt), 0, C.addressof(ws), 4096, None]
    for k, v in {1: 0, 2: 5, 3: -1, 4: 0, 5: 3, 0: None, 10: -1, 11: None}.items():
        a = list(sgood)
        a[k] = v
        assert ffr_lib.ffr_match_pairs_self(*a) == -1, k
    a = list(good)
    a[13] = 4                                                # FFR_FLAG_NO_RECHECK
    assert ffr_lib.ffr_match_pairs(*a) == -4
    if ffr_lib.ffr_device_count() == 0:
        assert ffr_lib.ffr_match_pairs(*good) == -2 and b"no CUDA device" in ffr_lib.ffr_last_error()
        assert ffr_lib.ffr_match_pairs_self(*sgood) == -2


def test_pair_wrappers_refuse_cpu_and_fp16_tensors(ffr_lib):
    import torch
    from face_detection_and_recognition_b200 import ops
    from face_detection_and_recognition_b200._lib import FfrError
    with pytest.raises(TypeError):
        ops.match_pairs(torch.zeros(2, 128), torch.zeros(4, 128), 0.5)
    with pytest.raises(TypeError):
        ops.self_pairs(torch.zeros(4, 128), 0.5)
    with pytest.raises(FfrError):
        ops.self_pairs(torch.zeros(4, 128, dtype=torch.float16), 0.5)
    with pytest.raises(FfrError):
        ops.match_pairs(torch.zeros(2, 128, dtype=torch.float16), torch.zeros(4, 128, dtype=torch.float16), 0.5)
