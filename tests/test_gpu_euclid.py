"""Euclid gallery filtering on the tensor cores (K1 + K2 with the per-reference bias + K3 Euclid form + the value pass).

Contract (DESIGN.md section 5): best_idx equals the exact fp32 CUDA-core result (FFR_FLAG_FORCE_FP32) except on rows whose two
smallest fp64 distances differ by less than 1e-6 relative (fp32 ties); keep and best_val are bit-identical to it wherever the index
agrees; the band list is exact.  Against the NumPy oracle: distances within 1e-3 relative (absolute below 1), keep exact outside
the fp64 band of the threshold.
"""
import glob
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import oracle

pytestmark = pytest.mark.gpu

TIE_REL = 1e-6          # fp32 ties: the two smallest fp64 distances closer than this (relative)
VAL_REL = 1e-3


@pytest.fixture(scope="module")
def ops(ffr_lib, cuda_dev):
    from face_detection_and_recognition_b200 import ops as _ops
    return _ops


def _dist64(ref, cand, block=2048):
    """fp64 shadow: (smallest, second smallest) distance per candidate row.  |c|^2 + |r|^2 - 2 c.r in fp64: its cancellation
    error (~1e-16 of the squared norms) is far below the 1e-6 relative tie bar for these data."""
    r = ref.astype(np.float64)
    rr = np.einsum("ij,ij->i", r, r)
    d1 = np.empty(len(cand))
    d2 = np.empty(len(cand))
    for s in range(0, len(cand), block):
        c = cand[s:s + block].astype(np.float64)
        d = np.sqrt(np.maximum(rr[:, None] + np.einsum("ij,ij->i", c, c)[None, :] - 2.0 * (r @ c.T), 0.0))
        if d.shape[0] == 1:
            d1[s:s + block], d2[s:s + block] = d[0], np.inf
            continue
        part = np.partition(d, 1, axis=0)
        d1[s:s + block], d2[s:s + block] = part[0], part[1]
    return d1, d2


def _run(ops, ref, cand, thr, flags=0, band_tol=1e-3, base=0):
    dev = torch.device("cuda:0")
    res = ops.face_filter(torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), thr, metric="euclid",
                          band_tol=band_tol, flags=flags, want_stats=True, ref_index_base=base)
    torch.cuda.synchronize()
    return res


def _check_euclid(ops, ref, cand, thr, sample=None, base=0):
    """Default routing (tcgen05) against FORCE_FP32 (K2s) on all rows and against the oracle + fp64 shadow on ``sample``."""
    res = _run(ops, ref, cand, thr, base=base)
    assert res.stats["path"] == "tcgen05", res.stats
    exact = _run(ops, ref, cand, thr, flags=ops.FLAG_FORCE_FP32, base=base)
    assert exact.stats["path"] == "fp32", exact.stats
    keep, idx, val = res.keep.cpu().numpy(), res.best_idx.cpu().numpy(), res.best_val.cpu().numpy()
    ke, ie, ve = exact.keep.cpu().numpy(), exact.best_idx.cpu().numpy(), exact.best_val.cpu().numpy()
    rows = np.arange(len(cand)) if sample is None else np.sort(np.asarray(sample))
    d1, d2 = _dist64(ref, cand[rows])
    tie = (d2 - d1) <= TIE_REL * np.maximum(d1, 1e-30)
    # identity with the exact path
    same = idx == ie
    bad = np.flatnonzero(~same[rows] & ~tie)
    assert bad.size == 0, (f"{bad.size} index mismatches vs FORCE_FP32 outside fp32 ties, rows {rows[bad[:5]]} got "
                           f"{idx[rows[bad[:5]]]} want {ie[rows[bad[:5]]]} stats {res.stats}")
    assert np.array_equal(keep[same], ke[same]) and np.array_equal(val[same].view(np.uint32), ve[same].view(np.uint32))
    assert np.mean(same) > 0.999, np.mean(same)
    agree = set(np.flatnonzero(same).tolist())
    band, band_e = set(res.band_rows.cpu().numpy().tolist()), set(exact.band_rows.cpu().numpy().tolist())
    assert band & agree == band_e & agree
    # against the oracle
    ko, io, so = oracle.filter_euclid(ref, cand[rows], thr)
    k, i, v = keep[rows], idx[rows] - base, val[rows]
    assert np.all(np.abs(v - so) <= VAL_REL * np.maximum(1.0, so)), np.max(np.abs(v - so) / np.maximum(1.0, so))
    bad = np.flatnonzero((i != io) & ~tie)
    assert bad.size == 0, (bad.size, rows[bad[:5]], i[bad[:5]], io[bad[:5]])
    near = np.abs(d1 - thr) <= TIE_REL * max(1.0, thr)
    bad = np.flatnonzero((k != ko) & ~near)
    assert bad.size == 0, (bad.size, rows[bad[:5]], d1[bad[:5]])
    return res


def _planted(ref, n_cand, dim, thr, seed, scale=1.0):
    """Candidates that sit on the decision surfaces: at distance thr * (1 +- u) of a chosen reference, equidistant from two
    references (within 1e-5 relative), with two references a hair apart (beyond fp32 noise, inside the fp16 window), and zero
    rows."""
    rng = np.random.default_rng(seed)
    n = len(ref)
    out = []
    for _ in range(n_cand // 4):
        k = rng.integers(0, n)
        u = rng.uniform(-2e-3, 2e-3)
        g = rng.standard_normal(dim)
        out.append(ref[k] + g / np.linalg.norm(g) * thr * (1 + u))
    for _ in range(n_cand // 4):
        a, b = rng.choice(n, 2, replace=False)
        eps = rng.uniform(-1e-5, 1e-5)
        out.append(0.5 * (ref[a] + ref[b]) + eps * (ref[a] - ref[b]))
    for _ in range(n_cand // 4):
        a, b = rng.choice(n, 2, replace=False)
        eps = rng.uniform(2e-5, 2e-4) * rng.choice([-1, 1])
        out.append(0.5 * (ref[a] + ref[b]) + eps * (ref[a] - ref[b]))
    while len(out) < n_cand:
        out.append(np.zeros(dim))
    return (np.asarray(out) * scale).astype(np.float32)


SHAPES = [(9, 1000, 128), (40, 200, 128), (257, 50_000, 100), (300, 20_000, 130), (1000, 100_000, 128),
          (6144, 80_000, 512), (4097, 80_000, 256), (10_000, 200_000, 512)]


@pytest.mark.parametrize("unit_norm", [True, False])
@pytest.mark.parametrize("n_ref,n_cand,dim", SHAPES)
def test_euclid_parity(ops, n_ref, n_cand, dim, unit_norm):
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=n_ref + dim, unit_norm=unit_norm)
    thr = 0.9 if unit_norm else 4.0
    n_adv = min(400, n_cand // 4)
    cand[:n_adv] = _planted(ref, n_adv, dim, thr, seed=n_ref)
    cand[n_adv] = 0.0
    ref[n_ref // 2] = 0.0
    rng = np.random.default_rng(7)
    sample = None if n_cand * n_ref <= 2e8 else np.unique(np.r_[np.arange(n_adv + 1), rng.choice(n_cand, 1500, replace=False)])
    _check_euclid(ops, ref, cand, thr, sample=sample)


def test_euclid_norm_spread(ops):
    """Row norms from 1e-3 to 1e3 (log-uniform): the per-row window grows with max|bias| / |c|; tiny rows are rescanned."""
    rng = np.random.default_rng(5)
    n_ref, n_cand, dim = 600, 30_000, 128
    ref = rng.standard_normal((n_ref, dim)).astype(np.float32)
    ref *= (10.0 ** rng.uniform(-3, 3, (n_ref, 1)) / np.linalg.norm(ref, axis=1, keepdims=True)).astype(np.float32)
    k = rng.integers(0, n_ref, n_cand)
    cand = (ref[k] * (1 + 0.3 * rng.standard_normal((n_cand, 1))) +
            0.05 * np.linalg.norm(ref[k], axis=1, keepdims=True) * rng.standard_normal((n_cand, dim)) / np.sqrt(dim))
    cand = cand.astype(np.float32)
    sample = np.unique(np.r_[np.arange(300), rng.choice(n_cand, 3000, replace=False)])
    _check_euclid(ops, ref, cand, 1.0, sample=sample)


def test_euclid_duplicates_folded(ops):
    """Exact copies among >= 2048 references with the fold engaged: the first occurrence wins; near copies go to K3."""
    n_ref, n_cand, dim = 4096, 500_000, 128
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=11, unit_norm=False)
    rng = np.random.default_rng(3)
    ref[rng.choice(np.arange(n_ref // 2, n_ref - 50), 300, replace=False)] = ref[rng.integers(0, n_ref // 2, 300)]
    near = rng.integers(0, n_ref // 2, 50)
    ref[n_ref - 50:] = ref[near] * (1 + 1e-5 * rng.standard_normal((50, dim))).astype(np.float32)
    k = np.r_[near, rng.integers(0, n_ref, 950)]
    cand[:1000] = ref[k] + 0.01 * rng.standard_normal((1000, dim)).astype(np.float32)
    sample = np.unique(np.r_[np.arange(1000), rng.choice(n_cand, 1000, replace=False)])
    res = _check_euclid(ops, ref, cand, 3.0, sample=sample)
    assert res.stats["refs_scanned"] < n_ref, res.stats


def test_euclid_index_base_and_empty(ops):
    ref, cand = oracle.make_synthetic(50, 3000, 128, seed=4, unit_norm=False)
    _check_euclid(ops, ref, cand, 4.0, base=1000)
    res = ops.face_filter(torch.from_numpy(ref).cuda(), torch.zeros((0, 128), device="cuda"), 4.0, metric="euclid")
    assert res.keep.numel() == 0


def test_euclid_host_filter_chunks(ops):
    from face_detection_and_recognition_b200.ops import HostFilter
    ref, cand = oracle.make_synthetic(700, 50_000, 128, seed=8, unit_norm=False)
    hf = HostFilter(device=0, max_ref=1024, chunk_cand=16_384, max_dim=512)
    keep, idx, val = hf(ref, cand, 4.0, metric="euclid")
    hf.close()
    dev = _run(ops, ref, cand, 4.0)
    assert dev.stats["path"] == "tcgen05"
    assert np.array_equal(keep, dev.keep.cpu().numpy()) and np.array_equal(idx, dev.best_idx.cpu().numpy())
    assert np.array_equal(val.view(np.uint32), dev.best_val.cpu().numpy().view(np.uint32))


def test_euclid_graphed_replay(ops):
    ref, cand = oracle.make_synthetic(1000, 20_000, 128, seed=9, unit_norm=False)
    r, c = torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda()
    g = ops.GraphedFilter.capture(r, c, 4.0, metric="euclid")
    c.mul_(1.5)                                                     # replay sees the new contents
    out = g.replay()
    torch.cuda.synchronize()
    eager = ops.face_filter(r, c, 4.0, metric="euclid")
    torch.cuda.synchronize()
    assert torch.equal(out.keep, eager.keep) and torch.equal(out.best_idx, eager.best_idx)
    assert torch.equal(out.best_val, eager.best_val)


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
    ref, cand = oracle.make_synthetic(300, 20_003, 128, seed=13, unit_norm=False)
    sh = CandidateSharder(rank, world, device=rank, gather="nccl")
    a, b, _ = sh.local_range(len(cand))
    keep, idx, _ = sh.filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand[a:b]).cuda(), 4.0, len(cand), metric="euclid")
    torch.cuda.synchronize()
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), keep=keep.cpu().numpy(), idx=idx.cpu().numpy())
    sh.close()
    dist.destroy_process_group()


def test_euclid_sharded_nccl(ops, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    ref, cand = oracle.make_synthetic(300, 20_003, 128, seed=13, unit_norm=False)
    one = _run(ops, ref, cand, 4.0)
    for r in range(2):
        g = np.load(tmp_path / f"r{r}.npz")
        assert np.array_equal(g["keep"], one.keep.cpu().numpy()) and np.array_equal(g["idx"], one.best_idx.cpu().numpy())


def test_euclid_cli_gallery(tmp_path, ops):
    from face_detection_and_recognition_b200.filter_faces_using_reference import main
    from test_dropin_cli import StubModel, _embed, _make_dataset
    rng = np.random.default_rng(2)
    ud, rd = _make_dataset(str(tmp_path), rng, classes=("carol",), n_ref=12, n_cand=30)
    td = str(tmp_path / "out")
    model = StubModel()
    refs = sorted(glob.glob(os.path.join(rd, "carol", "*.jpg")))
    cands = sorted(glob.glob(os.path.join(ud, "carol", "*.jpg")))
    er, ec = _embed(model, refs), _embed(model, cands)
    d1, _ = _dist64(er, ec)
    thr = float(np.median(d1))
    main(["--ud", ud, "--rd", rd, "--td", td, "--gallery", "--metric", "euclid", "--threshold", str(thr), "-r", "12"], model=model)
    ko, _, _ = oracle.filter_euclid(er, ec, thr)
    assert 0 < ko.sum() < len(ko)
    for p, k, d in zip(cands, ko, d1):
        if abs(d - thr) > 1e-6 * max(1.0, thr):
            assert os.path.exists(os.path.join(td, "clean" if k else "unclean", "carol", os.path.basename(p)))


def test_euclid_routing_unchanged(ops):
    """n_ref <= 8, FLAG_NO_RECHECK and dim > 512 keep the exact K2s path; fp16 rows and FORCE_MMA with n_ref <= 8 are refused."""
    from face_detection_and_recognition_b200._lib import FfrError
    dev = torch.device("cuda:0")
    ref, cand = oracle.make_synthetic(8, 2000, 128, seed=1, unit_norm=False)
    assert _run(ops, ref, cand, 4.0).stats["path"] == "fp32"
    ref, cand = oracle.make_synthetic(100, 2000, 128, seed=1, unit_norm=False)
    assert _run(ops, ref, cand, 4.0, flags=ops.FLAG_NO_RECHECK).stats["path"] == "fp32"
    ref, cand = oracle.make_synthetic(100, 2000, 640, seed=1, unit_norm=False)
    assert _run(ops, ref, cand, 4.0).stats["path"] == "fp32"
    ref, cand = oracle.make_synthetic(100, 256, 128, seed=1)
    r16 = ops.l2norm_rows(torch.from_numpy(ref).to(dev), want_f16=True, want_f32=False)["f16"]
    c16 = ops.l2norm_rows(torch.from_numpy(cand).to(dev), want_f16=True, want_f32=False)["f16"]
    with pytest.raises(FfrError):
        ops.face_filter(r16, c16, 0.5, metric="euclid")
    with pytest.raises(FfrError):
        ops.face_filter(torch.from_numpy(ref[:8]).to(dev), torch.from_numpy(cand).to(dev), 0.5, metric="euclid",
                        flags=ops.FLAG_FORCE_MMA)
