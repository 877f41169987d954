"""Gallery (reference-axis) sharding: every rank holds a contiguous range of the references and all candidates, and one max
all-reduce of a packed {value, index} key per candidate merges the ranks.  CPU: gloo processes with an fp32 filter injected
(ranges, key order, cross-rank ties, empty shards, identical results everywhere).  GPU: the real filter and the library's NCCL
all-reduce (ffr_allreduce_best) on every visible GPU, checked against the one-GPU call on the whole gallery."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import oracle


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _exact_filter(ref, cand, thr, metric="cosine", ref_index_base=0):
    """fp32 result of each pair computed in fp64 and rounded: a pair's value does not depend on the shard it sits in."""
    r, c = ref.numpy().astype(np.float64), cand.numpy().astype(np.float64)
    if metric == "cosine":
        s = (c @ r.T) / np.outer(np.linalg.norm(c, axis=1), np.linalg.norm(r, axis=1))
        s = s.astype(np.float32)
        i = np.argmax(s, axis=1)
        keep = s[np.arange(len(c)), i] >= thr
    else:
        s = np.sqrt(((c[:, None, :] - r[None, :, :]) ** 2).sum(-1)).astype(np.float32)
        i = np.argmin(s, axis=1)
        keep = s[np.arange(len(c)), i] <= thr
    v = s[np.arange(len(c)), i]
    return SimpleNamespace(keep=torch.from_numpy(keep.astype(np.uint8)), best_idx=torch.from_numpy((i + ref_index_base).astype(np.int32)),
                           best_val=torch.from_numpy(v))


def _gallery(n_ref, n_cand, dim, metric, seed):
    """Synthetic gallery whose last reference is an exact copy of reference 0 (a tie that crosses ranks: the copy sits in the
    last shard) with a few candidates planted next to it."""
    ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=seed, n_adversarial=min(8, n_cand), unit_norm=metric == "cosine")
    if n_ref >= 2:
        ref[-1] = ref[0]
        rng = np.random.default_rng(seed)
        for j in range(0, n_cand, 5):
            cand[j] = ref[0] + 0.05 * rng.standard_normal(dim).astype(np.float32)
    return ref, cand


def test_gallery_shard_range():
    from face_detection_and_recognition_b200.sharding import GallerySharder, shard_range
    for n in (1, 2, 7, 1000, 1001):
        for world in (1, 2, 3, 8):
            covered = []
            for r in range(world):
                sh = GallerySharder(r, world, reduce="dist", filter_fn=_exact_filter)
                a, b = sh.shard_range(n)
                assert (a, b) == shard_range(n, world, r)[:2]
                covered += list(range(a, b))
            assert covered == list(range(n))
    with pytest.raises(ValueError):
        GallerySharder(0, 2, reduce="dist")              # "dist" merges best_val as it is: an fp32 filter must be injected
    with pytest.raises(ValueError):
        GallerySharder(0, 2, reduce="allgather", filter_fn=_exact_filter)


def test_best_key_order():
    """Larger cosine score wins, smaller Euclid distance wins, equal values go to the lower index, idx < 0 is the identity."""
    from face_detection_and_recognition_b200.sharding import pack_best_keys, unpack_best_keys
    idx = torch.tensor([5, 3, 7, 2, 9, -1], dtype=torch.int32)
    cos = torch.tensor([0.5, 0.5, 0.9, -0.2, float("-inf"), 1.0])
    k = pack_best_keys(cos, idx, "cosine")
    order = torch.argsort(k, descending=True).tolist()
    assert order == [2, 1, 0, 3, 4, 5]
    dist = torch.tensor([0.5, 0.5, 0.1, 3.0, 0.0, 0.0])
    k = pack_best_keys(dist, idx, "euclid")
    assert torch.argsort(k, descending=True).tolist() == [4, 2, 1, 0, 3, 5]
    for metric, v in (("cosine", cos), ("euclid", dist)):
        v2, i2 = unpack_best_keys(pack_best_keys(v, idx, metric), metric)
        assert torch.equal(i2, idx)
        assert torch.equal(v2[:5], v[:5])
        assert v2[5].item() == (float("inf") if metric == "euclid" else float("-inf"))


def _gloo_worker(rank, world, port, cases, out_dir):
    import torch.distributed as dist
    from face_detection_and_recognition_b200.sharding import GallerySharder
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    sh = GallerySharder(rank, world, reduce="dist", filter_fn=_exact_filter)
    for ci, (metric, n_ref, n_cand, dim, thr) in enumerate(cases):
        ref, cand = _gallery(n_ref, n_cand, dim, metric, seed=100 + ci)
        a, b = sh.shard_range(n_ref)
        res = sh.filter(torch.from_numpy(ref[a:b]), torch.from_numpy(cand), thr, n_ref, metric=metric, band_tol=0.05)
        np.savez(os.path.join(out_dir, f"c{ci}_r{rank}.npz"), keep=res.keep.numpy(), idx=res.best_idx.numpy(),
                 val=res.best_val.numpy(), band=res.band_rows.numpy())
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_gallery_sharding_gloo(tmp_path, world):
    # (n_ref = 2 with world 3 and n_ref = 1: ranks without references)
    cases = [("cosine", 301, 97, 32, 0.5), ("euclid", 301, 97, 32, 0.9), ("cosine", 2, 40, 16, 0.3), ("euclid", 1, 10, 16, 1.0)]
    mp.spawn(_gloo_worker, args=(world, _free_port(), cases, str(tmp_path)), nprocs=world, join=True)
    for ci, (metric, n_ref, n_cand, dim, thr) in enumerate(cases):
        ref, cand = _gallery(n_ref, n_cand, dim, metric, seed=100 + ci)
        want = _exact_filter(torch.from_numpy(ref), torch.from_numpy(cand), thr, metric=metric)
        r0 = np.load(tmp_path / f"c{ci}_r0.npz")
        for r in range(world):
            g = np.load(tmp_path / f"c{ci}_r{r}.npz")
            for key in ("keep", "idx", "val", "band"):
                assert np.array_equal(g[key].view(np.uint8), r0[key].view(np.uint8)), (ci, r, key)
        assert np.array_equal(r0["idx"], want.best_idx.numpy()), ci
        assert np.array_equal(r0["val"], want.best_val.numpy()), ci
        assert np.array_equal(r0["keep"], want.keep.numpy()), ci
        band = np.nonzero(np.abs(want.best_val.numpy() - thr) <= 0.05)[0]
        assert np.array_equal(r0["band"], band), ci
        if n_ref >= 2:     # planted rows: the copy of reference 0 in the last shard never wins the tie
            assert not np.any(r0["idx"] == n_ref - 1), ci


def test_allreduce_best_workspace_bytes(ffr_lib):
    assert ffr_lib.ffr_allreduce_best_workspace_bytes(-1) == 0
    assert ffr_lib.ffr_allreduce_best_workspace_bytes(0) == 256
    assert ffr_lib.ffr_allreduce_best_workspace_bytes(1) == 256
    assert ffr_lib.ffr_allreduce_best_workspace_bytes(1000) == 8192
    assert ffr_lib.ffr_allreduce_best_workspace_bytes(10 ** 6) == 8 * 10 ** 6


# ---- GPU ----------------------------------------------------------------------------------------------------------------
_GPU_CASES = [("cosine", 50_003, 1000, 128, 0.5), ("euclid", 50_003, 1000, 128, 6.0), ("cosine", 20_000, 1, 512, 0.5),
              ("euclid", 30_001, 100, 256, 9.0), ("cosine", 7, 300, 64, 0.5), ("euclid", 7, 300, 64, 3.0)]


def _nccl_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from face_detection_and_recognition_b200.sharding import GallerySharder
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    sh = GallerySharder(rank, world, device=rank, reduce="nccl")
    for ci, (metric, n_ref, n_cand, dim, thr) in enumerate(_GPU_CASES):
        ref, cand = _gallery(n_ref, n_cand, dim, metric, seed=200 + ci)
        a, b = sh.shard_range(n_ref)
        ref_local = torch.from_numpy(ref[a:b]).cuda() if b > a else None
        res = sh.filter(ref_local, torch.from_numpy(cand).cuda(), thr, n_ref, metric=metric, band_tol=1e-3)
        torch.cuda.synchronize()
        np.savez(os.path.join(out_dir, f"c{ci}_r{rank}.npz"), keep=res.keep.cpu().numpy(), idx=res.best_idx.cpu().numpy(),
                 val=res.best_val.cpu().numpy(), band=res.band_rows.cpu().numpy())
    sh.close()
    dist.destroy_process_group()


def _check_against_one_gpu(metric, ref, cand, thr, keep, idx, val, band):
    """The one-GPU gallery contract over the whole gallery (DESIGN.md section 5), against face_filter on cuda:0."""
    from face_detection_and_recognition_b200 import ops
    one = ops.face_filter(torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda(), thr, metric=metric, band_tol=1e-3)
    torch.cuda.synchronize()
    k1, i1, v1 = one.keep.cpu().numpy(), one.best_idx.cpu().numpy(), one.best_val.cpu().numpy()
    if metric == "cosine":
        ko, io, so = oracle.filter_cosine(ref, cand, thr)
        _, _, s64 = oracle.filter_cosine(ref, cand, thr, dtype=np.float64)
        rn = ref / np.linalg.norm(ref, axis=1, keepdims=True)
        cn = cand / np.linalg.norm(cand, axis=1, keepdims=True)
        pair = lambda i: np.einsum("ij,ij->i", cn.astype(np.float64), rn[i].astype(np.float64))   # noqa: E731
    else:
        ko, io, so = oracle.filter_euclid(ref, cand, thr)
        _, _, s64 = oracle.filter_euclid(ref, cand, thr, dtype=np.float64)
        pair = lambda i: np.linalg.norm(cand.astype(np.float64) - ref[i].astype(np.float64), axis=1)   # noqa: E731
    # index: the oracle's except on fp32 ties (the two references' exact values within 1e-6)
    tie = np.abs(pair(idx) - pair(io)) <= 1e-6 * np.maximum(1.0, np.abs(s64))
    assert np.all((idx == io) | tie), np.nonzero(~((idx == io) | tie))[0][:10]
    far = np.abs(s64 - thr) > 1e-6
    assert np.array_equal(keep[far], ko[far])
    assert np.max(np.abs(val - so)) < 1e-5 * max(1.0, float(np.max(np.abs(so))))
    assert np.array_equal(band, np.nonzero(np.abs(val - thr) <= 1e-3)[0])
    agree = idx == i1
    assert agree.mean() > 0.999
    if metric == "euclid":          # bit-identical to the one-GPU call wherever the index agrees
        assert np.array_equal(val[agree].view(np.uint32), v1[agree].view(np.uint32))
        assert np.array_equal(keep[agree], k1[agree])
    else:
        assert np.max(np.abs(val - v1)) < 1e-3


@pytest.mark.gpu
def test_gallery_sharding_nccl(tmp_path, ffr_lib, cuda_dev):
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs two or more GPUs")
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for ci, (metric, n_ref, n_cand, dim, thr) in enumerate(_GPU_CASES):
        ref, cand = _gallery(n_ref, n_cand, dim, metric, seed=200 + ci)
        r0 = np.load(tmp_path / f"c{ci}_r0.npz")
        for r in range(1, world):
            g = np.load(tmp_path / f"c{ci}_r{r}.npz")
            for key in ("keep", "idx", "val", "band"):
                assert np.array_equal(g[key].view(np.uint8), r0[key].view(np.uint8)), (ci, r, key)
        assert not np.any(r0["idx"] == n_ref - 1), ci          # the cross-rank copy of reference 0 loses the tie
        _check_against_one_gpu(metric, ref, cand, thr, r0["keep"], r0["idx"], r0["val"], r0["band"])


@pytest.mark.gpu
@pytest.mark.parametrize("metric,thr", [("cosine", 0.5), ("euclid", 6.0)])
def test_allreduce_best_single_rank(ffr_lib, cuda_dev, metric, thr):
    """World 1: the merge pass alone.  best_val becomes the fp32 value of the chosen reference (cosine: within fp32 rounding of
    the oracle even where face_filter reports the fp16-operand score), the index is face_filter's, Euclid bit-identical."""
    from face_detection_and_recognition_b200 import ops
    rg = ops.ResultGather(0, 1, 0)
    ref, cand = _gallery(20_011, 2000, 128, metric, seed=7)
    r, c = torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda()
    base = 1000
    one = ops.face_filter(r, c, thr, metric=metric, ref_index_base=base)
    res = rg.allreduce_best(r, c, thr, one.best_idx, ref_index_base=base, metric=metric, band_tol=1e-3)
    torch.cuda.synchronize()
    idx = res.best_idx.cpu().numpy()
    assert np.array_equal(idx, one.best_idx.cpu().numpy())
    _check_against_one_gpu(metric, ref, cand, thr, res.keep.cpu().numpy(), idx - base, res.best_val.cpu().numpy(),
                           res.band_rows.cpu().numpy())
    # a rank without references contributes the identity: nothing found
    empty = rg.allreduce_best(None, c, thr, torch.full((2000,), -1, dtype=torch.int32, device="cuda"), metric=metric)
    torch.cuda.synchronize()
    assert torch.all(empty.best_idx == -1) and torch.all(empty.keep == 0)
    assert torch.all(empty.best_val == (float("inf") if metric == "euclid" else float("-inf")))
    rg.close()


@pytest.mark.gpu
@pytest.mark.parametrize("metric,thr", [("cosine", 0.5), ("euclid", 6.0)])
def test_allreduce_best_unaligned_candidates(ffr_lib, cuda_dev, metric, thr):
    """A contiguous candidate view that starts 4 bytes into its storage (dim % 4 == 0, aligned gallery): the merge pass takes
    its scalar form instead of reading the rows as float4, and returns the aligned call's index with values within fp32
    rounding of it."""
    from face_detection_and_recognition_b200 import ops
    rg = ops.ResultGather(0, 1, 0)
    ref, cand = _gallery(5003, 777, 128, metric, seed=9)
    r, c = torch.from_numpy(ref).cuda(), torch.from_numpy(cand).cuda()
    storage = torch.empty(c.numel() + 1, dtype=torch.float32, device="cuda")
    c_off = storage[1:].view(c.shape)
    c_off.copy_(c)
    assert c_off.is_contiguous() and c_off.data_ptr() % 16 == 4
    idx = ops.face_filter(r, c, thr, metric=metric).best_idx
    a = rg.allreduce_best(r, c, thr, idx, metric=metric)
    b = rg.allreduce_best(r, c_off, thr, idx, metric=metric)
    torch.cuda.synchronize()
    assert torch.equal(a.best_idx, b.best_idx)
    assert torch.max(torch.abs(a.best_val - b.best_val)).item() <= 1e-6 * max(1.0, torch.max(torch.abs(a.best_val)).item())
    far = torch.abs(a.best_val - thr) > 1e-5
    assert torch.equal(a.keep[far], b.keep[far])
    rg.close()


@pytest.mark.gpu
def test_allreduce_best_rejects_bad_best_idx(ffr_lib, cuda_dev):
    from face_detection_and_recognition_b200 import ops
    rg = ops.ResultGather(0, 1, 0)
    r, c = torch.randn(100, 64, device="cuda"), torch.randn(10, 64, device="cuda")
    for bad in (torch.zeros(9, dtype=torch.int32, device="cuda"), torch.zeros(10, dtype=torch.int64, device="cuda"),
                torch.zeros(10, dtype=torch.int32)):
        with pytest.raises(ValueError):
            rg.allreduce_best(r, c, 0.5, bad)
    rg.close()
