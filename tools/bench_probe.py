"""Small probe batches against large galleries: the one-GPU call, and the gallery sharded over the GPUs of the box.

One GPU: probes {1, 16, 256, 1000, 4096} x galleries {1 M x 512, 10 M x 128}, cosine and Euclid, ``face_filter`` on the
whole gallery.  CUDA events around each call after a warm-up (inputs resident; the gallery is larger than L2), and around the
tensor-core kernel K2 alone (the library's K2 event hook).  At 1000 probes, the first 16 are verified against the oracle
over the whole gallery: index mismatches outside fp32 ties (fp64 shadow) and keep mismatches outside 1e-6 of the threshold.

Gallery over GPUs: 1000 probes x 10 M x 128, cosine and Euclid, ``sharding.GallerySharder`` (NCCL) on 1, 2, 4 and 8 GPUs (as
many as are visible), one process per GPU.  Rank 0 times the whole sharded call with a host clock: every rank synchronises and
meets at a barrier before the call, and rank 0's call ends in a device synchronise after the all-reduce, which needs every
rank's contribution.  Strong scaling is against world 1 in the same run.  Each world's merged result is compared with the
plain one-GPU ``face_filter`` on the whole gallery (rank 0, same data): index agreement, keep where the index agrees, and the
value where the index agrees -- bit for bit (the Euclid contract) and as the largest difference (cosine: the plain call
returns fp16-operand scores for rows its re-check did not visit, the merge fp32 values).

Device name, power limit and max SM clock are read in the same run.

    python tools/bench_probe.py [--reps 20] [--out profiles/r05_bench_probe.jsonl] [--skip-one-gpu] [--skip-sharded]
"""
import argparse
import json
import os
import socket
import subprocess
import sys
import time

import numpy as np
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GALLERIES = [(1_000_000, 512), (10_000_000, 128)]
PROBES = [1, 16, 256, 1000, 4096]
THR = {"cosine": 0.5, "euclid": 1.0}


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unavailable"
    return {"device": name, "power_limit_and_max_sm_clock": out, "sms": torch.cuda.get_device_properties(0).multi_processor_count,
            "gpus": torch.cuda.device_count()}


def make_gallery(n_ref, dim, metric, dev, seed=1):
    """Seeded on the device (identical on every GPU): unit-norm rows for cosine, norms in [0.5, 2] for Euclid."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    ref = torch.randn((n_ref, dim), generator=g, device=dev)
    ref /= ref.norm(dim=1, keepdim=True)
    if metric == "euclid":
        ref *= 0.5 + 1.5 * torch.rand((n_ref, 1), generator=g, device=dev)
    return ref


def make_probes(ref, n, seed=2):
    """Half the probes are noisy copies of gallery rows (a match exists), half independent noise."""
    g = torch.Generator(device=ref.device)
    g.manual_seed(seed)
    cand = torch.randn((n, ref.shape[1]), generator=g, device=ref.device)
    cand /= cand.norm(dim=1, keepdim=True)
    k = n // 2
    if k:
        pick = torch.randint(0, ref.shape[0], (k,), generator=g, device=ref.device)
        cand[:k] = ref[pick] + 0.03 * cand[:k] * ref[pick].norm(dim=1, keepdim=True)
    return cand.contiguous()


def verify(ref, cand, res, metric, thr, n=16):
    """The first n probes against the oracle over the whole gallery; ties and the threshold band from fp64 values of the pairs."""
    from oracle import oracle
    r, c = ref.cpu().numpy(), cand[:n].cpu().numpy()
    f = oracle.filter_cosine if metric == "cosine" else oracle.filter_euclid
    ko, io, _ = f(r, c, thr)
    idx, keep = res.best_idx[:n].cpu().numpy(), res.keep[:n].cpu().numpy()
    c64 = c.astype(np.float64)
    if metric == "cosine":
        c64 /= np.linalg.norm(c64, axis=1, keepdims=True)
        pair = lambda i: np.einsum("ij,ij->i", c64, r[i] / np.linalg.norm(r[i].astype(np.float64), axis=1, keepdims=True))   # noqa: E731
    else:
        pair = lambda i: np.linalg.norm(c64 - r[i].astype(np.float64), axis=1)   # noqa: E731
    s64 = pair(io)
    tie = np.abs(pair(idx) - s64) <= 1e-6 * np.maximum(1.0, np.abs(s64))
    far = np.abs(s64 - thr) > 1e-6
    return {"verified_probes": int(len(c)), "verified_pairs": int(len(c) * len(r)),
            "idx_mismatch_outside_ties": int(np.sum((idx != io) & ~tie)), "keep_mismatch_outside_band": int(np.sum((keep != ko) & far))}


def one_gpu(reps, info, out):
    from face_detection_and_recognition_b200 import _lib, ops
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    e0, e1, k0, k1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    k0.record(); k1.record()                # materialise the cudaEvent_t handles the library records into
    for n_ref, dim in GALLERIES:
        for metric in ("cosine", "euclid"):
            ref = make_gallery(n_ref, dim, metric, dev)
            for n in PROBES:
                cand = make_probes(ref, n)
                thr = THR[metric]
                for _ in range(2):
                    res = ops.face_filter(ref, cand, thr, metric=metric)
                call, k2 = [], []
                lib.ffr_debug_set_k2_events(k0.cuda_event, k1.cuda_event)
                for _ in range(reps):
                    e0.record()
                    res = ops.face_filter(ref, cand, thr, metric=metric)
                    e1.record()
                    torch.cuda.synchronize()
                    call.append(e0.elapsed_time(e1))
                    k2.append(k0.elapsed_time(k1))
                lib.ffr_debug_set_k2_events(None, None)
                stats = ops.face_filter(ref, cand, thr, metric=metric, want_stats=True).stats
                row = {"kind": "one_gpu", **info, "metric": metric, "n_ref": n_ref, "dim": dim, "probes": n,
                       "call_ms_median": float(np.median(call)), "k2_ms_median": float(np.median(k2)),
                       "k2_tiles_of_probes": -(-n // 256), "path": stats["path"], "k2_grid": stats.get("k2", {}).get("grid"),
                       **(verify(ref, cand, res, metric, thr) if n == 1000 else {})}
                print(json.dumps(row), flush=True)
                out.write(json.dumps(row) + "\n")
            del ref
            torch.cuda.empty_cache()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_worker(rank, world, port, reps, n_ref, dim, n_probes, metric, out_dir):
    import torch.distributed as dist
    from face_detection_and_recognition_b200.sharding import GallerySharder
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    sh = GallerySharder(rank, world, device=rank, reduce="nccl")
    full = make_gallery(n_ref, dim, metric, dev)
    cand = make_probes(full, n_probes)
    a, b = sh.shard_range(n_ref)
    thr = THR[metric]
    if rank == 0:       # the plain one-GPU call on the whole gallery: what every world's merged result is compared with
        from face_detection_and_recognition_b200 import ops
        one = ops.face_filter(full, cand, thr, metric=metric)
        np.savez(os.path.join(out_dir, f"plain{world}_{metric}.npz"), keep=one.keep.cpu().numpy(),
                 idx=one.best_idx.cpu().numpy(), val=one.best_val.cpu().numpy())
        del one
    ref = full[a:b].clone()
    del full
    torch.cuda.empty_cache()
    for _ in range(3):
        res = sh.filter(ref, cand, thr, n_ref, metric=metric)
    times = []
    for _ in range(reps):
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        res = sh.filter(ref, cand, thr, n_ref, metric=metric)
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    if rank == 0:
        np.savez(os.path.join(out_dir, f"w{world}_{metric}.npz"), keep=res.keep.cpu().numpy(), idx=res.best_idx.cpu().numpy(),
                 val=res.best_val.cpu().numpy(), times=np.array(times))
    sh.close()
    dist.destroy_process_group()


def sharded(reps, info, out, out_dir):
    n_ref, dim, n_probes = 10_000_000, 128, 1000
    worlds = [w for w in (1, 2, 4, 8) if w <= torch.cuda.device_count()]
    for metric in ("cosine", "euclid"):
        for w in worlds:
            mp.spawn(_sharded_worker, args=(w, _free_port(), reps, n_ref, dim, n_probes, metric, out_dir), nprocs=w, join=True)
        t1 = float(np.median(np.load(os.path.join(out_dir, f"w1_{metric}.npz"))["times"]))
        for w in worlds:
            g = np.load(os.path.join(out_dir, f"w{w}_{metric}.npz"))
            plain = np.load(os.path.join(out_dir, f"plain{w}_{metric}.npz"))
            agree = g["idx"] == plain["idx"]
            dv = g["val"][agree] - plain["val"][agree]
            row = {"kind": "gallery_sharded", **info, "metric": metric, "n_ref": n_ref, "dim": dim, "probes": n_probes, "gpus": w,
                   "call_ms_median": float(np.median(g["times"])), "call_ms_min": float(np.min(g["times"])),
                   "speedup_vs_1gpu": t1 / float(np.median(g["times"])),
                   "vs_plain_face_filter": {"idx_agree": float(agree.mean()),
                                            "keep_mismatch_where_idx_agrees": int(np.sum(g["keep"][agree] != plain["keep"][agree])),
                                            "val_bit_mismatch_where_idx_agrees": int(np.sum(g["val"][agree].view(np.uint32) != plain["val"][agree].view(np.uint32))),
                                            "val_max_abs_diff_where_idx_agrees": float(np.max(np.abs(dv))) if dv.size else 0.0}}
            print(json.dumps(row), flush=True)
            out.write(json.dumps(row) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_probe.jsonl"))
    ap.add_argument("--skip-one-gpu", action="store_true")
    ap.add_argument("--skip-sharded", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_probe.py needs a CUDA device")
    import tempfile
    info = device_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as out, tempfile.TemporaryDirectory() as tmp:
        if not args.skip_sharded:
            sharded(args.reps, info, out, tmp)
        if not args.skip_one_gpu:
            one_gpu(args.reps, info, out)


if __name__ == "__main__":
    main()
