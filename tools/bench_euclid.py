"""Euclid gallery filtering on the tensor cores against cosine on the same data and against the exact CUDA-core kernel K2s.

Un-normalised embeddings (oracle.make_synthetic(unit_norm=False): rows scaled by 0.5-12) with planted rows on the decision
surfaces.  Each workload times the Euclid and the cosine call alternately in one process (CUDA events around each call after
warm-up, inputs resident, the candidate matrices far larger than L2 at 10 k x 1.25 M x 512 and L2-resident at 1 k x 100 k x 128,
as a user of either shape would see them); K2s (FLAG_FORCE_FP32) is timed at 1 k x 100 k x 128.  Every workload verifies a
sample of >= 10 k rows, the planted ones included, against oracle.filter_euclid.  Prints one JSON line per workload, with the
device name and power limit read in the same run.

    python tools/bench_euclid.py [--reps 10] [--out profiles/r03_bench_euclid.jsonl]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from face_detection_and_recognition_b200 import ops  # noqa: E402
from oracle import oracle  # noqa: E402


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unavailable"
    return {"device": name, "power_limit_and_max_sm_clock": out}


def planted(ref, cand, thr, n, seed):
    """n rows at distance thr * (1 +- 2e-3) of a reference, n equidistant from two references (1e-5 relative)."""
    rng = np.random.default_rng(seed)
    dim = ref.shape[1]
    k = rng.integers(0, len(ref), n)
    g = rng.standard_normal((n, dim)).astype(np.float32)
    g /= np.linalg.norm(g, axis=1, keepdims=True)
    cand[:n] = ref[k] + g * (thr * (1 + rng.uniform(-2e-3, 2e-3, (n, 1)))).astype(np.float32)
    a, b = rng.integers(0, len(ref), n), rng.integers(0, len(ref), n)
    eps = rng.uniform(-1e-5, 1e-5, (n, 1)).astype(np.float32)
    cand[n:2 * n] = 0.5 * (ref[a] + ref[b]) + eps * (ref[a] - ref[b])
    return 2 * n


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def verify(res, ref, cand, thr, rows):
    keep, idx, val = res.keep.cpu().numpy()[rows], res.best_idx.cpu().numpy()[rows], res.best_val.cpu().numpy()[rows]
    ko, io, so = oracle.filter_euclid(ref, cand[rows], thr)
    # fp64 shadow of the two smallest distances (fp32 ties are exempt from the index check, the band from the keep check)
    r = ref.astype(np.float64)
    rr = np.einsum("ij,ij->i", r, r)
    d1, d2 = np.empty(len(rows)), np.empty(len(rows))
    for s in range(0, len(rows), 2048):
        c = cand[rows[s:s + 2048]].astype(np.float64)
        d = np.sqrt(np.maximum(rr[:, None] + np.einsum("ij,ij->i", c, c)[None, :] - 2.0 * (r @ c.T), 0.0))
        d = np.partition(d, 1, axis=0)
        d1[s:s + 2048], d2[s:s + 2048] = d[0], d[1]
    tie = d2 - d1 <= 1e-6 * np.maximum(d1, 1e-30)
    near = np.abs(d1 - thr) <= 1e-6 * max(1.0, thr)
    return {"rows": int(len(rows)), "idx_mismatch_outside_ties": int(np.sum((idx != io) & ~tie)),
            "keep_mismatch_outside_band": int(np.sum((keep != ko) & ~near)),
            "max_rel_dist_err": float(np.max(np.abs(val - so) / np.maximum(1.0, so))),
            "ok": bool(np.all((idx == io) | tie) and np.all((keep == ko) | near) and np.all(np.abs(val - so) <= 1e-3 * np.maximum(1.0, so)))}


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 10
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    dev = torch.device("cuda:0")
    info = device_info()
    lines = []
    for name, n_ref, n_cand, dim, thr in [("cfg3_shard", 10_000, 1_250_000, 512, 4.0), ("cfg1", 1000, 100_000, 128, 4.0)]:
        ref, cand = oracle.make_synthetic(n_ref, n_cand, dim, seed=n_ref, unit_norm=False)
        n_pl = planted(ref, cand, thr, 2000, seed=dim)
        r, c = torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev)
        # cosine on the same rows with a threshold that keeps a similar share of them
        e = ops.face_filter(r, c, thr, metric="euclid", want_stats=True)
        co = ops.face_filter(r, c, 0.5, metric="cosine", want_stats=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < 2.0:                     # clocks up, both paths warm
            ops.face_filter(r, c, thr, metric="euclid")
            ops.face_filter(r, c, 0.5, metric="cosine")
            torch.cuda.synchronize()
        te, tc = [], []
        for _ in range(reps):                                      # alternated
            te += timed(lambda: ops.face_filter(r, c, thr, metric="euclid"), 1)
            tc += timed(lambda: ops.face_filter(r, c, 0.5, metric="cosine"), 1)
        line = {"workload": name, "n_ref": n_ref, "n_cand": n_cand, "dim": dim, "data": "unit_norm=False (0.5-12)",
                "euclid_ms_median": round(float(np.median(te)), 4), "cosine_ms_median": round(float(np.median(tc)), 4),
                "euclid_over_cosine": round(float(np.median(te) / np.median(tc)), 3),
                "euclid_ms_min_max": [round(min(te), 4), round(max(te), 4)], "cosine_ms_min_max": [round(min(tc), 4), round(max(tc), 4)],
                "euclid_stats": e.stats, "cosine_stats": co.stats}
        if name == "cfg1":
            ops.face_filter(r, c, thr, metric="euclid", flags=ops.FLAG_FORCE_FP32)
            torch.cuda.synchronize()
            tk = timed(lambda: ops.face_filter(r, c, thr, metric="euclid", flags=ops.FLAG_FORCE_FP32), max(3, reps // 3))
            line["k2s_ms_median"] = round(float(np.median(tk)), 4)
            line["k2s_over_euclid"] = round(float(np.median(tk) / np.median(te)), 1)
        rng = np.random.default_rng(1)
        rows = np.unique(np.r_[np.arange(n_pl), rng.choice(n_cand, 10_000, replace=False)])
        res = ops.face_filter(r, c, thr, metric="euclid")
        torch.cuda.synchronize()
        line["verified"] = verify(res, ref, cand, thr, rows)
        line.update(info)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del r, c
        torch.cuda.empty_cache()
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
