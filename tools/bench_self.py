"""Self mode (ops.self_filter) against the gallery call face_filter(x, x) of the same shape, cosine.

Unit-norm random rows with 1 % planted near-duplicates (a noisy copy of an earlier row at cosine thr +- 2e-3) and 1 %
bit-identical copies of earlier rows.  Per shape, FFR_SELF_OTHERS, FFR_SELF_EARLIER and the gallery call are timed alternately
in one process (CUDA events around each call after a warm-up, inputs resident).  Pairs/s counts n^2 (others, gallery) and
n(n-1)/2 (earlier).  Each self mode verifies a sample of >= 10 k rows against oracle_self.filter_self: index mismatches outside
fp32 ties (fp64 shadow) and keep mismatches outside 1e-6 of the threshold must be 0.  The per-CTA-pair work of FFR_SELF_EARLIER
(reference tiles summed over the candidate tiles a pair is dealt) is computed from the shape for the ascending and the
descending tile order: the last-wave imbalance.  Device name, power limit and max SM clock are read in the same run.

    python tools/bench_self.py [--reps 10] [--out profiles/r04_bench_self.jsonl]
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
from oracle.oracle_self import filter_self  # noqa: E402

THR = 0.8


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unavailable"
    return {"device": name, "power_limit_and_max_sm_clock": out, "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def make_set(n, dim, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim), dtype=np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    m = n // 100
    j = rng.choice(np.arange(1, n), 2 * m, replace=False)
    k = (rng.random(2 * m) * j).astype(np.int64)
    g = rng.standard_normal((m, dim)).astype(np.float32)
    g -= np.sum(g * x[k[:m]], axis=1, keepdims=True) * x[k[:m]]
    g /= np.linalg.norm(g, axis=1, keepdims=True)
    c = (THR + rng.uniform(-2e-3, 2e-3, (m, 1))).astype(np.float32)
    x[j[:m]] = c * x[k[:m]] + np.sqrt(1 - c * c) * g
    x[j[m:]] = x[k[m:]]
    return x, np.unique(j)


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def verify(res, x, mode, rows):
    keep, idx = res.keep.cpu().numpy()[rows], res.best_idx.cpu().numpy()[rows]
    ko, io, _ = filter_self(x, THR, "cosine", mode, rows=rows)
    bad_i = np.flatnonzero(idx != io)
    n_tie = 0
    if bad_i.size:                                 # fp64 shadow of the two leading scores of the disagreeing rows only
        x64 = x.astype(np.float64)
        x64 /= np.linalg.norm(x64, axis=1, keepdims=True)
        sc = x64[rows[bad_i]] @ x64.T
        col = np.arange(len(x))[None, :]
        g = rows[bad_i][:, None]
        sc[(col >= g) if mode == "earlier" else (col == g)] = -np.inf
        p = -np.partition(-sc, 1, axis=1)
        n_tie = int(np.sum(p[:, 0] - p[:, 1] <= 1e-6))
    x64 = x[rows].astype(np.float64)
    sel = np.where(io >= 0, io, 0)
    b64 = np.einsum("ij,ij->i", x64, x[sel].astype(np.float64)) / (np.linalg.norm(x64, axis=1) * np.linalg.norm(x[sel].astype(np.float64), axis=1))
    near = np.abs(b64 - THR) <= 1e-6
    return {"rows": int(len(rows)), "idx_mismatch_outside_ties": int(bad_i.size - n_tie),
            "keep_mismatch_outside_band": int(np.sum((keep != ko) & ~near))}


def earlier_imbalance(n, sms):
    """Reference tiles per CTA pair (FFR_SELF_EARLIER, row_begin 0, tiles dealt round-robin): max / mean over the pairs, for the
    shipped ascending order and for a descending one."""
    tiles = (n + 255) // 256
    work = np.array([min(n - 1, 256 * t + 255) // 256 + (1 if min(n - 1, 256 * t + 255) % 256 else 0) for t in range(tiles)])
    pairs = min(tiles, sms // 2)
    out = {}
    for name, order in (("ascending", np.arange(tiles)), ("descending", np.arange(tiles)[::-1])):
        per = np.zeros(pairs)
        for i, t in enumerate(order):
            per[i % pairs] += work[t]
        out[name] = round(float(per.max() / per.mean()), 4)
    return out


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 10
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    dev = torch.device("cuda:0")
    info = device_info()
    lines = []
    for n, dim in [(100_000, 512), (1_000_000, 128)]:
        x, planted = make_set(n, dim, seed=dim)
        xt = torch.from_numpy(x).to(dev)
        calls = {"others": lambda: ops.self_filter(xt, THR, mode="others"),
                 "earlier": lambda: ops.self_filter(xt, THR, mode="earlier"),
                 "gallery": lambda: ops.face_filter(xt, xt, THR)}
        stats = {"others": ops.self_filter(xt, THR, mode="others", want_stats=True).stats,
                 "earlier": ops.self_filter(xt, THR, mode="earlier", want_stats=True).stats,
                 "gallery": ops.face_filter(xt, xt, THR, want_stats=True).stats}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < 2.0:
            for f in calls.values():
                f()
            torch.cuda.synchronize()
        ts = {k: [] for k in calls}
        for _ in range(reps):                                      # alternated
            for k, f in calls.items():
                ts[k].append(timed(f))
        med = {k: float(np.median(v)) for k, v in ts.items()}
        line = {"n": n, "dim": dim, "metric": "cosine", "thr": THR,
                "ms_median": {k: round(v, 4) for k, v in med.items()},
                "ms_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in ts.items()},
                "pairs_per_s": {"others": n * n / (med["others"] * 1e-3), "gallery": n * n / (med["gallery"] * 1e-3),
                                "earlier": n * (n - 1) / 2 / (med["earlier"] * 1e-3)},
                "others_over_gallery": round(med["others"] / med["gallery"], 3),
                "earlier_over_others": round(med["earlier"] / med["others"], 3),
                "earlier_pair_work_max_over_mean": earlier_imbalance(n, info["sms"]),
                "stats": stats}
        rng = np.random.default_rng(1)
        rows = np.unique(np.r_[planted[:2000], rng.choice(n, 10_000, replace=False)])
        line["verified"] = {m: verify(ops.self_filter(xt, THR, mode=m), x, m, rows) for m in ("others", "earlier")}
        line.update(info)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del xt
        torch.cuda.empty_cache()
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
