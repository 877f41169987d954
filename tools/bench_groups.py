"""Near-duplicate groups (ffr_self_groups) against the match list of the same set (ffr_match_pairs_self).

Workloads: bench_self.make_set at 100 k x 512 and 1 M x 128 (cosine, thr 0.8: the self-mode workloads of tools/bench_pairs.py);
a heavy-edge set, 200 k x 512 in 2 000 groups of 100 noisy copies of a unit row (cosine about 0.92 between copies, thr 0.8:
about 9.9 M edges); an un-normalised Euclid set, 200 k x 256 with row norms 1..12 and 2 % noisy copies of earlier rows at
distance 0.05 |row| (thr 1.0).

Per workload the two C calls are timed alternately in one process with CUDA events after a warm-up, inputs resident, both with
the list capacity the first pairs call's count + 10 % (so both keep a raw list of the same size; the groups call keeps its edges
in the workspace, the pairs call writes them to the caller's arrays).  The ops.self_groups wrapper (default cap, so it retries
where the default overflows; the count read is a host synchronisation) is timed on the host.  A separate torch.profiler run of
the groups call sums the union-find kernels (groups_init / groups_hook / groups_finalise) per call.  The labels are verified
against the host union-find (oracle_groups.components) of the pairs call's edge list on the same input: mismatches must be 0.
Device name, power limit and max SM clock are read in the same run.

    python tools/bench_groups.py [--reps 10] [--out profiles/r09_bench_groups.jsonl] [--only self_100k_512,heavy_200k_512]
"""
import ctypes as C
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_self import device_info, make_set  # noqa: E402
from face_detection_and_recognition_b200 import _lib, ops  # noqa: E402
from oracle.oracle_groups import components  # noqa: E402

UF_KERNELS = ("groups_init_kernel", "groups_hook_kernel", "groups_finalise_kernel")


class Calls:
    """ffr_match_pairs_self and ffr_self_groups on x with buffers sized once (cap = the first pairs call's count + 10 %)."""

    def __init__(self, lib, dev, x, metric, thr):
        self.lib, self.dev, self.x, self.thr = lib, dev, x, float(thr)
        self.m = _lib.METRIC_EUCLID if metric == "euclid" else _lib.METRIC_COSINE
        self.n, self.dim = x.shape
        self.count = torch.zeros(1, dtype=torch.int64, device=dev)
        self.labels = torch.empty(self.n, dtype=torch.int32, device=dev)
        self.gcount = torch.zeros(2, dtype=torch.int64, device=dev)
        self._alloc(0)
        self.pairs()
        torch.cuda.synchronize()
        self._alloc(int(int(self.count.item()) * 1.1) + 1024)

    def _alloc(self, cap):
        self.cap = cap
        self.ws_p = torch.empty(int(self.lib.ffr_match_pairs_self_workspace_bytes(self.n, self.n, self.dim, self.m, cap)),
                                dtype=torch.uint8, device=self.dev)
        self.ws_g = torch.empty(int(self.lib.ffr_self_groups_workspace_bytes(self.n, self.dim, self.m, cap)), dtype=torch.uint8,
                                device=self.dev)
        self.out = [torch.empty(max(cap, 1), dtype=t, device=self.dev) for t in (torch.int32, torch.int32, torch.float32)]

    def _s(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def pairs(self):
        pc, pr, pv = (t.data_ptr() for t in self.out)
        _lib.check(self.lib.ffr_match_pairs_self(self.x.data_ptr(), self.n, 0, self.n, self.dim, self.m, self.thr, pc, pr, pv,
                                                 self.cap, self.count.data_ptr(), 0, self.ws_p.data_ptr(), self.ws_p.numel(),
                                                 self._s()))

    def groups(self):
        _lib.check(self.lib.ffr_self_groups(self.x.data_ptr(), self.n, self.dim, self.m, self.thr, self.labels.data_ptr(),
                                            self.gcount.data_ptr(), self.cap, self.gcount[1:].data_ptr(), 0, self.ws_g.data_ptr(),
                                            self.ws_g.numel(), self._s()))

    def stats(self):
        arr = (C.c_int64 * 8)()
        _lib.check(self.lib.ffr_filter_stats(self.ws_g.data_ptr(), arr, self._s()))
        return {"raw_pairs": int(arr[0]), "path": "tcgen05" if arr[2] == 1 else "fp32", "launches": int(arr[3])}


def timed_events(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def timed_host(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def profile_union_find(calls, reps=5):
    """ms per call of each union-find kernel and of the whole groups call's kernels, from a torch.profiler run of its own"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            calls.groups()
        torch.cuda.synchronize()
    per = {k: 0.0 for k in UF_KERNELS}
    total = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:    # kernels and memsets on the device
            continue
        t = ev.time_range.elapsed_us()
        total += t
        for k in UF_KERNELS:
            if k in ev.name:
                per[k] += t
    per = {k: round(v / reps / 1e3, 4) for k, v in per.items()}         # us -> ms per call
    uf = sum(per.values())
    return {"kernels_ms": per, "union_find_ms": round(uf, 4), "all_device_ms": round(total / reps / 1e3, 4),
            "union_find_share": round(uf / (total / reps / 1e3), 4) if total else None}


def heavy_set(n_groups, size, dim, seed):
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((n_groups, dim), dtype=np.float32)
    base /= np.linalg.norm(base, axis=1, keepdims=True)
    x = np.repeat(base, size, axis=0) + (0.3 / np.sqrt(dim)) * rng.standard_normal((n_groups * size, dim), dtype=np.float32)
    return np.ascontiguousarray(x[rng.permutation(len(x))], dtype=np.float32)


def euclid_set(n, dim, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim), dtype=np.float32)
    x *= (rng.uniform(1.0, 12.0, (n, 1)) / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)
    j = rng.choice(np.arange(1, n), n // 50, replace=False)
    k = (rng.random(len(j)) * j).astype(np.int64)
    noise = rng.standard_normal((len(j), dim), dtype=np.float32)
    noise *= (0.05 * np.linalg.norm(x[k], axis=1, keepdims=True) / np.linalg.norm(noise, axis=1, keepdims=True))
    x[j] = x[k] + noise
    return x


def workloads():
    for n, dim in [(100_000, 512), (1_000_000, 128)]:
        yield f"self_{n // 1000}k_{dim}", "cosine", 0.8, lambda n=n, dim=dim: make_set(n, dim, seed=dim)[0]
    yield "heavy_200k_512", "cosine", 0.8, lambda: heavy_set(2000, 100, 512, seed=9)
    yield "euclid_200k_256", "euclid", 1.0, lambda: euclid_set(200_000, 256, seed=10)


def main():
    reps = int(sys.argv[sys.argv.index("--reps") + 1]) if "--reps" in sys.argv else 10
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    only = sys.argv[sys.argv.index("--only") + 1].split(",") if "--only" in sys.argv else None
    dev = torch.device("cuda:0")
    lib = _lib.load()
    info = device_info()
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        open(out, "w").close()
    for name, metric, thr, make in workloads():
        if only and name not in only:
            continue
        x = torch.from_numpy(make()).to(dev)
        calls = Calls(lib, dev, x, metric, thr)
        wrap = lambda: ops.self_groups(x, thr, metric)                              # noqa: E731
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < 2.0:
            calls.pairs(); calls.groups(); wrap()
            torch.cuda.synchronize()
        ts = {"pairs_c": [], "groups_c": [], "groups_wrapper": []}
        for _ in range(reps):                                                       # alternated
            ts["pairs_c"].append(timed_events(calls.pairs))
            ts["groups_c"].append(timed_events(calls.groups))
            ts["groups_wrapper"].append(timed_host(wrap))
        med = {k: float(np.median(v)) for k, v in ts.items()}
        calls.groups()
        stats = calls.stats()                                # (this workspace's call must be the thread's last one)
        prof = profile_union_find(calls)
        calls.pairs()
        calls.groups()
        torch.cuda.synchronize()
        n_edges, g_edges = int(calls.count.item()), int(calls.gcount[1].item())
        groups = int(calls.gcount[0].item())
        want = components(calls.n, calls.out[0][:n_edges].cpu().numpy(), calls.out[1][:n_edges].cpu().numpy())
        got = calls.labels.cpu().numpy().astype(np.int64)
        res = wrap()
        line = {"workload": name, "metric": metric, "thr": thr, "shape": list(x.shape), "cap": calls.cap,
                "edges": n_edges, "groups": groups,
                "ms_median": {k: round(v, 4) for k, v in med.items()},
                "ms_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in ts.items()},
                "groups_over_pairs": round(med["groups_c"] / med["pairs_c"], 4),
                "profile_groups_call": prof, "stats": stats,
                "verified": {"label_mismatches_vs_host_union_find": int((got != want).sum()),
                             "edge_count_equal": g_edges == n_edges,
                             "group_count_equal": groups == int((want == np.arange(calls.n)).sum()),
                             "wrapper_equal": bool(np.array_equal(res.labels.cpu().numpy(), got)) and res.n_edges == n_edges}}
        line.update(info)
        print(json.dumps(line), flush=True)
        if out:
            with open(out, "a") as f:
                f.write(json.dumps(line) + "\n")
        del calls, x, res
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
