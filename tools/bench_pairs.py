"""Match lists (ops.match_pairs / ops.self_pairs) against the one-answer call on the same inputs.

Workloads: bench.py's cfg1, cfg3 and dup8 data (bench.make_refs / bench.make_cands, cosine, thr 0.5); un-normalised Euclid
rows at 10 k x 1.25 M x 512 (oracle.make_synthetic(unit_norm=False), rows scaled by 0.5-12, thr 4.0, as tools/bench_euclid.py);
self mode on bench_self.make_set at 100 k x 512 and 1 M x 128 (cosine, thr 0.8) against self_filter(mode="earlier").

Per workload the pairs call and the one-answer call (face_filter / self_filter(mode="earlier")) are timed alternately in one
process with CUDA events after a warm-up, inputs resident.  The pairs call is timed twice: the C call alone (ffr_match_pairs*
into preallocated lists: the device work, split into K1 -- everything before K2, E1/E2 included for Euclid --, K2 through the K2
event hook, and the finishing pass) and the whole ops wrapper (count read, int64 conversion, sort).  Each line reports the pairs
found and the raw pairs K2 listed, and a sample of >= 10 k candidate rows verified against oracle_pairs: pairs missing or extra
outside 1e-6 of the threshold (Euclid: relative; fp64 value) must be 0.  Device name, power limit and max SM clock are read in
the same run.

    python tools/bench_pairs.py [--reps 10] [--out profiles/r08_bench_pairs.jsonl] [--only cfg1,self_100k]
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
import bench  # noqa: E402
from bench_self import device_info, make_set  # noqa: E402
from face_detection_and_recognition_b200 import _lib, ops  # noqa: E402
from oracle import oracle, oracle_pairs  # noqa: E402

VERIFY_ROWS = 10_240


class PairsCall:
    """ffr_match_pairs* into lists sized once (cap = the first call's count + 10 %), with the K1 / K2 / finishing split."""

    def __init__(self, lib, dev, metric, ref=None, cand=None, x=None, thr=0.5):
        self.lib, self.dev, self.thr = lib, dev, float(thr)
        self.m = _lib.METRIC_EUCLID if metric == "euclid" else _lib.METRIC_COSINE
        self.ref, self.cand, self.x = ref, cand, x
        self.count = torch.zeros(1, dtype=torch.int64, device=dev)
        self.ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        self.ev[1].record(); self.ev[2].record()            # materialise the cudaEvent_t handles the library records into
        self._alloc(0)
        self.launch()
        torch.cuda.synchronize()
        self._alloc(int(int(self.count.item()) * 1.1) + 1024)

    def _alloc(self, cap):
        self.cap = cap
        if self.x is None:
            n_ref, dim = self.ref.shape
            nb = self.lib.ffr_match_pairs_workspace_bytes(n_ref, self.cand.shape[0], dim, self.m, cap)
        else:
            n, dim = self.x.shape
            nb = self.lib.ffr_match_pairs_self_workspace_bytes(n, n, dim, self.m, cap)
        self.ws = torch.empty(int(nb), dtype=torch.uint8, device=self.dev)
        self.out = [torch.empty(max(cap, 1), dtype=t, device=self.dev) for t in (torch.int32, torch.int32, torch.float32)]

    def launch(self):
        s = torch.cuda.current_stream(self.dev).cuda_stream
        pc, pr, pv = (t.data_ptr() for t in self.out)
        if self.x is None:
            n_ref, dim = self.ref.shape
            rc = self.lib.ffr_match_pairs(self.ref.data_ptr(), n_ref, self.cand.data_ptr(), self.cand.shape[0], dim, self.m,
                                          self.thr, 0, pc, pr, pv, self.cap, self.count.data_ptr(), 0, self.ws.data_ptr(),
                                          self.ws.numel(), s)
        else:
            n, dim = self.x.shape
            rc = self.lib.ffr_match_pairs_self(self.x.data_ptr(), n, 0, n, dim, self.m, self.thr, pc, pr, pv, self.cap,
                                               self.count.data_ptr(), 0, self.ws.data_ptr(), self.ws.numel(), s)
        _lib.check(rc)

    def timed(self):
        """(total, K1, K2, finishing) ms of one call"""
        e0, k0, k1, e1 = self.ev
        self.lib.ffr_debug_set_k2_events(k0.cuda_event, k1.cuda_event)
        e0.record()
        self.launch()
        e1.record()
        self.lib.ffr_debug_set_k2_events(None, None)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), e0.elapsed_time(k0), k0.elapsed_time(k1), k1.elapsed_time(e1)

    def stats(self):
        arr = (C.c_int64 * 8)()
        _lib.check(self.lib.ffr_filter_stats(self.ws.data_ptr(), arr, torch.cuda.current_stream(self.dev).cuda_stream))
        return {"raw_pairs": int(arr[0]), "path": "tcgen05" if arr[2] == 1 else "fp32", "launches": int(arr[3]),
                "pairs": int(self.count.item())}


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


def verify(res, ref, cand, thr, metric, rows, self_mode):
    """Pairs of the sampled candidate rows against oracle_pairs; disagreements are judged by their fp64 value."""
    c_all, r_all, v_all = res.cand.cpu().numpy(), res.ref.cpu().numpy(), res.val.cpu().numpy()
    sel = np.isin(c_all, rows)
    got = set(zip(c_all[sel].tolist(), r_all[sel].tolist()))
    if self_mode:
        oc, orf, ov = oracle_pairs.self_pairs(ref, thr, metric, rows=rows, block=128)
    elif metric == "cosine":
        oc, orf, ov = oracle_pairs.match_pairs(ref, cand[rows], thr, metric, block=256)
    else:
        # Euclid: the oracle's direct differences over the references within 1.01 thr (fp64 norm expansion) of some row of a chunk
        # of 64 sampled rows; every other reference is farther than that from every row of the chunk
        r64 = ref.astype(np.float64)
        rr = np.einsum("ij,ij->i", r64, r64)
        parts = []
        for s in range(0, len(rows), 64):
            c64 = cand[rows[s:s + 64]].astype(np.float64)
            d2 = np.einsum("ij,ij->i", c64, c64)[:, None] + rr[None, :] - 2.0 * (c64 @ r64.T)
            u = np.flatnonzero((d2 <= (1.01 * thr) ** 2).any(axis=0))
            c_, r_, v_ = oracle_pairs.match_pairs(ref[u], cand[rows[s:s + 64]], thr, metric)
            parts.append((c_ + s, u[r_], v_))
        oc, orf, ov = (np.concatenate([p[i] for p in parts]) for i in range(3))
    want = set(zip(rows[oc].tolist(), orf.tolist()))
    cands = ref if self_mode else cand
    bad = 0
    for c, r in got ^ want:
        a, b = cands[c].astype(np.float64), ref[r].astype(np.float64)
        v = a @ b / (np.linalg.norm(a) * np.linalg.norm(b)) if metric == "cosine" else np.linalg.norm(a - b)
        bad += int(abs(v - thr) > (1e-6 if metric == "cosine" else 1e-6 * thr))
    o = dict(zip(zip(rows[oc].tolist(), orf.tolist()), ov.tolist()))
    dv = [abs(float(v) - o[(c, r)]) / (1.0 if metric == "cosine" else max(1.0, o[(c, r)]))
          for c, r, v in zip(c_all[sel].tolist(), r_all[sel].tolist(), v_all[sel]) if (c, r) in o]
    return {"rows": int(len(rows)), "pairs": len(want), "mismatch_outside_band": bad, "disagree_in_band": len(got ^ want) - bad,
            "max_value_err": float(max(dv) if dv else 0.0)}


def workloads(dev):
    for key in ("cfg1", "cfg3", "dup8"):
        w = bench.WORKLOADS[key]
        ref = bench.make_refs(w, dev)
        cand = bench.make_cands(w, ref, 0, w["n_cand"], dev)
        yield key, "cosine", bench.THR, ref, cand, None
    ref, cand = oracle.make_synthetic(10_000, 1_250_000, 512, seed=10_000, unit_norm=False)
    yield "euclid_10k_1.25M_512", "euclid", 4.0, torch.from_numpy(ref).to(dev), torch.from_numpy(cand).to(dev), None
    for n, dim in [(100_000, 512), (1_000_000, 128)]:
        x, _ = make_set(n, dim, seed=dim)
        yield f"self_{n // 1000}k_{dim}", "cosine", 0.8, None, None, torch.from_numpy(x).to(dev)


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
    for name, metric, thr, ref, cand, x in workloads(dev):
        if only and name not in only:
            continue
        self_mode = x is not None
        pc = PairsCall(lib, dev, metric, ref=ref, cand=cand, x=x, thr=thr)
        if self_mode:
            one = lambda: ops.self_filter(x, thr, metric, mode="earlier")             # noqa: E731
            wrap = lambda: ops.self_pairs(x, thr, metric)                            # noqa: E731
        else:
            one = lambda: ops.face_filter(ref, cand, thr, metric)                    # noqa: E731
            wrap = lambda: ops.match_pairs(ref, cand, thr, metric)                   # noqa: E731
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < 2.0:
            pc.launch(); one(); wrap()
            torch.cuda.synchronize()
        ts = {"pairs_c": [], "one_answer": [], "pairs_wrapper": []}
        split = []
        for _ in range(reps):                                                        # alternated
            t = pc.timed()
            ts["pairs_c"].append(t[0]); split.append(t[1:])
            ts["one_answer"].append(timed_events(one))
            ts["pairs_wrapper"].append(timed_host(wrap))
        med = {k: float(np.median(v)) for k, v in ts.items()}
        sp = np.median(np.array(split), axis=0)
        pc.launch()
        stats = pc.stats()                                   # (this workspace's call must be the thread's last one)
        res = wrap()
        n_rows = (x if self_mode else cand).shape[0]
        rows = np.sort(np.random.default_rng(1).choice(n_rows, VERIFY_ROWS, replace=False))
        xr = x.cpu().numpy() if self_mode else ref.cpu().numpy()
        xc = None if self_mode else cand.cpu().numpy()
        line = {"workload": name, "metric": metric, "thr": thr,
                "shape": list((x if self_mode else ref).shape) + ([] if self_mode else [int(cand.shape[0])]),
                "one_answer_call": "self_filter(mode='earlier')" if self_mode else "face_filter",
                "ms_median": {k: round(v, 4) for k, v in med.items()},
                "ms_min_max": {k: [round(min(v), 4), round(max(v), 4)] for k, v in ts.items()},
                "pairs_c_split_ms": {"k1": round(float(sp[0]), 4), "k2": round(float(sp[1]), 4), "finish": round(float(sp[2]), 4)},
                "pairs_over_one_answer": round(med["pairs_c"] / med["one_answer"], 3),
                "wrapper_over_one_answer": round(med["pairs_wrapper"] / med["one_answer"], 3),
                "stats": stats, "pairs_found": int(len(res.cand)),
                "verified": verify(res, xr, xc, thr, metric, rows, self_mode)}
        line.update(info)
        print(json.dumps(line), flush=True)
        if out:
            with open(out, "a") as f:
                f.write(json.dumps(line) + "\n")
        del pc, res, ref, cand, x
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
