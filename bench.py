#!/usr/bin/env python
"""Benchmark of the similar-face-filtering hot path: face pairs compared per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic embeddings that are already resident in HBM:
K1 (row L2-normalise + fp16 cast of the references; of the candidates too unless K2 does it in-kernel) -> K2 (tcgen05
cosine GEMM fused with the candidates' normalisation, the threshold and the running max/argmax) -> K3 (fp32 re-check
of near-tie / near-threshold rows) [-> K4 one grouped in-place NCCL allgather of {best_idx, keep} when N > 1].
Prints ONE JSON line (rank 0).  See DESIGN.md §6 for how every field is derived.

Workloads (BASELINE.json configs): the default, cfg3, is the per-GPU shard of configs[3] (10k references x 10M
candidates x 512-d, candidate-sharded over 8 GPUs -> 1.25M candidates per GPU, weak scaling: at --gpus 8 the job IS
configs[3]); cfg1 = configs[1] (1k x 100k x 128), cfg2 = configs[2] (10k x 1M x 512), cfg4 = per-GPU shard of
configs[4] (100k x 1.25M x 128); cfg3_full = configs[3] on ONE GPU (10k x 10M x 512, 20.5 GB), the strong-scaling
denominator; dup8 / near8 = cfg3's shape with a duplicate-heavy gallery (every identity enrolled 8 times).

What the line carries beyond the contract: ``verified`` (every rank checks a >= 10 k-row sample of what it timed against
the CPU oracle, and at N > 1 that rank r's slice of the gathered result is rank r's local result), ``secondary`` (short
runs of cfg1 / hbm256 / cfg4 / dup8 / near8 / n1 with their own rooflines, N = 1 only) and ``strong_scaling`` (the N-GPU job's candidates on one
GPU, measured in the same run).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # n_dup duplicated references are sized so that ~1e3 candidate rows of each workload sit on a duplicated reference
    # (SURVEY §8d: "~1e3 rows with duplicated references (exact ties)")
    "cfg1": dict(n_ref=1_000, n_cand=100_000, dim=128, adv_every=100, n_dup=10, graph=True,
                 name="configs[1]: 1k ref x 100k cand x 128-d, threshold filter"),
    "cfg2": dict(n_ref=10_000, n_cand=1_000_000, dim=512, adv_every=1000, n_dup=10,
                 name="configs[2]: 10k ref x 1M cand x 512-d, max/argmax"),
    "cfg3": dict(n_ref=10_000, n_cand=1_250_000, dim=512, adv_every=1250, n_dup=8,
                 name="configs[3] per-GPU shard: 10k ref x 1.25M cand x 512-d (10M candidates over 8 GPUs)"),
    "cfg3_full": dict(n_ref=10_000, n_cand=10_000_000, dim=512, adv_every=1250, n_dup=8,
                      name="configs[3] on ONE GPU: 10k ref x 10M cand x 512-d (strong-scaling denominator)"),
    "cfg4": dict(n_ref=100_000, n_cand=1_250_000, dim=128, adv_every=1250, n_dup=80,
                 name="configs[4] per-GPU shard: 100k ref x 1.25M cand x 128-d (10M candidates over 8 GPUs)"),
    # duplicate-heavy gallery (the realistic case for face data): 1250 identities, each enrolled 8 times -- 4 exact copies
    # (the same photo enrolled again) and 4 other photos of the same person (cos 0.9 to the first)
    "dup8": dict(n_ref=10_000, n_cand=1_250_000, dim=512, adv_every=1250, n_dup=0, dup_group=8, sib_cos=0.9,
                 name="duplicate-heavy gallery: 1250 identities x 8 enrolments (4 exact copies + 4 other photos, cos 0.9) x 1.25M cand x 512-d"),
    # the pathological variant: the 4 other enrolments are near-identical too (cos 0.99995: inside the fp16 window), so every
    # candidate has >= 5 leaders that only fp32 can tell apart -- K3's part rescan decides all of them
    "near8": dict(n_ref=10_000, n_cand=1_250_000, dim=512, adv_every=1250, n_dup=0, dup_group=8, sib_cos=0.99995,
                  name="near-identical gallery: 1250 identities x 8 enrolments (4 exact copies + 4 at cos 0.99995) x 1.25M cand x 512-d"),
    # configs[1]'s label says "HBM-bound regime", which holds for N <~ 530 references only (SURVEY §8d: add an N <= 256 sub-case that
    # truly is): 256 references, ONE reference tile per candidate tile -- K2 has to stream the fp32 candidates at HBM speed
    "hbm256": dict(n_ref=256, n_cand=2_000_000, dim=128, adv_every=2000, n_dup=2, bound="hbm",
                   name="HBM-bound sub-case of configs[1]: 256 ref x 2M cand x 128-d, threshold filter"),
    # the reference's literal mode (filter_faces_using_reference.py:186-189) at scale: ONE mean vector, Euclid keep test.
    # 0.5 FLOP/byte: the HBM-bound end of the path (exact fp32 streaming kernel K2s, no tensor cores)
    "n1": dict(n_ref=1, n_cand=10_000_000, dim=128, metric="euclid", thr=1.2, adv_every=0, n_dup=0,
               name="reference literal mode: 1 mean vector x 10M cand x 128-d, Euclid keep test (HBM-bound)"),
}
THR = 0.5
BLOCK = 62_500            # rows per synthetic block; data of a global row never depends on the GPU count
L2_BYTES = 126 * 1024 * 1024
VERIFY_ROWS = 10_240
DUMP_BYTES = 64_000_000   # --dump-outputs writes at most this much
METRIC_NAME = "face pairs compared/sec (ref x cand cosine+filter)"


def env_rank():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return int(os.environ.get("RANK", "0")), world, int(os.environ.get("LOCAL_RANK", "0"))


def host_threads(world=1):
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, n // max(1, world))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained"), hbm=d["hbm_gbs"],
                    source="MEASURED_PEAKS.json (of measured)")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm=6650.0, source="B200_PROFILING.md fallback (of fallback)")


def config_of(w, world):
    """The keys both arms (--impl b200 / reference) print: same workload, same metric."""
    return {"workload": w["name"], "n_ref": w["n_ref"], "n_cand_per_gpu": w["n_cand"], "dim": w["dim"],
            "threshold": w.get("thr", THR), "metric": w.get("metric", "cosine")}


# ------------------------------------------------------------------------------------------------ data
def make_refs(w, device):
    """Unit-norm references, seed 42 (the reference's seed, filter_faces...:24).  ``n_dup`` rows of the second half are
    exact copies of rows of the first half (SURVEY §8d: exact ties -> first-argmax rule); ``dup_group`` = G builds a
    duplicate-heavy gallery instead: identities of G consecutive rows, rows 1..G/2-1 exact copies of row 0, the rest at
    cosine ``sib_cos`` to it (0.9: other photos of the person; 0.99995: near-identical)."""
    import torch
    n_ref, dim = w["n_ref"], w["dim"]
    g = torch.Generator(device=device).manual_seed(42)
    ref = torch.nn.functional.normalize(torch.randn(n_ref, dim, device=device, generator=g))
    n_dup = min(int(w.get("n_dup", 0)), n_ref // 4)
    if n_dup:
        src = torch.randint(0, n_ref // 2, (n_dup,), device=device, generator=g)
        dst = n_ref // 2 + torch.randperm(n_ref - n_ref // 2, device=device, generator=g)[:n_dup]
        ref[dst] = ref[src]
    grp = int(w.get("dup_group", 0))
    if grp > 1:
        ids = n_ref // grp
        base = ref[:ids].clone()
        jit = torch.nn.functional.normalize(torch.randn(n_ref, dim, device=device, generator=g))
        out = base.repeat_interleave(grp, dim=0)
        k = torch.arange(ids * grp, device=device) % grp
        near = (k >= grp // 2)[:, None]
        c = float(w.get("sib_cos", 0.9))
        j = jit[:ids * grp]
        j = torch.nn.functional.normalize(j - (j * out).sum(1, keepdim=True) * out)
        out = torch.where(near, torch.nn.functional.normalize(c * out + (1 - c * c) ** 0.5 * j), out)
        ref[:ids * grp] = out
    return ref


def make_cands(w, ref, first_row, n_rows, device):
    """Unit-norm candidates for GLOBAL rows [first_row, first_row + n_rows): even rows are planted matches of a random
    reference with cos in [0.55, 0.95] (the noise is orthogonalised against the reference, so the planted cosine is exact),
    odd rows independent noise, and every ``adv_every``-th row is ADVERSARIAL: planted within +-2e-3 of the threshold
    (SURVEY §8d).  Every BLOCK rows has its own seed: a row's data never depends on the GPU count."""
    import torch
    n_ref, dim = ref.shape
    thr, adv = w.get("thr", THR), int(w.get("adv_every", 0))
    out = torch.empty(n_rows, dim, device=device)
    done = 0
    while done < n_rows:
        row = first_row + done
        blk, off = divmod(row, BLOCK)
        g = torch.Generator(device=device).manual_seed(1_000_003 + blk)
        noise = torch.nn.functional.normalize(torch.randn(BLOCK, dim, device=device, generator=g))
        k = torch.randint(0, n_ref, (BLOCK,), device=device, generator=g)
        c = torch.rand(BLOCK, device=device, generator=g) * 0.4 + 0.55
        u = torch.rand(BLOCK, device=device, generator=g) * 2 - 1
        grow = blk * BLOCK + torch.arange(BLOCK, device=device)
        if adv:
            c = torch.where(grow % adv == 0, thr + 2e-3 * u, c)
        r = ref[k]
        orth = torch.nn.functional.normalize(noise - (noise * r).sum(1, keepdim=True) * r)
        planted = torch.nn.functional.normalize(c[:, None] * r + torch.sqrt(1 - c * c)[:, None] * orth)
        block = torch.where((grow % 2 == 0)[:, None], planted, noise)
        take = min(BLOCK - off, n_rows - done)
        out[done:done + take] = block[off:off + take]
        done += take
        del noise, r, orth, planted, block
    return out


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, uuid):
        self.rows, self.proc, self.uuid = [], None, uuid

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.uuid, f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def summary(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        deadline = time.perf_counter() + 1.5                 # very short timed regions: wait for at least one sample
        while not self.rows and time.perf_counter() < deadline:
            time.sleep(0.02)
        time.sleep(0.06)
        inside = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.05] or [r for (_, r) in self.rows[-3:]]
        try:
            sm = [float(r[0]) for r in inside]
            reasons = set()
            for r in inside:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(inside[0][1]),
                    "power_w_max": max(float(r[2]) for r in inside), "samples": len(inside), "reasons": sorted(reasons)}
        except Exception as e:                                                     # pragma: no cover
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"parse error: {e}"]}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_port_rate(n_ref, dim, n_sample, seconds_target=None, threads=None, metric="cosine", thr=THR):
    """Times the oracle (the CPU restatement of the reference's arithmetic) on a bounded candidate-axis sample of the
    workload: vectorised fp32 normalise + R @ C^T + max/argmax + threshold, all host threads, NumPy and torch-CPU
    (the faster one is reported), plus the reference's literal per-pair Python loop on a tiny sub-sample."""
    import numpy as np
    import torch
    from oracle import oracle
    if threads is None:                       # torchrun exports OMP_NUM_THREADS=1: use every core this process may run on
        threads = host_threads()
    torch.set_num_threads(threads)
    rng = np.random.default_rng(42)
    ref = rng.standard_normal((n_ref, dim), dtype=np.float32)
    if metric == "euclid":
        # filter_faces_using_reference.py:186-189: vectorised (diff, row norm, <=) on all threads and the literal loop
        n_sample = int(min(n_sample, 4_000_000))
        cand = rng.standard_normal((n_sample, dim), dtype=np.float32)
        tc = torch.from_numpy(cand); tr = torch.from_numpy(ref)
        t = time.perf_counter(); k = (torch.linalg.vector_norm(tc - tr, dim=1) <= thr); t_torch = time.perf_counter() - t
        t = time.perf_counter(); k = (torch.linalg.vector_norm(tc - tr, dim=1) <= thr); t_torch = min(t_torch, time.perf_counter() - t)
        n_np = n_sample // 4
        t = time.perf_counter(); kn = oracle.filter_euclid(ref, cand[:n_np], thr)[0]; t_np = time.perf_counter() - t
        assert (k[:n_np].numpy().astype(np.uint8) == kn).mean() > 0.9999
        t = time.perf_counter(); oracle.euclid_keep_literal(cand[:100_000], ref, thr); r_lit = 100_000 / (time.perf_counter() - t)
        r_torch, r_np = n_ref * n_sample / t_torch, n_ref * n_np / t_np
        return dict(value=max(r_torch, r_np), torch_cpu=r_torch, numpy=r_np, literal_loop=r_lit, threads=threads,
                    n_sample=n_sample, seconds=t_torch)
    probe = rng.standard_normal((min(2048, n_sample), dim), dtype=np.float32)
    t = time.perf_counter(); oracle.filter_cosine_torch(ref, probe, THR); t_probe = time.perf_counter() - t
    t = time.perf_counter(); oracle.filter_cosine_torch(ref, probe, THR); t_probe = min(t_probe, time.perf_counter() - t)
    if seconds_target is not None:
        n_sample = int(max(2048, min(n_sample, probe.shape[0] * seconds_target / max(t_probe, 1e-6))))
    cand = rng.standard_normal((n_sample, dim), dtype=np.float32)
    t = time.perf_counter(); out_t = oracle.filter_cosine_torch(ref, cand, THR); t_torch = time.perf_counter() - t
    n_np = max(1024, n_sample // 8)
    t = time.perf_counter(); out_n = oracle.filter_cosine(ref, cand[:n_np], THR); t_np = time.perf_counter() - t
    assert (out_t[1][:n_np] == out_n[1]).mean() > 0.999
    r_torch, r_np = n_ref * n_sample / t_torch, n_ref * n_np / t_np
    # literal reference expression (extract_and_label_faces_from_dataset.py:106), Python double loop, 1 thread
    nl_r, nl_c = min(n_ref, 50), 200
    t = time.perf_counter()
    for j in range(nl_c):
        for i in range(nl_r):
            oracle.cosine_dist_literal(ref[i], cand[j])
    r_lit = nl_r * nl_c / (time.perf_counter() - t)
    return dict(value=max(r_torch, r_np), torch_cpu=r_torch, numpy=r_np, literal_loop=r_lit, threads=threads,
                n_sample=n_sample, seconds=t_torch)


def run_reference(args, rank, world, emit):
    """--impl reference: the reference's CPU arithmetic for this path (oracle port; the reference is pure Python/NumPy and
    its TensorFlow front end cannot run here, so there is no oracle/_ref) on the host cores, same config and metric."""
    if rank != 0:
        return
    import torch
    w = WORKLOADS[args.workload]
    n_ref, dim = w["n_ref"], w["dim"]
    metric, thr = w.get("metric", "cosine"), w.get("thr", THR)
    import numpy as np
    from oracle import oracle
    probe = cpu_port_rate(n_ref, dim, 4096 if metric == "cosine" else 400_000, metric=metric, thr=thr)
    n_sample = int(max(2048, min(w["n_cand"], 1.5 * probe["value"] / n_ref)))       # ~1.5 s per step
    rng = np.random.default_rng(42)
    ref = rng.standard_normal((n_ref, dim), dtype=np.float32)
    cand = rng.standard_normal((n_sample, dim), dtype=np.float32)
    if metric == "euclid":
        tr, tc = torch.from_numpy(ref), torch.from_numpy(cand)
        use_torch = probe["torch_cpu"] >= probe["numpy"]
        fn = (lambda r, c, t: (torch.linalg.vector_norm(tc - tr, dim=1) <= t)) if use_torch else oracle.filter_euclid
        how = ("torch-CPU" if use_torch else "NumPy") + " (diff, row norm, <=)"
    else:
        use_torch = probe["torch_cpu"] >= probe["numpy"]
        fn = oracle.filter_cosine_torch if use_torch else oracle.filter_cosine
        how = ("torch-CPU" if use_torch else "NumPy") + " sgemm + max/argmax + threshold"
    for _ in range(args.warmup):
        fn(ref, cand, thr)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn(ref, cand, thr)
    dt = time.perf_counter() - t0
    value = n_ref * n_sample * args.steps / dt
    cores = torch.get_num_threads()
    sample = (f"{n_sample} of {w['n_cand']} candidates per step x all {n_ref} references x {dim}-d, vectorised fp32 "
              f"restatement ({how}), {cores} threads; the reference's literal per-row Python loop = "
              f"{probe['literal_loop']:.3g} pairs/s on 1 thread")
    emit({
        "impl": "reference", "metric": METRIC_NAME, "value": value,
        "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_of(w, world),
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


# ------------------------------------------------------------------------------------------------ verification
def verify_sample(w, ref, cand, keep, idx, val, seed, threads):
    """What was timed is what is checked: a >= 10 k-row sample of this rank's shard (every adversarial row it holds, up to
    a quarter of the sample, plus random rows) against the CPU oracle, outside the timed region.  Bars as in
    tests/test_gpu_parity.py: similarity within 1e-3; index equal unless the two references' fp64 scores differ by
    < 1e-6 (fp32 summation noise); keep equal unless the fp64 best lies within 1e-6 of the threshold.  ``band_1e-3`` counts
    the sampled rows inside north_star's tolerance band (they agree too unless counted as mismatches)."""
    import numpy as np
    import torch
    from oracle import oracle
    try:
        from threadpoolctl import threadpool_limits
    except ImportError:                                                            # pragma: no cover
        from contextlib import nullcontext as threadpool_limits
    metric, thr = w.get("metric", "cosine"), w.get("thr", THR)
    n_cand = cand.shape[0]
    rng = np.random.default_rng(seed)
    n = min(VERIFY_ROWS, n_cand)
    adv = int(w.get("adv_every", 0))
    hard = np.arange(0, n_cand, adv)[: n // 4] if adv else np.zeros(0, dtype=np.int64)
    sel = np.unique(np.concatenate([hard, rng.choice(n_cand, n, replace=False)]))
    sel_t = torch.from_numpy(sel).to(cand.device)
    c = cand[sel_t].cpu().numpy()
    r = ref.cpu().numpy()
    k_g, i_g, v_g = keep[sel_t].cpu().numpy(), idx[sel_t].cpu().numpy(), val[sel_t].cpu().numpy()
    t0 = time.perf_counter()
    with threadpool_limits(limits=threads):
        if metric == "euclid":
            k_o, i_o, v_o = oracle.filter_euclid(r, c, thr)
        else:
            k_o, i_o, v_o = oracle.filter_cosine(r, c, thr, block=1024 if r.shape[0] > 20_000 else 8192)
    secs = time.perf_counter() - t0
    r64, c64 = r.astype(np.float64), c.astype(np.float64)

    def score64(rows, refs):
        a, b = c64[rows], r64[refs]
        if metric == "euclid":
            return np.linalg.norm(a - b, axis=1)
        return np.einsum("ij,ij->i", a, b) / (np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1))

    bad_i = np.flatnonzero(i_g != i_o)
    tie = np.abs(score64(bad_i, i_g[bad_i]) - score64(bad_i, i_o[bad_i])) < 1e-6 if bad_i.size else np.zeros(0, bool)
    best64 = score64(np.arange(len(sel)), i_o)
    eps = 1e-6 if metric == "cosine" else 1e-5 * max(1.0, thr)
    bad_k = np.flatnonzero(k_g != k_o)
    near = np.abs(best64[bad_k] - thr) < eps if bad_k.size else np.zeros(0, bool)
    val_err = float(np.max(np.abs(v_g - v_o))) if len(sel) else 0.0
    tol = 1e-3 if metric == "cosine" else 1e-5 * max(1.0, thr)
    mism = int((~tie).sum() + (~near).sum() + (1 if val_err > tol else 0))
    return {"rows": int(len(sel)), "adversarial_rows": int(len(hard)), "mismatch_outside_band": mism,
            "idx_mismatch": int((~tie).sum()), "idx_fp32_tie_rows": int(tie.sum()), "keep_mismatch": int((~near).sum()),
            "keep_within_1e-6_of_thr": int(near.sum()), "val_max_abs_err": val_err,
            "band_1e-3_rows": int((np.abs(best64 - thr) <= 1e-3).sum()), "oracle": "oracle.filter_" + metric + " (NumPy fp32) + fp64 shadow",
            "oracle_seconds": round(secs, 2), "ok": mism == 0}


def dump_outputs(out_dir, outputs, max_bytes=DUMP_BYTES, seed=0):
    """--dump-outputs: each array of ``outputs`` -> ``out_dir/<name>.npy``, float64 for indices (float32 is exact only up
    to 2**24), float32 otherwise, so that two builds can be compared output for output.  When the arrays would exceed
    ``max_bytes`` in all, each is cut to the same seeded sample of rows and ``<name>_rows.npy`` (float64) says which."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {}
    for name, t in outputs.items():
        a = t.cpu().numpy()
        host[name] = a.astype(np.float64 if a.dtype.kind in "iu" and a.dtype.itemsize > 2 else np.float32)
    budget = max_bytes - 256 * 2 * len(host)                   # room for the .npy headers
    sample = sum(a.nbytes for a in host.values()) > budget
    frac = budget / sum(a.nbytes + 8 * len(a) for a in host.values())
    for name, a in host.items():
        if sample:
            rows = np.sort(np.random.default_rng(seed).choice(len(a), int(len(a) * frac), replace=False))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def result_hash(keep, idx):
    import torch
    wgt = (torch.arange(idx.numel(), device=idx.device, dtype=torch.int64) % 1_000_003) + 1
    return (idx.to(torch.int64) * wgt).sum() + 7 * (keep.to(torch.int64) * wgt).sum()


# ------------------------------------------------------------------------------------------------ one workload on the GPU(s)
def run_workload(key, steps, warmup, ctx, first_row=None, n_cand=None, do_verify=True, use_gather=True, sampler=None,
                 keep_outputs=False):
    """Data generation, warm-up, the timed region (CUDA events on the launch stream, barrier + synchronize on both sides),
    per-launch K2 events, statistics, verification.  Returns a dict of raw measurements (this rank's; reduced by the
    caller); with ``keep_outputs``, ``outputs`` holds copies of the arrays the last timed step handed back."""
    import torch
    import torch.distributed as dist
    ops, lib, dev = ctx["ops"], ctx["lib"], ctx["dev"]
    rank, world = ctx["rank"], ctx["world"]
    w = WORKLOADS[key]
    n_ref, dim = w["n_ref"], w["dim"]
    n_cand = w["n_cand"] if n_cand is None else n_cand
    metric, thr = w.get("metric", "cosine"), w.get("thr", THR)
    gathering = use_gather and world > 1
    first_row = rank * n_cand if first_row is None else first_row

    ref = make_refs(w, dev)
    in_bytes = (n_cand + n_ref) * dim * 4
    n_buf = 1 if in_bytes > 2 * L2_BYTES else int(-(-3 * L2_BYTES // in_bytes))   # rotate copies when L2 could hold the input
    cands = [make_cands(w, ref, first_row + b * world * n_cand, n_cand, dev) for b in range(n_buf)]
    val = torch.empty(n_cand, dtype=torch.float32, device=dev)
    gather = ctx.get("gather") if gathering else None
    if gather is not None:
        keep_all, idx_all, keep, idx = gather.buffers(n_cand, dev)
    else:
        keep = torch.empty(n_cand, dtype=torch.uint8, device=dev)
        idx = torch.empty(n_cand, dtype=torch.int32, device=dev)
        keep_all, idx_all = keep, idx

    graphs = None
    if w.get("graph") and not gathering and os.environ.get("FFR_BENCH_GRAPH", "1") != "0":
        # launch-bound workload (~25 us of GPU work per step): the whole K1 -> K2 -> K3 sequence of one step is captured
        # once per rotating input and replayed -- same kernels, same arguments, no host work between the launches
        graphs = [ops.GraphedFilter.capture(ref, c, thr, metric=metric, out=(keep, idx, val)) for c in cands]

    def step(i):
        if graphs is not None:
            graphs[i % n_buf].replay()
            return
        ops.face_filter(ref, cands[i % n_buf], thr, metric=metric, out=(keep, idx, val))
        if gather is not None:
            gather.all_gather_inplace(keep_all, idx_all)

    def barrier():
        if world > 1 and use_gather:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(warmup):
        step(i)
    tensor_path = metric == "cosine" and n_ref > 8
    k2_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in k2_ev:
        a.record(); b.record()                                      # materialise the cudaEvent_t handles
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = ops.launch_count()
    t_host0 = time.perf_counter()
    ev0.record()
    for i in range(steps):
        if graphs is None:
            lib.ffr_debug_set_k2_events(k2_ev[i][0].cuda_event, k2_ev[i][1].cuda_event)
        step(i)
    ev1.record()
    lib.ffr_debug_set_k2_events(None, None)
    barrier()
    t_host1 = time.perf_counter()
    # copied before the eager K2 timing and the stats call below write the same buffers again
    outputs = {"keep": keep_all.clone(), "best_idx": idx_all.clone(), "best_val": val.clone()} if keep_outputs else None
    launches = ops.launch_count() - l0
    if graphs is not None:
        launches = steps * graphs[0].launches
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.summary(t_host0, t_host1) if sampler else None
    if graphs is not None:
        # per-launch K2 time of a graphed step: the same launch sequence, eagerly, with the library's event pair around K2
        for i in range(steps):
            lib.ffr_debug_set_k2_events(k2_ev[i][0].cuda_event, k2_ev[i][1].cuda_event)
            ops.face_filter(ref, cands[i % n_buf], thr, metric=metric, out=(keep, idx, val))
        lib.ffr_debug_set_k2_events(None, None)
        torch.cuda.synchronize()
    k2_ms = statistics.mean(a.elapsed_time(b) for a, b in k2_ev) if tensor_path else ms_total / steps

    # the result that is verified is the one the LAST timed step left behind
    last = (steps - 1) % n_buf
    res = {"key": key, "w": w, "n_cand": n_cand, "ms_total": ms_total, "k2_ms": k2_ms, "launches": launches, "steps": steps,
           "tensor_path": tensor_path, "n_buf": n_buf, "in_bytes": in_bytes, "clocks": clocks, "graph": graphs is not None,
           "keep_frac": float(keep.float().mean()), "outputs": outputs}
    if gather is not None:
        hashes = torch.stack([result_hash(keep_all[r * n_cand:(r + 1) * n_cand], idx_all[r * n_cand:(r + 1) * n_cand])
                              for r in range(world)])
        mine = torch.empty(world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(mine, hashes[rank].reshape(1))
        res["gather_ok"] = bool(torch.equal(mine, hashes))
    if do_verify:
        res["verified"] = verify_sample(w, ref, cands[last], keep, idx, val, seed=1234 + rank, threads=ctx["threads"])
        if gather is not None:
            res["verified"]["gather_ok"] = res["gather_ok"]
            res["verified"]["ok"] = res["verified"]["ok"] and res["gather_ok"]
    res["stats"] = ops.face_filter(ref, cands[last], thr, metric=metric, out=(keep, idx, val), want_stats=True).stats
    res["_data"] = (ref, cands, keep, idx, val)
    return res


def roofline_of(r, pk, traffic):
    w, n_cand = r["w"], r["n_cand"]
    n_ref, dim = w["n_ref"], w["dim"]
    ms_step = r["ms_total"] / r["steps"]
    hbm_bytes = 4.0 * dim * (n_ref + n_cand) + 9.0 * n_cand
    if not r["tensor_path"]:               # one HBM-bound kernel: the roofline is the measured copy bandwidth
        gbs = hbm_bytes / (ms_step * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "filter_fp32_kernel (K2s)", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
                "frac": gbs / pk["hbm"], "peak_source": pk["source"], "bytes_per_launch": hbm_bytes, "traffic": traffic}
    # FLOPs of the contraction K2 actually ran: bit-identical reference rows are folded before the scan (ffr_dedup.cu)
    n_scanned = int(r["stats"].get("refs_scanned") or n_ref)
    flops = 2.0 * n_scanned * n_cand * dim
    if w.get("bound") == "hbm":            # tensor-core kernel, but the candidates' fp32 rows are what takes the time
        gbs = hbm_bytes / (r["k2_ms"] * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "filter_mma_kernel (K2, stage32)", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s",
                "frac": gbs / pk["hbm"], "frac_whole_step": hbm_bytes / (ms_step * 1e-3) / 1e9 / pk["hbm"], "peak_source": pk["source"],
                "k2_ms": r["k2_ms"], "k2_share_of_step": r["k2_ms"] / ms_step, "bytes_per_launch": hbm_bytes,
                "tflops": flops / (r["k2_ms"] * 1e-3) / 1e12, "traffic": traffic}
    ach = flops / (r["k2_ms"] * 1e-3) / 1e12
    ach_step = flops / (ms_step * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": "filter_mma_kernel (K2)", "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s",
            "frac": ach / pk["tflops"],
            "frac_of_sustained": ach / pk["tflops_sustained"] if pk["tflops_sustained"] else None,
            "frac_whole_step": ach_step / pk["tflops"],
            "peak_source": pk["source"], "k2_ms": r["k2_ms"], "k2_share_of_step": r["k2_ms"] / ms_step,
            "flops_per_launch": flops, "refs_scanned": n_scanned, "traffic": traffic,
            "step_hbm": {"algorithmic_bytes": hbm_bytes, "gbs_over_step": hbm_bytes / (ms_step * 1e-3) / 1e9,
                         "frac_of_hbm_peak": hbm_bytes / (ms_step * 1e-3) / 1e9 / pk["hbm"]}}


def load_traffic(key):
    tp = os.path.join(ROOT, "profiles", "k2_traffic.json")
    if os.path.exists(tp):
        return json.load(open(tp)).get(key)
    return None


def details_of(r, world):
    return {"arithmetic": ("tcgen05 kind::f16: fp16 operands, fp32 accumulate in TMEM; fp32 re-check of near-tie / "
                           "near-threshold rows") if r["tensor_path"] else "fp32 CUDA cores (exact streaming kernel)",
            "sharding": "candidate axis; references replicated; one grouped in-place NCCL allgather of 5 B/candidate"
            if world > 1 else "single GPU",
            "l2": (f"inputs {r['in_bytes'] / 1e6:.0f} MB per GPU > L2 (126 MB)" if r["n_buf"] == 1 else
                   f"rotating {r['n_buf']} input copies ({r['n_buf'] * r['in_bytes'] / 1e6:.0f} MB > L2 126 MB)"),
            "launch": "one CUDA graph per step (K1 -> K2 -> K3 captured once per rotating input)" if r["graph"] else "eager launches",
            "data": "half planted matches (cos 0.55-0.95), adversarial rows within +-2e-3 of the threshold every "
                    f"{r['w'].get('adv_every', 0)} rows, " +
                    (f"duplicate-heavy gallery: identities of {r['w']['dup_group']} consecutive rows, {r['w']['dup_group'] // 2} exact copies + "
                     f"{r['w']['dup_group'] - r['w']['dup_group'] // 2} enrolments at cosine {r['w'].get('sib_cos', 0.9)} (every matched row has several leaders)"
                     if r['w'].get('dup_group', 0) > 1 else
                     f"{r['w'].get('n_dup', 0)} exactly duplicated references (~1e3 candidate rows with an exact tie)"),
            "keep_fraction": r["keep_frac"], "recheck": r["stats"]}


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the short cfg1 / hbm256 / cfg4 / dup8 / near8 / n1 runs of the default line")
    ap.add_argument("--no-strong", action="store_true", help="skip the one-GPU run of the whole N-GPU job")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (keep, best_idx, best_val) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    rank, world, local_rank = env_rank()
    # the contract is ONE JSON line on stdout: anything libraries print while we run (NCCL's version banner, warnings)
    # is sent to stderr by pointing fd 1 at fd 2 until the result line is written
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    if args.impl == "reference":
        return run_reference(args, rank, world, emit)

    import torch
    import torch.distributed as dist
    from face_detection_and_recognition_b200 import _lib, ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the filter has no CPU path (use --impl reference for the CPU arm)")
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    w = WORKLOADS[args.workload]
    n_ref, n_cand, dim = w["n_ref"], w["n_cand"], w["dim"]
    metric, thr = w.get("metric", "cosine"), w.get("thr", THR)
    pk = peaks()
    ctx = dict(ops=ops, lib=lib, dev=dev, rank=rank, world=world, threads=host_threads(world),
               gather=ops.ResultGather(rank, world, local_rank) if world > 1 else None)

    sampler = ClockSampler("GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)) if rank == 0 else None
    if sampler:
        sampler.start()
    r = run_workload(args.workload, args.steps, args.warmup, ctx, do_verify=not args.no_verify, sampler=sampler,
                     keep_outputs=bool(args.dump_outputs) and rank == 0)
    if sampler:
        sampler.stop()
    ref, cands, keep, idx, val = r.pop("_data")
    outputs = r.pop("outputs")
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
        del outputs
    ms_total, k2_ms, launches = r["ms_total"], r["k2_ms"], r["launches"]

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        ref_h = ref.cpu().pin_memory()
        cand_h = torch.empty((n_cand, dim), dtype=torch.float32).pin_memory()
        cand_h.copy_(cands[0])
        out_h = (torch.empty(n_cand, dtype=torch.uint8).pin_memory(), torch.empty(n_cand, dtype=torch.int32).pin_memory(),
                 torch.empty(n_cand, dtype=torch.float32).pin_memory())
        dev_res = ops.face_filter(ref, cands[0], thr, metric=metric)
        hf = ops.HostFilter(device=local_rank, max_ref=n_ref, chunk_cand=min(n_cand, 1 << 17), max_dim=dim)
        hf(ref_h, cand_h, thr, metric=metric, out=out_h)
        e2e_steps = max(2, min(args.steps, 10))
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            hf(ref_h, cand_h, thr, metric=metric, out=out_h)
        t_e2e = time.perf_counter() - t0
        same = bool(torch.equal(out_h[0], dev_res.keep.cpu()) and torch.equal(out_h[1], dev_res.best_idx.cpu()))
        hf.close()
        # the ceiling of that pipeline on this box: the same pinned bytes, plain H2D copies, nothing else, every rank at
        # the same time (at N > 1 the ranks share the host's PCIe / memory system)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            cands[0].copy_(cand_h, non_blocking=True)
        torch.cuda.synchronize()
        t_h2d = (time.perf_counter() - t0) / 3
        e2e = dict(seconds=t_e2e / e2e_steps, same_as_device_path=same, steps=e2e_steps, h2d_seconds=t_h2d)
        del cand_h, out_h

    # ---- strong scaling: the whole N-GPU job's candidates on ONE GPU, in this same run (rank 0; N = 1: configs[3] itself)
    strong = None
    if not args.no_strong and args.workload == "cfg3":
        if rank == 0:
            n_total = n_cand * max(world, 1) if world > 1 else WORKLOADS["cfg3_full"]["n_cand"]
            del cands
            torch.cuda.empty_cache()
            ctx1 = dict(ctx, world=1, rank=0, gather=None)
            rs = run_workload("cfg3", 3, 1, ctx1, first_row=0, n_cand=n_total, do_verify=not args.no_verify, use_gather=False)
            rs.pop("_data")
            torch.cuda.empty_cache()
            strong = {"n_cand_total": n_total, "t1_ms": rs["ms_total"] / rs["steps"], "steps": rs["steps"],
                      "k2_ms": rs["k2_ms"], "verified": rs.get("verified"),
                      "what": f"all {n_total} candidates of the {max(world, 1) if world > 1 else 8}-GPU job on one GPU (rank 0), same data"}
        if world > 1:
            dist.barrier()

    # ---- secondary workloads (N = 1 only): short runs with their own rooflines, so the driver's record carries every config
    secondary = None
    if world == 1 and not args.no_secondary and args.workload == "cfg3":
        try:
            del cands
        except NameError:
            pass
        secondary = {}
        for key in ("cfg1", "hbm256", "cfg4", "dup8", "near8", "n1"):
            torch.cuda.empty_cache()
            # (cfg1 is ~25 us per step: enough steps that the GPU leaves its idle clocks; the others are ms-sized)
            sec_steps, sec_warm = (64, 64) if key == "cfg1" else (5, 3)
            rs = run_workload(key, sec_steps, sec_warm, ctx, do_verify=not args.no_verify, use_gather=False)
            rs.pop("_data")
            ws = rs["w"]
            ms = rs["ms_total"] / rs["steps"]
            secondary[key] = {"config": config_of(ws, 1), "value": ws["n_ref"] * ws["n_cand"] / (ms * 1e-3), "unit": "pairs/s",
                              "ms_per_step": ms, "steps": rs["steps"], "warmup": sec_warm, "gpu_launches": rs["launches"],
                              "roofline": roofline_of(rs, pk, load_traffic(key)), "verified": rs.get("verified"),
                              "details": details_of(rs, 1)}

    # ---- reduce over ranks: slowest rank's time, total launches, everybody's verification
    if world > 1:
        t = torch.tensor([ms_total, k2_ms, e2e["seconds"] if e2e else 0.0, e2e["h2d_seconds"] if e2e else 0.0],
                         device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, k2_ms = float(t[0]), float(t[1])
        if e2e:
            e2e["seconds"], e2e["h2d_seconds"] = float(t[2]), float(t[3])
        v = r.get("verified") or {}
        lt = torch.tensor([launches, v.get("rows", 0), v.get("mismatch_outside_band", 0), v.get("idx_fp32_tie_rows", 0),
                           v.get("band_1e-3_rows", 0), 0 if v.get("gather_ok", True) else 1,
                           0 if (not e2e or e2e["same_as_device_path"]) else 1], device=dev, dtype=torch.int64)
        dist.all_reduce(lt)
        launches = int(lt[0])
        if v:
            v.update({"rows": int(lt[1]), "mismatch_outside_band": int(lt[2]), "idx_fp32_tie_rows": int(lt[3]),
                      "band_1e-3_rows": int(lt[4]), "gather_ok": int(lt[5]) == 0, "ranks": world})
            v["ok"] = v["mismatch_outside_band"] == 0 and v["gather_ok"]
        if e2e:
            e2e["same_as_device_path"] = int(lt[6]) == 0

    if rank == 0:
        r["ms_total"], r["k2_ms"], r["launches"] = ms_total, k2_ms, launches
        ms_step = ms_total / args.steps
        pairs_job = n_ref * n_cand * world
        out = {
            "metric": METRIC_NAME,
            "value": pairs_job / (ms_step * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16->f32" if r["tensor_path"] else "f32", "data": "synthetic",
            "config": config_of(w, world), "details": details_of(r, world),
            "roofline": roofline_of(r, pk, load_traffic(args.workload)),
            "gpu_launches": launches, "clocks": r["clocks"],
        }
        if r.get("verified") is not None:
            out["verified"] = r["verified"]
        if e2e:
            h2d_bytes = int((n_cand + n_ref) * dim * 4)
            out["e2e"] = {"value": pairs_job / e2e["seconds"], "unit": "pairs/s",
                          "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": int(9 * n_cand),
                          "ms_per_step": e2e["seconds"] * 1e3, "steps": e2e["steps"],
                          "api": "ffr_ctx_filter_host (pinned host buffers, chunked H2D overlapped with compute)",
                          "same_result_as_device_path": e2e["same_as_device_path"],
                          "h2d_gbs_per_gpu": h2d_bytes / e2e["seconds"] / 1e9,
                          "h2d_ceiling_gbs_per_gpu": n_cand * dim * 4 / e2e["h2d_seconds"] / 1e9,
                          "frac_of_h2d_ceiling": (h2d_bytes / e2e["seconds"]) / (n_cand * dim * 4 / e2e["h2d_seconds"]),
                          "h2d_ceiling": "plain cudaMemcpyAsync of the same pinned candidate buffer, all ranks at once, max over ranks"}
        if strong is not None:
            strong["tN_ms"] = ms_step if world > 1 else None
            strong["speedup"] = strong["t1_ms"] / ms_step if world > 1 else None
            out["strong_scaling"] = strong
            out["strong_scaling_t1_ms"] = strong["t1_ms"]
        if secondary is not None:
            out["secondary"] = secondary
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_port_rate(n_ref, dim, n_cand, seconds_target=10.0, metric=metric, thr=thr)
            out["cpu_baseline"] = {
                "value": cb["value"], "unit": "pairs/s", "cores": cb["threads"], "kind": "port",
                "sample": (f"{cb['n_sample']} of {n_cand} candidates x all {n_ref} references x {dim}-d "
                           f"({cb['seconds']:.1f} s): vectorised fp32 oracle, torch-CPU {cb['torch_cpu']:.3g} / NumPy "
                           f"{cb['numpy']:.3g} pairs/s on {cb['threads']} threads; the reference's literal per-pair Python "
                           f"loop: {cb['literal_loop']:.3g} pairs/s on 1 thread")}
        emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
