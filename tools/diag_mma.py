#!/usr/bin/env python
"""GPU diagnostic: raw tcgen05 score tiles against a torch fp32 matmul of the same fp16 rows, then quick timings.
Run on the GPU box:  [FFR_CTA_GROUP=2] python tools/diag_mma.py [--raw] [--perf] [--stream]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from face_detection_and_recognition_b200 import _lib, ops  # noqa: E402


def setenv(k, v):
    os.environ[k] = str(v)
    _lib.load().ffr_debug_reload_env()          # the library reads its FFR_* knobs once per process


def delenv(k):
    os.environ.pop(k, None)
    _lib.load().ffr_debug_reload_env()


def raw(n_ref, n_cand, dim):
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(1)
    ref = torch.randn(n_ref, dim, device="cuda", generator=g)
    cand = torch.randn(n_cand, dim, device="cuda", generator=g)
    r16 = ops.l2norm_rows(ref, want_f16=True, want_f32=False)["f16"]
    c16 = ops.l2norm_rows(cand, want_f16=True, want_f32=False)["f16"]
    ld = r16.shape[1]
    scores = torch.full((n_cand, n_ref), float("nan"), device="cuda")
    keep = torch.empty(n_cand, dtype=torch.uint8, device="cuda")
    idx = torch.empty(n_cand, dtype=torch.int32, device="cuda")
    val = torch.empty(n_cand, dtype=torch.float32, device="cuda")
    ws = torch.zeros(4096 + 64 * n_cand, dtype=torch.uint8, device="cuda")
    rc = lib.ffr_debug_mma_scores(r16.data_ptr(), n_ref, c16.data_ptr(), n_cand, ld, 0.5, keep.data_ptr(),
                                  idx.data_ptr(), val.data_ptr(), scores.data_ptr(), ws.data_ptr(), ws.numel(),
                                  torch.cuda.current_stream().cuda_stream)
    if rc != 0:
        print("  rc", rc, lib.ffr_last_error().decode())
        return False
    torch.cuda.synchronize()
    want = c16.float() @ r16.float().T
    err = (scores - want).abs()
    nan = torch.isnan(scores).sum().item()
    e = torch.nan_to_num(err, nan=9.0)
    print(f"  [{n_ref}x{n_cand}x{dim}] nan={nan} max_err={e.max().item():.3e} mean_err={e.mean().item():.3e} "
          f"val_err={(val - want.max(1).values).abs().max().item():.3e} "
          f"idx_match={(idx.long() == want.argmax(1)).float().mean().item():.4f}", flush=True)
    if e.max().item() > 1e-4:
        bad = (e > 1e-4)
        rows = bad.any(1).nonzero().flatten()
        cols = bad.any(0).nonzero().flatten()
        print("   bad rows: count", rows.numel(), "first", rows[:8].tolist(), "last", rows[-4:].tolist(),
              " bad cols: count", cols.numel(), "first", cols[:8].tolist(), "last", cols[-4:].tolist())
        print("   got[0,:6]", scores[0, :6].tolist(), " want[0,:6]", want[0, :6].tolist())
        r0 = rows[0].item()
        print(f"   got[{r0},:6]", scores[r0, :6].tolist(), f" want[{r0},:6]", want[r0, :6].tolist())
        return False
    return True


def perf(n_ref, n_cand, dim, flags=0, iters=5, metric="cosine", thr=0.5):
    g = torch.Generator(device="cuda").manual_seed(2)
    ref = torch.nn.functional.normalize(torch.randn(n_ref, dim, device="cuda", generator=g))
    cand = torch.nn.functional.normalize(torch.randn(n_cand, dim, device="cuda", generator=g))
    cand[::2] = torch.nn.functional.normalize(ref[torch.randint(0, n_ref, (cand[::2].shape[0],), device="cuda")] * 0.8
                                              + cand[::2] * 0.6)
    res = ops.face_filter(ref, cand, thr, flags=flags, want_stats=True, metric=metric)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    ev[0].record()
    for i in range(iters):
        ops.face_filter(ref, cand, thr, flags=flags, out=(res.keep, res.best_idx, res.best_val), metric=metric)
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = min(ev[i].elapsed_time(ev[i + 1]) for i in range(iters))
    pairs = n_ref * n_cand
    tag = f"cg={os.environ.get('FFR_CTA_GROUP', '1')}"
    print(f"  perf [{n_ref}x{n_cand}x{dim}] {metric} flags={flags} {tag}: {ms:.3f} ms  {pairs / ms / 1e6:.1f} Gpairs/s  "
          f"{2 * pairs * dim / ms / 1e9:.1f} TFLOP/s  {n_cand * dim * 4 / ms / 1e6:.0f} GB/s(cand)  stats={res.stats} "
          f"keep={res.keep.float().mean().item():.3f}", flush=True)


def prof(n_ref, n_cand, dim, easy=False, bench_data=False, flags=None):
    """Where does K2's pipeline wait?  Stall cycles of the TMA thread, the MMA thread and one epilogue warp.
    easy=True: every candidate is a near copy of reference 0, so the running best is final after the first chunk and the
    update path never runs again -- the epilogue's floor."""
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(2)
    ref = torch.nn.functional.normalize(torch.randn(n_ref, dim, device="cuda", generator=g))
    cand = torch.nn.functional.normalize(torch.randn(n_cand, dim, device="cuda", generator=g))
    if easy:
        cand = torch.nn.functional.normalize(ref[0][None, :] + 0.05 * cand)
    if bench_data:                       # exactly bench.py's synthetic embeddings (half planted matches)
        import bench
        w = dict(n_ref=n_ref, dim=dim, adv_every=1250, n_dup=min(1000, n_ref // 10))
        ref = bench.make_refs(w, torch.device("cuda"))
        cand = bench.make_cands(w, ref, 0, n_cand, torch.device("cuda"))
    flags = ops.FLAG_NO_RECHECK if flags is None else flags
    ops.face_filter(ref, cand, 0.5, flags=flags)
    buf = torch.zeros(160 * 32, dtype=torch.int64, device="cuda")
    lib.ffr_debug_set_prof(buf.data_ptr())
    ops.face_filter(ref, cand, 0.5, flags=flags)
    torch.cuda.synchronize()
    lib.ffr_debug_set_prof(None)
    b = buf.view(160, 32).double()
    b = b[b[:, 0] > 0]
    m = b.mean(0)
    lead = b[b[:, 4] > 0]
    ml = lead.mean(0)
    tiles = ml[8].item()
    print(f"  prof [{n_ref}x{n_cand}x{dim}] cg={os.environ.get('FFR_CTA_GROUP', '1')} ctas={b.shape[0]} (leaders {lead.shape[0]}), "
          f"ref tiles per CTA {tiles:.0f}")
    print(f"    TMA thread : total {m[0]:.3e} cyc; waiting a_empty {m[1] / m[0]:.1%}, b_empty {m[2] / m[0]:.1%}")
    print(f"    MMA thread : total {ml[4]:.3e} cyc ({ml[4] / tiles:.0f} per ref tile); waiting a_full {ml[5] / ml[4]:.1%}, "
          f"t_empty {ml[6] / ml[4]:.1%}, b_full {ml[7] / ml[4]:.1%}")
    print(f"    epilogue w4: total {m[10]:.3e} cyc; waiting t_full {m[11] / m[10]:.1%} "
          f"(busy {(m[10] - m[11]) / tiles:.0f} cyc per ref tile)", flush=True)
    if m[3] > 0:
        print(f"      epilogue w4 per ref tile: hot loop {m[3] / tiles:.0f} cyc; end-of-candidate-tile section {m[17] / tiles:.0f} cyc per ref tile "
              f"(of which waiting for the upper column part {m[16] / tiles:.0f})", flush=True)
    if m[12] > 0:
        ent = b[:, 15]
        print(f"    setup (entry -> barriers/TMEM/cluster sync done): mean {m[12] / 1e3:.2f} us, max {b[:, 12].max().item() / 1e3:.2f} us; "
              f"CTA entry spread {(ent.max() - ent.min()).item() / 1e3:.2f} us; first entry -> last exit {(b[:, 9].max() - ent.min()).item() / 1e3:.2f} us", flush=True)
    if m[13] > 0:
        print(f"    normaliser 0: total {m[13]:.3e} cyc for {m[14]:.0f} candidate tiles ({m[13] / max(m[14], 1):.0f} per tile); "
              f"stage32: waiting for the A stage {m[18] / m[13]:.1%}, for staged fp32 rows {m[19] / m[13]:.1%}, "
              f"merge + emit of finished tiles {m[20] / m[13]:.1%} ({m[20] / max(m[14], 1):.0f} cyc per tile)", flush=True)


if __name__ == "__main__":
    print(torch.cuda.get_device_name(0), _lib.load().ffr_build_info().decode(), "FFR_CTA_GROUP =", os.environ.get("FFR_CTA_GROUP"))
    ok = True
    if "--raw" in sys.argv:
        for shape in [(256, 128, 64), (256, 256, 128), (512, 256, 512), (100, 77, 128), (1000, 333, 192), (4096, 4096, 256)]:
            ok = raw(*shape) and ok
        print("RAW", "OK" if ok else "FAILED", flush=True)
    if "--perf" in sys.argv and ok:
        perf(1000, 100_000, 128)
        perf(1000, 100_000, 128, flags=ops.FLAG_NO_RECHECK)
        perf(10_000, 1_000_000, 512)
        perf(10_000, 1_000_000, 512, flags=ops.FLAG_NO_RECHECK)
        perf(100_000, 1_250_000, 128, flags=ops.FLAG_NO_RECHECK, iters=2)
        perf(256, 2_000_000, 128, flags=ops.FLAG_NO_RECHECK)
    if "--prof" in sys.argv:
        prof(10_000, 1_000_000, 512)
        prof(10_000, 500_000, 256)
        prof(100_000, 300_000, 128)
        prof(1000, 100_000, 128)
        prof(256, 2_000_000, 128)
    if "--prof-easy" in sys.argv:
        prof(100_000, 300_000, 128, easy=True)
        prof(1000, 100_000, 128, easy=True)
        prof(10_000, 500_000, 256, easy=True)
    if "--prof128" in sys.argv:
        prof(100_000, 300_000, 128)
        prof(1000, 100_000, 128)
    if "--grid" in sys.argv:
        # grid update path unconditional (every part) against gated (behind one branch on the part maximum), per shape
        for shape in [(1000, 100_000, 128), (256, 2_000_000, 128), (4000, 400_000, 128), (10_000, 500_000, 256),
                      (100_000, 300_000, 128)]:
            for g in ("0", "1000000"):
                setenv("FFR_GRID_UPDATE_REFS", g)
                print(f" FFR_GRID_UPDATE_REFS={g}")
                prof(*shape)
                perf(*shape, flags=ops.FLAG_NO_RECHECK, iters=3)
        delenv("FFR_GRID_UPDATE_REFS")
    if "--small" in sys.argv:
        for ex in ("auto",):
            print(f" FFR_GRID_EXACT={ex}")
            for shape in [(1000, 100_000, 128), (256, 2_000_000, 128), (4000, 400_000, 128), (100_000, 300_000, 128),
                          (10_000, 500_000, 256), (10_000, 300_000, 512)]:
                prof(*shape)
                perf(*shape, flags=ops.FLAG_NO_RECHECK, iters=3)
                perf(*shape, iters=3)
    if "--big" in sys.argv:
        prof(10_000, 1_000_000, 512)
        prof(10_000, 400_000, 384)
        perf(10_000, 1_250_000, 512, iters=3)
        perf(10_000, 1_000_000, 512, flags=ops.FLAG_NO_RECHECK, iters=3)
        perf(10_000, 400_000, 384, flags=ops.FLAG_NO_RECHECK, iters=3)
        perf(10_000, 500_000, 256, flags=ops.FLAG_NO_RECHECK, iters=3)
        perf(100_000, 1_250_000, 128, iters=2)
    if "--benchprof" in sys.argv:
        # the bench's own cfg3 / cfg4 inputs, re-check on: this round's K2 in cycles
        prof(10_000, 1_250_000, 512, bench_data=True, flags=0)
        prof(100_000, 1_250_000, 128, bench_data=True, flags=0)
        prof(1_000, 100_000, 128, bench_data=True, flags=0)
    if "--stage32" in sys.argv:
        for st in ("1",):
            setenv("FFR_STAGE32", st)
            print(f" FFR_STAGE32={st}")
            for shape in [(1000, 100_000, 128), (256, 2_000_000, 128), (64, 4_000_000, 128), (4000, 400_000, 128)]:
                prof(*shape)
                perf(*shape, iters=3)
        delenv("FFR_STAGE32")
    if "--st32prof" in sys.argv:
        prof(256, 2_000_000, 128)
        prof(1000, 100_000, 128)
        for shape in [(1000, 100_000, 128), (256, 2_000_000, 128), (64, 4_000_000, 128), (4000, 400_000, 128)]:
            perf(*shape, iters=3)
    if "--midn" in sys.argv:
        for shape in [(64, 4_000_000, 128), (256, 2_000_000, 128), (32, 2_000_000, 128), (500, 1_000_000, 128), (256, 1_000_000, 512)]:
            perf(*shape, iters=3)
    if "--stream" in sys.argv:
        perf(1, 10_000_000, 128, metric="euclid", thr=1.0)
        perf(1, 4_000_000, 512, metric="euclid", thr=1.0)
        perf(8, 10_000_000, 128)
    if "--perf2" in sys.argv:
        perf(1000, 100_000, 128, flags=ops.FLAG_NO_RECHECK)
        perf(100_000, 1_250_000, 128, flags=ops.FLAG_NO_RECHECK, iters=2)
        perf(10_000, 500_000, 256, flags=ops.FLAG_NO_RECHECK, iters=3)
        perf(10_000, 1_000_000, 512, flags=ops.FLAG_NO_RECHECK, iters=3)
