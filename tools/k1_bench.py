#!/usr/bin/env python
"""Times K1 (both matrices, one launch) alone: python tools/k1_bench.py [rows dim]"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from face_detection_and_recognition_b200 import ops
rows, dim = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (101_000, 128)
xs = [torch.randn(rows, dim, device="cuda") for _ in range(8)]          # rotate: 8 x 52 MB > L2
ops.l2norm_rows(xs[0], want_f16=True, want_f32=False)
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(41)]
ev[0].record()
for i in range(40):
    ops.l2norm_rows(xs[i % 8], want_f16=True, want_f32=False)
    ev[i + 1].record()
torch.cuda.synchronize()
ts = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(8, 40))
med = ts[len(ts) // 2]
print(f"K1 {rows}x{dim}: median {med * 1e3:.1f} us "
      f"min {ts[0] * 1e3:.1f} us  {rows * dim * 6 / med / 1e6:.0f} GB/s")
