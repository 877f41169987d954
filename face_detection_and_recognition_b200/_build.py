"""In-tree build of libffr_b200.so (hand-written sm_100a CUDA + the C ABI of include/ffr.h).

nvcc cross-compiles for sm_100a without a GPU; the resulting .so sits next to this file so that it
travels to the GPU box with the repo snapshot.  No torch / pybind involved: the library is plain C ABI.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libffr_b200.so")
SOURCES = ["ffr_api.cu", "ffr_l2norm.cu", "ffr_filter_fp32.cu", "ffr_filter_mma.cu", "ffr_recheck.cu", "ffr_gallery.cu", "ffr_dedup.cu",
           "ffr_groups.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(PKG_DIR), "include", "ffr.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link libffr_b200.so.  Returns the library path."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = _nvcc()
    obj_dir = os.path.join(PKG_DIR, "build")
    os.makedirs(obj_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), file=sys.stderr)
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out:
            print(out, file=sys.stderr)
        objs.append(obj)
    tmp = LIB_PATH + ".tmp"
    cmd = [nvcc, "-shared", "-o", tmp, *objs, "-cudart", "static", "-ldl", "-lpthread", "-lrt"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp, LIB_PATH)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
