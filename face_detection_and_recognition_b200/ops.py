"""Torch-facing wrappers over the C ABI (include/ffr.h).  PyTorch is plumbing here: it owns device memory
and the current stream; every computation happens in libffr_b200.so.

Reference expressions replaced (paths relative to SamSamhuns/face_detection_and_recognition):
  l2norm_rows        face_detection_and_extraction/modules/mobile_facenet/mobile_facenet.py:30-33
                     face_detection_and_extraction/face_extraction/extract_and_clean_imdb_wiki_faces.py:146
  face_filter        similar_face_filtering/filter_faces_using_reference.py:186-189 (euclid, one mean vector)
                     face_detection_and_extraction/face_extraction/extract_and_label_faces_from_dataset.py:101-116
  ref_mean_and_thres similar_face_filtering/filter_faces_using_reference.py:85-99
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import (DTYPE_F16, DTYPE_F32, ERR_UNSUPPORTED, FLAG_FORCE_FP32, FLAG_FORCE_MMA, FLAG_NO_RECHECK, METRIC_COSINE,
                   METRIC_EUCLID, SELF_EARLIER, SELF_OTHERS, FfrError, check)

__all__ = ["l2norm_rows", "face_filter", "self_filter", "cosine_filter", "ref_mean_and_thres", "FilterResult", "HostFilter", "GraphedFilter",
           "ResultGather", "launch_count", "METRIC_COSINE", "METRIC_EUCLID", "FLAG_FORCE_FP32", "FLAG_FORCE_MMA",
           "FLAG_NO_RECHECK", "SELF_OTHERS", "SELF_EARLIER"]

_METRICS = {"cosine": METRIC_COSINE, "euclid": METRIC_EUCLID, "euclidean": METRIC_EUCLID,
            METRIC_COSINE: METRIC_COSINE, METRIC_EUCLID: METRIC_EUCLID}
_SELF_MODES = {"others": SELF_OTHERS, "earlier": SELF_EARLIER, SELF_OTHERS: SELF_OTHERS, SELF_EARLIER: SELF_EARLIER}


def _stream_ptr(dev: torch.device) -> int:
    return torch.cuda.current_stream(dev).cuda_stream


def _require_cuda(t: torch.Tensor, name: str, dtype=torch.float32) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name} must be a CUDA tensor (the filter has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


_ws_cache: dict = {}


def _workspace(dev: torch.device, nbytes: int) -> torch.Tensor:
    """Grow-only per-(device, stream) scratch buffer; 256-byte aligned by the caching allocator."""
    key = (dev.index, _stream_ptr(dev))
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 4096), dtype=torch.uint8, device=dev)
        _ws_cache[key] = buf
    return buf


def launch_count() -> int:
    """Kernels launched by libffr_b200.so in this process so far."""
    return int(_lib.load().ffr_launch_count())


def l2norm_rows(x: torch.Tensor, want_f16: bool = False, want_f32: bool = True, want_norms: bool = False):
    """Row-wise ``x / ||x||_2`` (no epsilon).  Returns a dict with the requested outputs:
    ``f32`` [rows, dim] float32, ``f16`` [rows, padded_dim] float16 (zero padded to a multiple of 64: the
    layout the tensor-core filter consumes), ``norms`` [rows] float32."""
    lib = _lib.load()
    x = _require_cuda(x, "x")
    if x.dim() != 2:
        raise ValueError("x must be [rows, dim]")
    rows, dim = x.shape
    dev = x.device
    out = {}
    y32 = torch.empty_like(x) if want_f32 else None
    ld = int(lib.ffr_padded_dim(dim))
    y16 = torch.empty((rows, ld), dtype=torch.float16, device=dev) if want_f16 else None
    nrm = torch.empty((rows,), dtype=torch.float32, device=dev) if want_norms else None
    with torch.cuda.device(dev):
        check(lib.ffr_l2norm_rows_f32(x.data_ptr(), rows, dim, y16.data_ptr() if want_f16 else None, ld,
                                      y32.data_ptr() if want_f32 else None, nrm.data_ptr() if want_norms else None,
                                      _stream_ptr(dev)))
    if want_f32:
        out["f32"] = y32
    if want_f16:
        out["f16"] = y16
    if want_norms:
        out["norms"] = nrm
    return out


@dataclass
class FilterResult:
    keep: torch.Tensor                       # uint8 [M]   1 = similar ("clean"), 0 = discard ("unclean")
    best_idx: torch.Tensor                   # int32 [M]   first arg-best reference (+ ref_index_base)
    best_val: torch.Tensor                   # float32 [M] cosine similarity, or euclid distance
    band_rows: Optional[torch.Tensor] = None  # int64 [B]  rows with |best - thr| <= band_tol (sorted)
    stats: Optional[dict] = None


def face_filter(ref: torch.Tensor, cand: torch.Tensor, thr: float, metric="cosine", ref_index_base: int = 0,
                band_tol: Optional[float] = None, flags: int = 0, want_stats: bool = False,
                out: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None) -> FilterResult:
    """Fused reference x candidate filter on one GPU.

    cosine: best = max_i cos(r_i, c), keep = best >= thr;  euclid: best = min_i |c - r_i|, keep = best <= thr.
    ``ref`` [N, D], ``cand`` [M, D]: float32 CUDA tensors (raw embeddings; normalisation is internal), or both
    float16 rows produced by ``l2norm_rows(want_f16=True)`` (cosine only).  ``band_tol`` additionally returns
    the rows whose best lies within that tolerance of ``thr``.

    Both metrics use the tensor cores from 9 references up (dim <= 512).  Euclid then returns the index of the exact fp32
    kernel (``FLAG_FORCE_FP32``) except on fp32 ties (two smallest distances within 1e-6 relative), and the same keep and
    distance bit for bit wherever the index agrees; with ``FLAG_NO_RECHECK`` Euclid runs the exact kernel."""
    lib = _lib.load()
    m = _METRICS[metric]
    if ref.dtype == torch.float16:
        dtype = DTYPE_F16
        ref = _require_cuda(ref, "ref", torch.float16)
        cand = _require_cuda(cand, "cand", torch.float16)
        dim = ref.shape[1]
        if dim != lib.ffr_padded_dim(dim):
            raise ValueError("float16 rows must have a leading dimension that is a multiple of 64")
    else:
        dtype = DTYPE_F32
        ref = _require_cuda(ref, "ref")
        cand = _require_cuda(cand, "cand")
        dim = ref.shape[1]
    if ref.dim() != 2 or cand.dim() != 2 or cand.shape[1] != ref.shape[1]:
        raise ValueError(f"ref {tuple(ref.shape)} and cand {tuple(cand.shape)} must be [N, D] and [M, D]")
    if ref.device != cand.device:
        raise ValueError("ref and cand must be on the same device")
    n_ref, n_cand = ref.shape[0], cand.shape[0]
    dev = cand.device
    if out is None:
        keep = torch.empty((n_cand,), dtype=torch.uint8, device=dev)
        idx = torch.empty((n_cand,), dtype=torch.int32, device=dev)
        val = torch.empty((n_cand,), dtype=torch.float32, device=dev)
    else:
        keep, idx, val = out
    ws_bytes = int(lib.ffr_filter_workspace_bytes(n_ref, n_cand, dim, dtype, m))
    ws = _workspace(dev, ws_bytes)
    band_count = band_rows = None
    if band_tol is not None:
        band_count = torch.zeros((1,), dtype=torch.int32, device=dev)
        band_rows = torch.empty((max(n_cand, 1),), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        check(lib.ffr_filter_ex(ref.data_ptr(), n_ref, cand.data_ptr() if n_cand else None, n_cand, dim, dtype,
                                None, None, m, float(thr), int(ref_index_base),
                                keep.data_ptr() if n_cand else None, idx.data_ptr() if n_cand else None,
                                val.data_ptr() if n_cand else None,
                                float(band_tol or 0.0), band_count.data_ptr() if band_count is not None else None,
                                band_rows.data_ptr() if band_rows is not None else None, n_cand, int(flags),
                                ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
        res = FilterResult(keep, idx, val)
        if band_tol is not None:
            n = int(band_count.item())
            res.band_rows = torch.sort(band_rows[:min(n, n_cand)]).values
        if want_stats:
            res.stats = _stats(lib, ws, dev)
    return res


def _stats(lib, ws, dev) -> dict:
    arr = (C.c_int64 * 8)()
    check(lib.ffr_filter_stats(ws.data_ptr(), arr, _stream_ptr(dev)))
    stats = {"rechecked": arr[0], "part_rescans": arr[4], "full_rescans": arr[1],
             "path": "tcgen05" if arr[2] == 1 else "fp32", "launches": arr[3], "refs_scanned": arr[5]}
    if arr[2] == 1:
        cfg = (C.c_int32 * 8)()
        lib.ffr_debug_last_k2_config(cfg)
        stats["k2"] = {"cta_group": cfg[0], "grid_exact": cfg[1], "grid_updates": cfg[2],
                       "normalise": ("k1", "fused_scratch", "stage32+tail_offload", "stage32")[cfg[3]], "a_stages": cfg[4],
                       "b_stages": cfg[5], "grid": cfg[6]}
    return stats


def self_filter(x: torch.Tensor, thr: float, metric="cosine", mode="others", rows: Optional[Tuple[int, int]] = None,
                band_tol: Optional[float] = None, flags: int = 0, want_stats: bool = False,
                out: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None) -> FilterResult:
    """Each row's best match among the OTHER rows of the same set ``x`` [N, D] (float32 CUDA): near-duplicates, repeated
    enrolments, a face that matches none of its classmates.

    ``mode="others"``: best over every row i != j.  ``mode="earlier"``: best over i < j -- with keep = 1 row j is a near-duplicate
    of an earlier row, so dropping exactly the kept rows leaves the first occurrence of every group.  ``rows=(begin, end)``
    filters only those candidate rows against all N (candidate-axis sharding); results are local to the range, ``best_idx`` is a
    global row of ``x``.  A row with no eligible reference (row 0 in "earlier", or N = 1) gets keep 0, index -1 and -inf (cosine)
    / +inf (Euclid).  Metric, threshold, band and precision contract are ``face_filter``'s on the masked problem; bit-identical
    rows are not folded.  fp16 rows and ``FLAG_NO_RECHECK`` are refused."""
    lib = _lib.load()
    m = _METRICS[metric]
    md = _SELF_MODES[mode]
    if isinstance(x, torch.Tensor) and x.dtype == torch.float16:
        raise FfrError(ERR_UNSUPPORTED, "self_filter takes float32 embeddings (fp16 rows are not supported)")
    x = _require_cuda(x, "x")
    if x.dim() != 2:
        raise ValueError(f"x {tuple(x.shape)} must be [N, D]")
    n, dim = x.shape
    begin, end = (0, n) if rows is None else (int(rows[0]), int(rows[1]))
    n_rows = max(end - begin, 0)
    dev = x.device
    if out is None:
        keep = torch.empty((n_rows,), dtype=torch.uint8, device=dev)
        idx = torch.empty((n_rows,), dtype=torch.int32, device=dev)
        val = torch.empty((n_rows,), dtype=torch.float32, device=dev)
    else:
        keep, idx, val = out
    ws = _workspace(dev, int(lib.ffr_filter_self_workspace_bytes(n, n_rows, dim, m)))
    band_count = band_rows = None
    if band_tol is not None:
        band_count = torch.zeros((1,), dtype=torch.int32, device=dev)
        band_rows = torch.empty((max(n_rows, 1),), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        check(lib.ffr_filter_self(x.data_ptr(), n, begin, end - begin, dim, m, md, float(thr),
                                  keep.data_ptr() if n_rows else None, idx.data_ptr() if n_rows else None,
                                  val.data_ptr() if n_rows else None,
                                  float(band_tol or 0.0), band_count.data_ptr() if band_count is not None else None,
                                  band_rows.data_ptr() if band_rows is not None else None, n_rows, int(flags),
                                  ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
        res = FilterResult(keep, idx, val)
        if band_tol is not None:
            res.band_rows = torch.sort(band_rows[:min(int(band_count.item()), n_rows)]).values
        if want_stats:
            res.stats = _stats(lib, ws, dev)
    return res


class GraphedFilter:
    """``face_filter`` for fixed shapes captured once into a CUDA graph: the whole K1 -> K2 -> K3 launch sequence replays
    as ONE graph launch with no host work between the kernels.  Worth it when the step is launch-bound (BASELINE
    configs[1]: ~25 us of GPU work).  Either own static input tensors (``GraphedFilter(n_ref, n_cand, dim, thr)``; inputs
    are copied in by ``__call__``) or wrap the caller's tensors in place (``GraphedFilter.capture(ref, cand, thr, out=...)``:
    ``replay()`` re-runs the filter on whatever those tensors hold)."""

    def __init__(self, n_ref: int, n_cand: int, dim: int, thr: float, metric="cosine", device: int = 0, flags: int = 0,
                 _tensors=None):
        self.dev = torch.device("cuda", device)
        self.thr, self.metric, self.flags = float(thr), metric, flags
        if _tensors is None:
            self.ref = torch.zeros((n_ref, dim), dtype=torch.float32, device=self.dev)
            self.cand = torch.zeros((n_cand, dim), dtype=torch.float32, device=self.dev)
            out = (torch.empty(n_cand, dtype=torch.uint8, device=self.dev), torch.empty(n_cand, dtype=torch.int32, device=self.dev),
                   torch.empty(n_cand, dtype=torch.float32, device=self.dev))
            self.ref.normal_()
            self.cand.normal_()
        else:
            self.ref, self.cand, out = _tensors
        side = torch.cuda.Stream(self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):                              # warm-up on the side stream (workspace, attributes)
            l0 = launch_count()
            face_filter(self.ref, self.cand, self.thr, metric=metric, flags=flags, out=out)
            self.launches = launch_count() - l0                    # kernels of this library per replay
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=side):
            self.result = face_filter(self.ref, self.cand, self.thr, metric=metric, flags=flags, out=out)

    @classmethod
    def capture(cls, ref: torch.Tensor, cand: torch.Tensor, thr: float, metric="cosine", flags: int = 0, out=None):
        ref, cand = _require_cuda(ref, "ref"), _require_cuda(cand, "cand")
        if out is None:
            out = (torch.empty(cand.shape[0], dtype=torch.uint8, device=cand.device),
                   torch.empty(cand.shape[0], dtype=torch.int32, device=cand.device),
                   torch.empty(cand.shape[0], dtype=torch.float32, device=cand.device))
        return cls(ref.shape[0], cand.shape[0], ref.shape[1], thr, metric=metric, device=cand.device.index, flags=flags,
                   _tensors=(ref, cand, out))

    def replay(self) -> FilterResult:
        self.graph.replay()
        return self.result

    def __call__(self, ref: torch.Tensor, cand: torch.Tensor) -> FilterResult:
        self.ref.copy_(ref, non_blocking=True)
        self.cand.copy_(cand, non_blocking=True)
        return self.replay()


def cosine_filter(ref, cand, thr, **kw) -> FilterResult:
    return face_filter(ref, cand, thr, metric="cosine", **kw)


def ref_mean_and_thres(ref_feat: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Mean vector and max distance from it (filter_faces_using_reference.py:85-99).  ``ref_feat`` [R, D] or
    [R, 1, D] float32 CUDA.  Returns (mean [1, D], thres [] ) on the device."""
    lib = _lib.load()
    ref_feat = _require_cuda(ref_feat, "ref_feat")
    if ref_feat.dim() == 3:
        ref_feat = ref_feat.reshape(ref_feat.shape[0], -1)
    r, d = ref_feat.shape
    dev = ref_feat.device
    mean = torch.empty((1, d), dtype=torch.float32, device=dev)
    thres = torch.empty((), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib.ffr_ref_mean_and_thres(ref_feat.data_ptr(), r, d, mean.data_ptr(), thres.data_ptr(), _stream_ptr(dev)))
    return mean, thres


def ref_mean_and_thres_batched(ref_feat: torch.Tensor, counts) -> Tuple[torch.Tensor, torch.Tensor]:
    """All classes in one launch: ``ref_feat`` [sum(counts), D] float32 CUDA holds the reference embeddings of class 0,
    then class 1, ...; returns (mean [C, D], thres [C]) with the per-class arithmetic of ``ref_mean_and_thres``."""
    lib = _lib.load()
    ref_feat = _require_cuda(ref_feat, "ref_feat")
    dev = ref_feat.device
    counts = [int(c) for c in counts]
    if sum(counts) != ref_feat.shape[0]:
        raise ValueError("counts must sum to the number of reference rows")
    offs = torch.tensor([0] + list(np.cumsum(counts)), dtype=torch.int32, device=dev)
    d = ref_feat.shape[1]
    mean = torch.empty((len(counts), d), dtype=torch.float32, device=dev)
    thres = torch.empty((len(counts),), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib.ffr_ref_mean_and_thres_batched(ref_feat.data_ptr(), offs.data_ptr(), len(counts), d, mean.data_ptr(),
                                                 thres.data_ptr(), _stream_ptr(dev)))
    return mean, thres


class FaceGallery:
    """Device-resident face gallery with the reference tracker's semantics (extract_and_label_faces_from_dataset.py
    :101-121): ``match`` processes the queries in order; the FIRST gallery entry that satisfies
    ``(dist < normal_thres and iou > 0.1) or dist < harsh_thres`` is overwritten by the query, otherwise the query is
    appended.  Returns (found bool[q], faceid int[q]) with faceid = position + 1 like ``add_face`` (:118-121)."""

    def __init__(self, dim: int, capacity: int = 4096, metric="cosine", normal_thres: float = 1.0,
                 harsh_thres: float = 0.72, device: int = 0):
        self._lib = _lib.load()
        self.dev = torch.device("cuda", device)
        self.dim, self.capacity, self.metric = dim, capacity, _METRICS[metric]
        self.normal_thres, self.harsh_thres = float(normal_thres), float(harsh_thres)
        self.feat = torch.zeros((capacity, dim), dtype=torch.float32, device=self.dev)
        self.bbox = torch.zeros((capacity, 4), dtype=torch.float32, device=self.dev)
        self.count = torch.zeros((1,), dtype=torch.int32, device=self.dev)

    def __len__(self) -> int:
        return int(self.count.item())

    def clear(self):
        self.count.zero_()

    def match(self, feats, bboxes=None):
        q = torch.as_tensor(feats, dtype=torch.float32).to(self.dev).contiguous().reshape(-1, self.dim)
        b = None if bboxes is None else torch.as_tensor(bboxes, dtype=torch.float32).to(self.dev).contiguous().reshape(-1, 4)
        out = torch.empty((q.shape[0],), dtype=torch.int32, device=self.dev)
        with torch.cuda.device(self.dev):
            check(self._lib.ffr_first_match_stream(self.feat.data_ptr(), self.bbox.data_ptr(), self.count.data_ptr(),
                                                   self.capacity, q.data_ptr(), b.data_ptr() if b is not None else None,
                                                   q.shape[0], self.dim, self.metric, self.normal_thres, self.harsh_thres,
                                                   out.data_ptr(), _stream_ptr(self.dev)))
        m = out.cpu().numpy()
        if (m == np.iinfo(np.int32).min).any():
            raise RuntimeError(f"gallery capacity {self.capacity} exhausted")
        found = m >= 0
        faceid = np.where(found, m, -1 - m) + 1
        return found, faceid.astype(np.int32)


class HostFilter:
    """Host-buffer entry point (ffr_ctx_*): NumPy / pinned-torch arrays in, NumPy arrays out; candidates are
    streamed to the GPU in chunks while the previous chunk is being filtered."""

    def __init__(self, device: int = 0, max_ref: int = 1 << 14, chunk_cand: int = 1 << 18, max_dim: int = 512):
        self._lib = _lib.load()
        self._h = C.c_void_p()
        check(self._lib.ffr_ctx_create(int(device), int(max_ref), int(chunk_cand), int(max_dim), C.byref(self._h)))

    def close(self):
        if self._h:
            self._lib.ffr_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(self._lib.ffr_ctx_launch_count(self._h))

    @staticmethod
    def _ptr(a):
        if isinstance(a, torch.Tensor):
            if a.is_cuda:
                raise TypeError("HostFilter takes host arrays; use face_filter for CUDA tensors")
            return a.data_ptr()
        return a.ctypes.data

    def __call__(self, ref, cand, thr: float, metric="cosine", ref_index_base: int = 0, flags: int = 0, out=None):
        m = _METRICS[metric]
        if not isinstance(ref, torch.Tensor):
            ref = np.ascontiguousarray(ref, dtype=np.float32)
        if not isinstance(cand, torch.Tensor):
            cand = np.ascontiguousarray(cand, dtype=np.float32)
        n_ref, dim = ref.shape
        n_cand = cand.shape[0]
        if out is None:
            keep = np.empty(n_cand, dtype=np.uint8)
            idx = np.empty(n_cand, dtype=np.int32)
            val = np.empty(n_cand, dtype=np.float32)
        else:
            keep, idx, val = out
        check(self._lib.ffr_ctx_filter_host(self._h, self._ptr(ref), n_ref, self._ptr(cand) if n_cand else None, n_cand,
                                            dim, m, float(thr), int(ref_index_base),
                                            self._ptr(keep) if n_cand else None, self._ptr(idx) if n_cand else None,
                                            self._ptr(val) if n_cand else None, int(flags)))
        return keep, idx, val


class ResultGather:
    """K4: one NCCL allgather of the packed per-candidate {best_idx, keep} over NVLink (ffr_comm_*); for a gallery sharded
    over the ranks, one uint64 max all-reduce of each row's packed best match (``allreduce_best``).

    The 128-byte NCCL unique id is created on rank 0 and broadcast through ``torch.distributed`` (any backend)."""

    def __init__(self, rank: int, world_size: int, device: int):
        import torch.distributed as dist
        self._lib = _lib.load()
        self.rank, self.world_size, self.device = rank, world_size, device
        uid = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            buf = (C.c_uint8 * 128)()
            check(self._lib.ffr_nccl_unique_id(buf))
            uid = torch.tensor(list(buf), dtype=torch.uint8)
        if world_size > 1:
            obj = [uid]
            dist.broadcast_object_list(obj, src=0)
            uid = obj[0]
        raw = (C.c_uint8 * 128)(*uid.tolist())
        self._h = C.c_void_p()
        check(self._lib.ffr_comm_create(raw, world_size, rank, device, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ffr_comm_destroy(self._h)
            self._h = C.c_void_p()

    def buffers(self, m_local: int, device=None):
        """In-place form: returns (keep_all, idx_all, keep_mine, idx_mine).  Hand ``keep_mine`` / ``idx_mine`` (views of
        this rank's slice) to ``face_filter(out=...)`` and call ``all_gather_inplace`` -- no pack / unpack kernels."""
        dev = torch.device("cuda", self.device) if device is None else device
        key = (m_local, dev)
        if getattr(self, "_buf_key", None) != key:
            self._keep_all = torch.empty((m_local * self.world_size,), dtype=torch.uint8, device=dev)
            self._idx_all = torch.empty((m_local * self.world_size,), dtype=torch.int32, device=dev)
            self._buf_key = key
        a, b = self.rank * m_local, (self.rank + 1) * m_local
        return self._keep_all, self._idx_all, self._keep_all[a:b], self._idx_all[a:b]

    def all_gather_inplace(self, keep_all: torch.Tensor, idx_all: torch.Tensor):
        m = keep_all.numel() // self.world_size
        dev = keep_all.device
        with torch.cuda.device(dev):
            check(self._lib.ffr_allgather_results_inplace(self._h, keep_all.data_ptr(), idx_all.data_ptr(), m,
                                                          _stream_ptr(dev)))
        return keep_all, idx_all

    def allreduce_best(self, ref_local: Optional[torch.Tensor], cand: torch.Tensor, thr: float, best_idx: torch.Tensor,
                       ref_index_base: int = 0, metric="cosine", band_tol: Optional[float] = None,
                       out: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None) -> FilterResult:
        """Gallery sharded over the ranks (ffr_allreduce_best): ``best_idx`` is this rank's ``face_filter(ref_local, cand, thr,
        ref_index_base=ref_index_base).best_idx`` (global indices; ``ref_local`` None or empty: this rank has no references
        and ran no filter).  Returns the result for the whole gallery, identical on every rank: the fp32 value of each rank's
        winner is recomputed, the best (then the smallest global index) wins one uint64 max all-reduce, and keep / band follow
        from ``thr``.  A row no rank had a reference for gets keep 0, index -1 and -inf (cosine) / +inf (Euclid)."""
        m = _METRICS[metric]
        cand = _require_cuda(cand, "cand")
        if cand.dim() != 2:
            raise ValueError(f"cand {tuple(cand.shape)} must be [M, D]")
        n_cand, dim = cand.shape
        dev = cand.device
        n_ref = 0 if ref_local is None else int(ref_local.shape[0])
        if n_ref:
            ref_local = _require_cuda(ref_local, "ref_local")
            if ref_local.dim() != 2 or ref_local.shape[1] != dim or ref_local.device != dev:
                raise ValueError(f"ref_local {tuple(ref_local.shape)} must be [N, {dim}] on {dev}")
        if (not isinstance(best_idx, torch.Tensor) or best_idx.dtype != torch.int32 or best_idx.device != dev
                or tuple(best_idx.shape) != (n_cand,)):
            raise ValueError(f"best_idx must be an int32 tensor of shape ({n_cand},) on {dev}, got "
                             f"{getattr(best_idx, 'dtype', type(best_idx))} {tuple(getattr(best_idx, 'shape', ()))} "
                             f"on {getattr(best_idx, 'device', None)}")
        if out is None:
            out = (torch.empty((n_cand,), dtype=torch.uint8, device=dev), torch.empty((n_cand,), dtype=torch.int32, device=dev),
                   torch.empty((n_cand,), dtype=torch.float32, device=dev))
        keep, idx, val = out
        if idx.data_ptr() != best_idx.data_ptr():
            idx.copy_(best_idx)
        band_count = band_rows = None
        if band_tol is not None:
            band_count = torch.zeros((1,), dtype=torch.int32, device=dev)
            band_rows = torch.empty((max(n_cand, 1),), dtype=torch.int64, device=dev)
        ws = _workspace(dev, int(self._lib.ffr_allreduce_best_workspace_bytes(n_cand)))
        with torch.cuda.device(dev):
            check(self._lib.ffr_allreduce_best(self._h, ref_local.data_ptr() if n_ref else None, n_ref, int(ref_index_base),
                                               cand.data_ptr() if n_cand else None, n_cand, dim, m, float(thr),
                                               keep.data_ptr() if n_cand else None, idx.data_ptr() if n_cand else None,
                                               val.data_ptr() if n_cand else None, float(band_tol or 0.0),
                                               band_count.data_ptr() if band_count is not None else None,
                                               band_rows.data_ptr() if band_rows is not None else None, n_cand,
                                               ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
        res = FilterResult(keep, idx, val)
        if band_tol is not None:
            res.band_rows = torch.sort(band_rows[:min(int(band_count.item()), n_cand)]).values
        return res

    def all_gather(self, keep_local: torch.Tensor, idx_local: torch.Tensor):
        m = keep_local.numel()
        dev = keep_local.device
        keep_all = torch.empty((m * self.world_size,), dtype=torch.uint8, device=dev)
        idx_all = torch.empty((m * self.world_size,), dtype=torch.int32, device=dev)
        nbytes = int(self._lib.ffr_allgather_workspace_bytes(self.world_size, m))
        ws = _workspace(dev, nbytes)
        with torch.cuda.device(dev):
            check(self._lib.ffr_allgather_results(self._h, keep_local.data_ptr(), idx_local.data_ptr(), m,
                                                  keep_all.data_ptr(), idx_all.data_ptr(), ws.data_ptr(), ws.numel(),
                                                  _stream_ptr(dev)))
        return keep_all, idx_all
