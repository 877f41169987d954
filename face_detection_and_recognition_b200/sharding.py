"""Candidate-axis and gallery (reference-axis) sharding across the GPUs of one box (SURVEY.md §8e, DESIGN.md §7).

Every candidate's result depends only on that candidate and the (replicated) reference set, so candidates are split
into contiguous, equal ranges -- ``m_local = ceil(M / G)`` rows per rank, the last range padded -- each rank runs the
single-GPU filter on its range with ``ref_index_base = 0`` (indices stay global), and the per-candidate
``{best_idx i32, keep u8}`` records are gathered with ONE all-gather of 5 bytes per candidate.  No reduction across
ranks exists on this path; nothing else crosses NVLink.

Two gather back ends share one wire format ([idx i32 x m_pad][keep u8 x m_pad] per rank, m_pad = m_local rounded up
to 16):
  * ``"nccl"``  libffr_b200.so's own communicator (ffr_comm_*, K4: every rank's filter writes its slice of the final
    arrays, one grouped in-place ncclAllGather fills in the others), used on GPUs;
  * ``"dist"``  ``torch.distributed.all_gather_into_tensor`` on the process group the caller initialised -- this is
    what the world_size-2 ``gloo`` tests exercise on CPU (host-side plumbing only; the filter itself is injected).

``GallerySharder`` splits the REFERENCES instead (a gallery too large for one GPU, or a probe batch too small to keep every
GPU busy streaming the whole gallery): each rank filters the replicated candidates against its contiguous gallery range with
``ref_index_base`` = the range's start, and one max all-reduce of a 64-bit key per candidate -- the winner's value, then
its smallest global index -- merges the ranks (``ops.ResultGather.allreduce_best``; ``pack_best_keys`` for ``"dist"``).
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch

__all__ = ["shard_range", "pack_results", "unpack_results", "CandidateSharder", "pack_best_keys", "unpack_best_keys",
           "GallerySharder"]


def shard_range(n_cand: int, world: int, rank: int) -> Tuple[int, int, int]:
    """(start, stop, m_local) of ``rank``'s contiguous candidate range; ``stop - start <= m_local`` (the tail ranks
    may be short or empty), ``m_local = ceil(n_cand / world)`` is what every rank contributes to the gather."""
    if world <= 0 or not 0 <= rank < world:
        raise ValueError(f"bad rank {rank} / world {world}")
    m_local = -(-n_cand // world) if n_cand > 0 else 0
    start = min(rank * m_local, n_cand)
    stop = min(start + m_local, n_cand)
    return start, stop, m_local


def _m_pad(m_local: int) -> int:
    return (m_local + 15) // 16 * 16


def pack_results(keep: torch.Tensor, idx: torch.Tensor, m_local: int) -> torch.Tensor:
    """[idx i32 x m_pad][keep u8 x m_pad] as one uint8 buffer (rows beyond len(keep) are zero)."""
    m_pad = _m_pad(m_local)
    buf = torch.zeros(5 * m_pad, dtype=torch.uint8, device=keep.device)
    n = keep.numel()
    buf[:4 * n] = idx.to(torch.int32).contiguous().view(torch.uint8)
    buf[4 * m_pad:4 * m_pad + n] = keep.to(torch.uint8)
    return buf


def unpack_results(gathered: torch.Tensor, world: int, m_local: int, n_cand: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Inverse of ``pack_results`` over ``world`` rank blocks; returns (keep u8 [n_cand], idx i32 [n_cand])."""
    m_pad = _m_pad(m_local)
    blocks = gathered.view(world, 5 * m_pad)
    idx = blocks[:, :4 * m_pad].contiguous().view(torch.int32).view(world, m_pad)[:, :m_local].reshape(-1)[:n_cand]
    keep = blocks[:, 4 * m_pad:][:, :m_local].reshape(-1)[:n_cand]
    return keep.contiguous(), idx.contiguous()


class CandidateSharder:
    """Runs the filter on this rank's candidate range and gathers everybody's results.

    ``filter_fn(ref, cand_local, thr, metric=...)`` must return an object with ``.keep`` (uint8) and ``.best_idx``
    (int32) -- ``ops.face_filter`` on a GPU."""

    def __init__(self, rank: int, world: int, device: Optional[int] = None, gather: str = "nccl",
                 filter_fn: Optional[Callable] = None):
        self.rank, self.world, self.device = rank, world, device
        if gather not in ("nccl", "dist"):
            raise ValueError("gather must be 'nccl' or 'dist'")
        self.gather = gather
        self._rg = None
        if filter_fn is None:
            from . import ops
            filter_fn = ops.face_filter
        self.filter_fn = filter_fn
        if gather == "nccl" and world > 1:
            from . import ops
            self._rg = ops.ResultGather(rank, world, device if device is not None else 0)

    def local_range(self, n_cand: int) -> Tuple[int, int, int]:
        return shard_range(n_cand, self.world, self.rank)

    def filter(self, ref: torch.Tensor, cand_local: torch.Tensor, thr: float, n_cand_total: int, metric="cosine"):
        """``cand_local`` = rows [start, stop) of the global candidate matrix.  Returns (keep, best_idx) for ALL
        ``n_cand_total`` candidates on every rank, plus this rank's local result object."""
        start, stop, m_local = self.local_range(n_cand_total)
        if cand_local.shape[0] != stop - start:
            raise ValueError(f"rank {self.rank} expects {stop - start} local candidates, got {cand_local.shape[0]}")
        return self._gather(self.filter_fn(ref, cand_local, thr, metric=metric), m_local, n_cand_total)

    def self_filter(self, x: torch.Tensor, thr: float, metric="cosine", mode="others"):
        """Self mode (``ops.self_filter``) sharded over the candidate axis: every rank passes the FULL ``x`` and filters its
        ``shard_range`` of the rows against all of them.  Returns (keep, best_idx) for all rows on every rank, plus this rank's
        local result object."""
        from . import ops
        start, stop, m_local = self.local_range(x.shape[0])
        res = ops.self_filter(x, thr, metric=metric, mode=mode, rows=(start, stop))
        return self._gather(res, m_local, x.shape[0])

    def _gather(self, res, m_local: int, n_cand_total: int):
        """Every rank's (keep, best_idx) for all ``n_cand_total`` candidates, from this rank's local result ``res``."""
        if self.world == 1:
            return res.keep, res.best_idx, res
        if self.gather == "nccl":
            # in-place gather: this rank's slice of the final arrays is filled, one grouped NCCL launch fills the rest
            # (callers that own the output buffers skip even this copy: ResultGather.buffers + face_filter(out=...))
            n = res.keep.numel()
            keep_all, idx_all, keep_mine, idx_mine = self._rg.buffers(m_local, res.keep.device)
            keep_mine[:n], idx_mine[:n] = res.keep, res.best_idx
            keep_mine[n:], idx_mine[n:] = 0, 0
            self._rg.all_gather_inplace(keep_all, idx_all)
            return keep_all[:n_cand_total], idx_all[:n_cand_total], res
        import torch.distributed as dist
        send = pack_results(res.keep, res.best_idx, m_local)
        recv = torch.empty(self.world * send.numel(), dtype=torch.uint8, device=send.device)
        dist.all_gather_into_tensor(recv, send)
        keep_all, idx_all = unpack_results(recv, self.world, m_local, n_cand_total)
        return keep_all, idx_all, res

    def close(self):
        if self._rg is not None:
            self._rg.close()
            self._rg = None


_EUCLID = ("euclid", "euclidean", 1)
_U32 = 0xFFFFFFFF
_KEY_EMPTY = -(1 << 63)


def pack_best_keys(val: torch.Tensor, idx: torch.Tensor, metric="cosine") -> torch.Tensor:
    """int64 merge key of each row's best match: the C key of ffr_allreduce_best, ``(orderable(v) << 32) | ~idx`` with
    v = score (cosine) or -distance (Euclid), with its top bit flipped so that a SIGNED max orders it like the unsigned C
    key: the larger value wins, then the smaller index.  ``idx < 0`` (no reference on this rank) packs the identity,
    the smallest int64."""
    v = val.to(torch.float32).contiguous()
    if metric in _EUCLID:
        v = -v
    u = v.view(torch.int32).to(torch.int64) & _U32
    o = torch.where(u >= (1 << 31), (~u) & _U32, u | (1 << 31))
    idx = idx.to(torch.int64)
    keys = ((o - (1 << 31)) << 32) | (_U32 - (idx & _U32))
    return torch.where(idx >= 0, keys, torch.full_like(keys, _KEY_EMPTY))


def unpack_best_keys(keys: torch.Tensor, metric="cosine") -> Tuple[torch.Tensor, torch.Tensor]:
    """Inverse of ``pack_best_keys``: (best_val f32, best_idx i32); the identity gives index -1 and -inf (cosine) /
    +inf (Euclid)."""
    o = (keys >> 32) + (1 << 31)
    u = torch.where(o >= (1 << 31), o & 0x7FFFFFFF, (~o) & _U32)
    v = (u - (u >= (1 << 31)).to(torch.int64) * (1 << 32)).to(torch.int32).view(torch.float32)
    idx = (_U32 - (keys & _U32)).to(torch.int64)
    idx = (idx - (idx >= (1 << 31)).to(torch.int64) * (1 << 32)).to(torch.int32)
    euclid = metric in _EUCLID
    if euclid:
        v = -v
    empty = keys == _KEY_EMPTY
    v = torch.where(empty, torch.full_like(v, float("inf") if euclid else float("-inf")), v)
    return v, torch.where(empty, torch.full_like(idx, -1), idx)


class GallerySharder:
    """Gallery (reference-axis) sharding: rank r holds references ``shard_range(n_ref, world, r)`` and every rank the same
    candidates (probes); ``filter`` returns the result for the whole gallery, identical on every rank.

    ``reduce="nccl"``: the library's communicator (``ops.ResultGather.allreduce_best``: the fp32 value of every rank's
    winner is recomputed on the GPU before the merge, so ``face_filter``'s fp16-operand scores are never compared).
    ``reduce="dist"``: the same keys packed in torch and ``torch.distributed.all_reduce(MAX)`` on int64 over the caller's
    process group; it merges ``filter_fn``'s ``best_val`` as it is, so it needs an injected fp32 ``filter_fn`` (the CPU
    ``gloo`` tests inject the oracle).  ``filter_fn(ref_local, cand, thr, metric=..., ref_index_base=...)`` returns an
    object with ``.best_idx`` (and ``.best_val`` for ``"dist"``)."""

    def __init__(self, rank: int, world: int, device: Optional[int] = None, reduce: str = "nccl",
                 filter_fn: Optional[Callable] = None):
        if reduce not in ("nccl", "dist"):
            raise ValueError("reduce must be 'nccl' or 'dist'")
        if reduce == "dist" and filter_fn is None:
            raise ValueError("reduce='dist' merges filter_fn's best_val as it is: inject an fp32 filter_fn")
        self.rank, self.world, self.device, self.reduce = rank, world, device, reduce
        if filter_fn is None:
            from . import ops
            filter_fn = ops.face_filter
        self.filter_fn = filter_fn
        self._rg = None
        if reduce == "nccl":
            from . import ops
            self._rg = ops.ResultGather(rank, world, device if device is not None else 0)

    def shard_range(self, n_ref: int) -> Tuple[int, int]:
        """[start, stop) of this rank's references; ``start`` is its ``ref_index_base``."""
        start, stop, _ = shard_range(n_ref, self.world, self.rank)
        return start, stop

    def filter(self, ref_local: Optional[torch.Tensor], cand: torch.Tensor, thr: float, n_ref_total: int,
               metric="cosine", band_tol: Optional[float] = None):
        """``ref_local`` = rows ``shard_range(n_ref_total)`` of the gallery (None or empty on a rank without any), ``cand``
        the full candidate set.  Returns an ``ops.FilterResult`` for the whole gallery, the same on every rank."""
        if n_ref_total <= 0:
            raise ValueError("the gallery is empty")
        start, stop = self.shard_range(n_ref_total)
        n_local = 0 if ref_local is None else int(ref_local.shape[0])
        if n_local != stop - start:
            raise ValueError(f"rank {self.rank} expects {stop - start} gallery rows, got {n_local}")
        n_cand = cand.shape[0]
        res = self.filter_fn(ref_local, cand, thr, metric=metric, ref_index_base=start) if n_local else None
        if self.reduce == "nccl":
            idx = res.best_idx if res is not None else torch.full((n_cand,), -1, dtype=torch.int32, device=cand.device)
            return self._rg.allreduce_best(ref_local if n_local else None, cand, thr, idx, ref_index_base=start,
                                           metric=metric, band_tol=band_tol)
        import torch.distributed as dist
        from .ops import FilterResult
        if res is not None:
            keys = pack_best_keys(res.best_val, res.best_idx, metric)
        else:
            keys = torch.full((n_cand,), _KEY_EMPTY, dtype=torch.int64, device=cand.device)
        dist.all_reduce(keys, op=dist.ReduceOp.MAX)
        val, idx = unpack_best_keys(keys, metric)
        keep = ((val <= thr) if metric in _EUCLID else (val >= thr)).to(torch.uint8)
        out = FilterResult(keep, idx, val)
        if band_tol is not None:
            out.band_rows = torch.nonzero((val - thr).abs() <= band_tol).reshape(-1)
        return out

    def close(self):
        if self._rg is not None:
            self._rg.close()
            self._rg = None
