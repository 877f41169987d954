"""Candidate-axis sharding across the GPUs of one box (SURVEY.md §8e).

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
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch

__all__ = ["shard_range", "pack_results", "unpack_results", "CandidateSharder"]


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
