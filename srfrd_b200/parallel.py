"""Host-side data-parallel protocol (one process per GPU, torch.distributed; NCCL over NVLink on the GPU box).

Training (SURVEY.md 8e): the global batch is split by rows, parameters and Adam state are replicated, and
    loss = sum_ranks [ sum_{t in rank} w_t * bce_t ] / W        with  W = all_reduce(sum_t w_t)
so every rank divides by the GLOBAL weight sum (the reference's mean over ``pos != 0`` of the whole batch,
trainer.py:36-38) and gradients are SUM-all-reduced: G ranks on B/G sequences reproduce one rank on B.
FusedTrainer implements exactly this on the device (two tiny all-reduces for W and the loss, one for the flat
gradient buffer).

Catalogue scoring: the (N+1)-row item table is row-sharded, every rank scores all users against its rows, and the
per-rank top-k lists (8 max(k, 10) B per user) are all-gathered and merged with the tie-break (score desc, id asc).
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch
import torch.distributed as dist


def shard_rows(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous row range [lo, hi) of rank `rank` when n rows are split over `world` ranks (ceil split)."""
    per = (n + world - 1) // world
    return min(rank * per, n), min((rank + 1) * per, n)


def shard_batch(batch: Dict[str, torch.Tensor], rank: int, world: int) -> Dict[str, torch.Tensor]:
    """Rank r takes rows [r*B/G, (r+1)*B/G) of every (B, ...) tensor in the batch."""
    B = next(iter(batch.values())).shape[0]
    lo, hi = shard_rows(B, rank, world)
    return {k: v[lo:hi] for k, v in batch.items()}


def allreduce_sum_(t: torch.Tensor, group=None) -> torch.Tensor:
    """In-place SUM all-reduce (no-op without a process group / at world size 1).  FusedTrainer uses it for the weight
    sums (loss normaliser, global count of pos != 0 -- trainer.py:36-38) and for the flat gradient bucket whose tail
    carries the loss accumulators, so one collective per step moves gradients AND loss."""
    if group is not None and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def broadcast_parameters(flat_params: torch.Tensor, src: int = 0, group=None) -> None:
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.broadcast(flat_params, src, group=group)


def allgather_packed_topk(packed: torch.Tensor, group=None) -> torch.Tensor:
    """(U, 2L) per rank (L fp32 scores + L int32 ids per user, L = max(k, 10): the scoring kernel's wire format)
    -> (G, U, 2L) on every rank with ONE all-gather."""
    G = dist.get_world_size(group)
    U, W = packed.shape
    out = torch.empty(G * U, W, dtype=packed.dtype, device=packed.device)      # (G * U, W): rank-major concatenation
    dist.all_gather_into_tensor(out, packed.contiguous(), group=group)
    return out.view(G, U, W)


def allgather_rows(rows: torch.Tensor, group=None) -> torch.Tensor:
    """(n, W) per rank (same n everywhere) -> (G * n, W) on every rank, rank-major: the user-sharded encode's exchange."""
    G = dist.get_world_size(group)
    n, W = rows.shape
    out = torch.empty(G * n, W, dtype=rows.dtype, device=rows.device)
    dist.all_gather_into_tensor(out, rows.contiguous(), group=group)
    return out


def merge_packed_topk_host(gathered: torch.Tensor, k: int = 10):
    """Host restatement of srfrd_merge_topk_packed (tie-break: score desc, id asc) for the CPU protocol tests.
    gathered: (G, U, 2L) wire rows of any list length L; returns the best k of the G * L entries per user."""
    import numpy as np
    g = gathered.cpu().numpy()
    G, U, W = g.shape
    sc = g[:, :, :W // 2].transpose(1, 0, 2).reshape(U, -1)
    ids = g[:, :, W // 2:].view(np.int32).transpose(1, 0, 2).reshape(U, -1).astype(np.int64)
    sc = np.where(ids < 0, -np.inf, sc)
    order = np.lexsort((ids, -sc), axis=1)[:, :k]
    return np.take_along_axis(sc, order, 1), np.take_along_axis(ids, order, 1)
