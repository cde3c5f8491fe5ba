"""Multi-GPU plumbing: envs shard across ranks with no data-path collective (SURVEY.md section 8e).

One process per GPU (torchrun); rank r owns a contiguous slice of the global env index range; the only
exchange is a sum all-reduce of the 72-double episode-info vector (and, when a trainer logs it, of the int64
exploration-map sum), once per rollout, over NCCL on GPUs (gloo in the CPU tests).  Timing of multi-rank runs is
the max over ranks.
"""
from __future__ import annotations

from typing import Tuple


def shard_range(n_total: int, rank: int, world: int) -> Tuple[int, int]:
    """[start, stop) of the global env ids owned by `rank` (contiguous, sizes differ by at most one)."""
    if not (0 <= rank < world) or n_total < 0:
        raise ValueError("bad shard arguments")
    base, extra = divmod(n_total, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def all_reduce_info(info_sum, group=None):
    """In-place sum of the per-rank info vectors (slot 0 = env count).  No-op without a process group.

    Any dtype: the int64 [444, 436] exploration-map sum (VecEnvironment.exploration_map_sum) goes through the same call,
    1.5 MB per all-reduce, and stays exact; so do the int64 [130] event-flag counts (VecEnvironment.event_counts)."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(info_sum, op=dist.ReduceOp.SUM, group=group)
    return info_sum


def max_over_ranks(seconds: float, device=None, group=None) -> float:
    """Wall/device time of a multi-rank run = max over ranks."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return float(seconds)
    t = torch.tensor([seconds], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())
