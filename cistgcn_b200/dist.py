"""Batch-sharded evaluation over the GPUs of one box (SURVEY.md 8e).

Samples are independent in eval mode, so inference shards the batch by rank with NO data-path
collective: every rank (one process per GPU, launched by torchrun) runs the fused forward on its own
contiguous chunk.  The only exchange is the MPJPE bookkeeping: per-frame error sums (output_n doubles
= 200 bytes) are summed over ranks once per evaluation -- `torch.distributed.all_reduce`, which is NCCL
over NVLink on the GPU box and gloo in the CPU tests.  Grouped evaluation (one row per action or
sub-dataset, `sharded_eval_grouped`) exchanges G*T frame sums and G sample counts in one all-reduce.
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch
import torch.distributed as dist


def shard_bounds(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced partition of range(n): the first n % world ranks get one extra sample."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def combine_frame_sums(frame_sums: torch.Tensor, count: int, group=None) -> Tuple[torch.Tensor, int]:
    """Sum the per-frame error sums and the (sample x joint) counts over all ranks."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return frame_sums, count
    buf = torch.cat([frame_sums.to(torch.float64), frame_sums.new_tensor([float(count)], dtype=torch.float64)])
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return buf[:-1], int(round(float(buf[-1])))


def sharded_eval_mpjpe(forward_mpjpe: Callable, x: torch.Tensor, target: torch.Tensor, rank: Optional[int] = None,
                       world: Optional[int] = None, group=None):
    """Evaluate MPJPE of a global batch held by every rank: each rank processes only its shard.

    forward_mpjpe(x_shard, target_shard) -> (pred_shard, frame_sums) -- normally CISTGCN.forward_mpjpe.
    Returns (pred_shard, (lo, hi), mpjpe_all, mpjpe_per_frame) with the two MPJPE figures global, i.e.
    losses.mpjpe(..., reduce_axis=[]) and reduce_axis=(0, 2) of the whole batch."""
    if rank is None:
        rank = dist.get_rank(group) if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size(group) if dist.is_initialized() else 1
    lo, hi = shard_bounds(x.shape[0], rank, world)
    V, To = target.shape[2], target.shape[1]
    if hi > lo:
        pred, sums = forward_mpjpe(x[lo:hi].contiguous(), target[lo:hi].contiguous())
    else:
        pred, sums = target[lo:hi], torch.zeros(To, dtype=torch.float64, device=x.device)
    tot, cnt = combine_frame_sums(sums, (hi - lo) * V, group)
    per_frame = tot / max(cnt, 1)
    return pred, (lo, hi), per_frame.mean(), per_frame


def sharded_eval_grouped(fn: Callable, x: torch.Tensor, target: torch.Tensor, groups: torch.Tensor, n_groups: int,
                         rank: Optional[int] = None, world: Optional[int] = None, group=None):
    """Per-group per-frame MPJPE of a global batch held by every rank (e.g. one row per H3.6M action): each rank
    processes only its contiguous shard with the matching slice of `groups`.

    fn(x_shard, target_shard, groups_shard, n_groups) -> (pred_shard, sums (G, T), counts (G,)) -- normally
    CISTGCN.forward_mpjpe or CISTGCN.rollout_mpjpe.  The sums and counts of all ranks are combined in ONE all-reduce of
    G*T + G doubles.  Returns (pred_shard, (lo, hi), per_group_per_frame (G, T) float64, counts (G,) int64), where row g
    is losses.mpjpe(..., reduce_axis=(0, 2)) over group g's samples (NaN for a group without samples).  Raises
    ValueError when the global counts do not add up to the global batch (ids outside [0, n_groups))."""
    if rank is None:
        rank = dist.get_rank(group) if dist.is_initialized() else 0
    if world is None:
        world = dist.get_world_size(group) if dist.is_initialized() else 1
    B = x.shape[0]
    if not isinstance(groups, torch.Tensor) or groups.shape != (B,):
        raise ValueError("sharded_eval_grouped: groups must be a (B,) tensor of group ids")
    lo, hi = shard_bounds(B, rank, world)
    V, T = target.shape[2], target.shape[1]
    if hi > lo:
        pred, sums, counts = fn(x[lo:hi].contiguous(), target[lo:hi].contiguous(), groups[lo:hi], n_groups)
    else:
        pred = target[lo:hi]
        sums = torch.zeros(n_groups, T, dtype=torch.float64, device=x.device)
        counts = torch.zeros(n_groups, dtype=torch.int64, device=x.device)
    buf = torch.cat([sums.to(torch.float64).reshape(-1), counts.to(sums.device, torch.float64)])
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    tot = buf[:-n_groups].view(n_groups, T)
    cnt = buf[-n_groups:].round().to(torch.int64)
    n = int(cnt.sum())
    if n != B:
        raise ValueError(f"sharded_eval_grouped: the groups count {n} samples, the batch has {B} "
                         f"(group ids outside [0, {n_groups})?)")
    per = torch.where(cnt[:, None] > 0, tot / (cnt[:, None].to(torch.float64) * V).clamp(min=1), float("nan"))
    return pred, (lo, hi), per, cnt
