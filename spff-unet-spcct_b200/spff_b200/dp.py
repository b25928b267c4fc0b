"""Data-parallel plumbing of the hot path (one process per GPU, torch.distributed).

The reference trains on one device with the DDP strategy lines commented out (train.py:1486-1503);
what DDP would do for this graph is: every rank computes the gradient of ITS batch-mean loss, the
gradients are averaged across ranks, every rank applies the same optimizer step. Here that is one
all-reduce (sum) over the flat fp32 gradient buffer with the 1/world factor folded into the Adam
kernel. Works with any backend (NCCL on the GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.distributed as dist


def world() -> Tuple[int, int]:
    """(rank, world_size); (0, 1) when torch.distributed is not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def allreduce_grads(flat_grad: torch.Tensor) -> float:
    """Sum the flat gradient buffer over ranks in place (ONE collective); returns the scale (1/world)
    the optimizer must apply so that the step uses the mean of the rank gradients."""
    _, n = world()
    if n > 1:
        dist.all_reduce(flat_grad, op=dist.ReduceOp.SUM)
    return 1.0 / n


def allreduce_async(flat_grad_range: torch.Tensor):
    """Start the sum all-reduce of one contiguous range of the flat gradient buffer and return the work
    handle (wait() before the optimizer). With NCCL the collective runs on its own stream after the
    kernels already enqueued, i.e. concurrently with whatever the compute stream is given next."""
    return dist.all_reduce(flat_grad_range, op=dist.ReduceOp.SUM, async_op=True)


def allreduce_tally(nll: torch.Tensor, count: torch.Tensor, confusion: torch.Tensor) -> None:
    """Global loss statistics for logging (≈ 1.4 KB): sum of nll, valid voxels, confusion tally."""
    _, n = world()
    if n > 1:
        for t in (nll, count, confusion):
            dist.all_reduce(t, op=dist.ReduceOp.SUM)


def allreduce_hist(hist: torch.Tensor) -> None:
    """Sum the softmax histograms of the evaluation step ([K,2,T] int64) over ranks in place, so that every rank
    derives the same ROC / PR curves."""
    _, n = world()
    if n > 1:
        dist.all_reduce(hist, op=dist.ReduceOp.SUM)


def allreduce_calibration(calib: torch.Tensor, brier: torch.Tensor, unc: torch.Tensor) -> None:
    """Sum the ensemble's calibration statistics over ranks in place: the [3,T] int64 confidence histogram, the fp64
    Brier sum and the int64 [2] uncertainty sums (fixed point, so the sum does not depend on the rank order)."""
    _, n = world()
    if n > 1:
        for t in (calib, brier, unc):
            dist.all_reduce(t, op=dist.ReduceOp.SUM)


def allreduce_temp_fit(sums: torch.Tensor, counted: torch.Tensor) -> None:
    """Sum the temperature-fit statistics over ranks in place: the fp64 [2,G] sums of the tempered nll and its derivative
    and the int64 [1] count of their voxels (one all-reduce: the count travels as the fp64 value it is, exact below
    2^53), so every rank solves for the same temperature."""
    _, n = world()
    if n > 1:
        buf = torch.cat([sums.reshape(-1), counted.to(torch.float64)])
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        sums.copy_(buf[:-1].view_as(sums))
        counted.copy_(buf[-1:].to(torch.int64))


def shard_range(total: int, rank: int | None = None, world_size: int | None = None) -> Tuple[int, int]:
    """[lo, hi) of the `total` independent units (slices / sliding-window tiles = whole z-slices)
    owned by `rank`: contiguous, sizes differ by at most one. No collective is involved."""
    if rank is None or world_size is None:
        rank, world_size = world()
    base, rem = divmod(total, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


# Optional measurement of the all-reduce time that is NOT hidden behind the backward: CUDA events on the compute stream
# around "backward enqueued" -> "every range reduced" (bench.py sets EXPOSED = [] and reads the event pairs).
EXPOSED = None


def exposed_timer_start():
    if EXPOSED is None:
        return None
    e0 = torch.cuda.Event(enable_timing=True)
    e0.record()
    return e0


def exposed_timer_stop(e0) -> None:
    if e0 is None:
        return
    e1 = torch.cuda.Event(enable_timing=True)
    e1.record()
    EXPOSED.append((e0, e1))
