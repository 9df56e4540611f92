"""The exchanges of a multi-GPU engine (SURVEY.md §8e), both one all-gather of a global-indexed per-set table over
NCCL / NVLink, rank-major:

* every sweep: each rank's per-set best (cbo_set_best: value f64, index i64, nan count i32: 24 bytes per set), followed on
  every rank by the same deterministic reduction (csrc/sweep.cu combine_kernel: larger value wins, ties to the lower grid
  index, then across sets the first set attaining the maximum, NaN = -inf);
* every off-grid refinement (SweepEngine.refine, opt-in): the refined maximum of each set its owner rank refined
  (cbo_refine_result: 56 bytes per set); every rank takes set g's record from the row of partition.refine_owners()[g].

No other data crosses GPUs: candidates are independent given the per-set state, which each rank rebuilds for the sets it
touches."""
from __future__ import annotations

import torch


def gather_set_bests(local_table: torch.Tensor, gathered: torch.Tensor, world: int, group=None) -> torch.Tensor:
    """local_table: uint8 tensor of one per-set record table (this rank's global-indexed table: S*24 bytes of
    cbo_set_best, -inf/-1 where it holds nothing, or S*56 bytes of cbo_refine_result); gathered: uint8 tensor of
    world * local_table.numel() bytes, filled rank-major (with world = 1 a copy).  Works with the nccl backend on device
    tensors and with gloo on CPU tensors (the world_size-2 CPU tests)."""
    import torch.distributed as dist
    if world == 1:
        gathered[:local_table.numel()].copy_(local_table)
        return gathered
    chunks = list(gathered.view(world, -1).unbind(0))
    dist.all_gather(chunks, local_table, group=group)
    return gathered
