"""Multi-GPU plumbing: environments shard across ranks with no data-path collective; the exchanges are one
all-reduce of the episode-statistics vector (the columns of the reference's DataLogger row, data_logger.py:55-68,
summed over envs) per rollout / report and, under FleetVecNormalize, one all-reduce of its batch-moments vector per
step.  torch.distributed over NCCL on GPUs (gloo in the CPU tests)."""
import os

import torch

try:
    import torch.distributed as dist
except Exception:  # pragma: no cover
    dist = None


def world():
    """(rank, world_size, local_rank) from torchrun's environment; (0, 1, 0) when not launched distributed."""
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def shard_range(total_envs: int, rank: int, world_size: int):
    """Contiguous env range [lo, hi) of `rank`: ranks 0..r-1 get one extra env when total % world != 0."""
    if not (0 <= rank < world_size) or total_envs < 0:
        raise ValueError("bad rank / world_size / total_envs")
    base, rem = divmod(total_envs, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_reduce_stats(stats: torch.Tensor) -> torch.Tensor:
    """Sum the per-GPU partial statistics (float64 [FLEET_S__COUNT]) over all ranks, in place."""
    if dist is not None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats


def all_reduce_moments(moments: torch.Tensor) -> torch.Tensor:
    """Sum FleetVecNormalize's batch moments (float64 [2D+4], shifted sums about the running means every rank holds
    identically) over all ranks, in place, so that every rank merges the same global batch into its statistics."""
    return all_reduce_stats(moments)
