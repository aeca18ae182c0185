"""Multi-GPU plumbing: env-axis sharding and the one collective on this path.

Envs are independent, so the step path has no communication: rank r owns the
contiguous global env ids ``[offset, offset + count)`` and passes ``offset`` as
``env_offset`` so the in-kernel Philox stream -- keyed by (seed, global env id,
step, mass) -- makes results independent of the number of ranks.  The only
collective is a SUM all-reduce of the 8-double episode-statistics vector
(NCCL on GPUs; gloo in the CPU tests), once per rollout, off the step stream.
"""
from __future__ import annotations

import os
from typing import Dict, Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(total_envs: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous split of ``total_envs`` over ``world`` ranks; the first
    ``total_envs % world`` ranks get one extra env.  Returns ``(offset, count)``."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, extra = divmod(int(total_envs), int(world))
    count = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return offset, count


def env_from_torchrun() -> Tuple[int, int, int]:
    """(rank, world_size, local_rank) from the torchrun environment (defaults: single process)."""
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")),
            int(os.environ.get("LOCAL_RANK", "0")))


def all_reduce_stats(vec: torch.Tensor) -> torch.Tensor:
    """SUM all-reduce of the stats vector [return, return^2, length, count, non-finite count, non-finite length, 0, 0]
    (float64)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        vec = vec.clone()
        dist.all_reduce(vec, op=dist.ReduceOp.SUM)
    return vec


def finalize_stats(vec, nonfinite: bool = False) -> Dict[str, float]:
    """Turn the (all-reduced) stats vector into mean / std / count.  ``nonfinite``: the env counts episodes with a
    non-finite return apart (``BatchedPhysicsEnv(nonfinite="count" | "end")``); the return statistics then cover the
    finite episodes, and ``nonfinite_episodes`` / ``nonfinite_length_mean`` describe the others."""
    s = [float(x) for x in (vec.tolist() if hasattr(vec, "tolist") else vec)]
    n = s[3]
    nan = float("nan")
    if n <= 0:
        out = {"episodes": 0, "return_mean": nan, "return_std": nan, "length_mean": nan,
               "return_sum": s[0], "return_sqsum": s[1], "length_sum": s[2]}
    else:
        mean = s[0] / n
        var = max(s[1] / n - mean * mean, 0.0)
        out = {"episodes": int(n), "return_mean": mean, "return_std": var ** 0.5, "length_mean": s[2] / n,
               "return_sum": s[0], "return_sqsum": s[1], "length_sum": s[2]}
    if nonfinite:
        out["nonfinite_episodes"] = int(s[4])
        out["nonfinite_length_mean"] = s[5] / s[4] if s[4] > 0 else nan
    return out


def make_sharded_env(creature, total_envs: int, *, device: Optional[torch.device] = None, **kwargs):
    """Build this rank's ``BatchedPhysicsEnv`` shard of a ``total_envs``-wide job."""
    from .batched import BatchedPhysicsEnv
    rank, world, local = env_from_torchrun()
    offset, count = shard_range(total_envs, rank, world)
    if device is None:
        device = torch.device("cuda", local)
    return BatchedPhysicsEnv(creature, count, device, env_offset=offset, **kwargs)
