"""Multi-GPU sharding of an environment batch: one process per GPU, no collective on the step path.

Environments are independent (the reference has exactly one per process), so a global batch of
``n_total`` envs is cut into contiguous slices, one per rank.  The Philox counter of an env is its
GLOBAL id (``env_id_base + n``), so every trajectory is independent of how many GPUs share the
batch.  The only communication is an optional all-gather of episode statistics (a few int64 per
rank) over ``torch.distributed`` -- NCCL for CUDA tensors on the 8xB200 NVSwitch box, gloo in the
CPU tests -- and it is never inside the timed step loop.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

STAT_KEYS = ("env_steps", "episodes", "deaths", "contained", "burnouts", "ticks")


def shard_range(n_total: int, world_size: int, rank: int) -> Tuple[int, int]:
    """(first global env id, number of envs) of ``rank``: contiguous, sizes differ by at most one."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(n_total, world_size)
    count = base + (1 if rank < rem else 0)
    start = rank * base + min(rank, rem)
    return start, count


def dist_info() -> Tuple[int, int]:
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def gather_stats(local: Dict[str, int], device: Optional[torch.device] = None) -> Dict[str, object]:
    """All-gather the per-rank episode statistics; returns per-rank lists and the totals."""
    import torch.distributed as dist
    rank, world = dist_info()
    t = torch.tensor([int(local.get(k, 0)) for k in STAT_KEYS], dtype=torch.int64, device=device or "cpu")
    if world > 1:
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t)
    else:
        out = [t]
    per_rank = [{k: int(v[i]) for i, k in enumerate(STAT_KEYS)} for v in out]
    total = {k: sum(p[k] for p in per_rank) for k in STAT_KEYS}
    return {"per_rank": per_rank, "total": total, "world_size": world}


class ShardedForestFire:
    """This rank's slice of a global batch of ``n_total`` environments (one CUDA device per rank)."""

    def __init__(self, n_total: int, device=None, obs_dtype=torch.uint8, **metadata):
        from .batched import BatchedForestFire
        self.rank, self.world_size = dist_info()
        self.n_total = int(n_total)
        self.env_id_base, self.n_local = shard_range(self.n_total, self.world_size, self.rank)
        if self.n_local < 1:
            raise ValueError("more ranks than environments")
        metadata = dict(metadata)
        metadata["env_id_base"] = int(metadata.get("env_id_base", 0)) + self.env_id_base
        self.local = BatchedForestFire(self.n_local, device=device, obs_dtype=obs_dtype, **metadata)

    def __getattr__(self, name):  # reset / step / rollout / get_state ... act on the local slice
        return getattr(self.local, name)

    def global_stats(self):
        return gather_stats(self.local.stats(), device=self.local.device)
