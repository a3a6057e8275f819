"""Multi-GPU plumbing of the rollout: episodes are independent, so every rank owns its own
episodes, weight replica and random stream and there is NO data-path collective (the reference
already runs its environments in separate processes, l_dgn.py:137).  torch.distributed is only
used to agree on the timing (max over ranks) and to add up the work (sum over ranks)."""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def rank_seed_range(base_seed: int, rank: int, pool_count: int):
    """Env seeds of rank ``rank``'s reset-tuple pool: ``base_seed + rank*pool_count + k`` for k in [0, pool_count).
    The reference seeds vector env i with ``seed + i`` (tianshou ``venv.seed``); here the global env index runs over
    all ranks, so the pools of different ranks are disjoint by construction (no rank replays another rank's episodes).
    -> (first_seed, first_global_index)"""
    first = int(rank) * int(pool_count)
    return int(base_seed) + first, first


def rank_slot_offset(rank: int, episodes_per_rank: int) -> int:
    """``slot_offset`` of rank ``rank``'s :class:`melissa_b200.batched_env.EpisodeStream`: ``rank * episodes_per_rank``.
    The device episode stream is keyed by the global slot (episode index + slot_offset), so ranks of equal batch size
    that share a seed draw disjoint episode sequences, as :func:`rank_seed_range` gives disjoint pools."""
    return int(rank) * int(episodes_per_rank)


def shard_tuples(arrays, rank: int, episodes_per_rank: int, world: int = 1):
    """Slice of a SHARED reset-tuple pool owned by ``rank``: rows [rank*P, (rank+1)*P) with
    P = len(pool) // world >= episodes_per_rank.  Raises when the pool is too small for disjoint slices."""
    n = len(arrays[0])
    per = n // max(1, int(world))
    if per < episodes_per_rank:
        raise ValueError(f"reset-tuple pool of {n} rows cannot give {world} ranks {episodes_per_rank} disjoint episodes each")
    return tuple(a[rank * per:(rank + 1) * per] for a in arrays)


def reduce_job(ms: float, units: float, device=None):
    """-> (max over ranks of ms, sum over ranks of units).  Works on gloo (CPU) and nccl."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return float(ms), float(units)
    t = torch.tensor([float(ms)], dtype=torch.float64, device=device)
    u = torch.tensor([float(units)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(u, op=dist.ReduceOp.SUM)
    return float(t.item()), float(u.item())


def whole_job_throughput(ms: float, units: float, device=None) -> float:
    """units per second of the whole job: all ranks' units / the slowest rank's time."""
    ms_max, total = reduce_job(ms, units, device)
    return total / (ms_max / 1e3) if ms_max > 0 else 0.0
