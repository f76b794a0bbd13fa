"""Env sharding across the GPUs of one box and the path's only collective.

Envs are independent (SURVEY.md §8e): GPU g owns the contiguous block
[g*N/G, (g+1)*N/G) of global env indices, all buffers are local, and nothing crosses
GPUs on the data path.  The single exchange is the all-reduce of the 16-entry
episode-statistics vector (the reference's `_step_info` means and counts,
trifinger_env.py:554, :1067-1068, :1076, :1098-1099) when a caller wants job-wide
numbers: NCCL over NVLink on GPUs, gloo in the CPU tests.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import _native as nat

MEAN_SLOTS = tuple(range(7)) + (nat.STAT_SUCCESSES, nat.STAT_REWARD)


def shard_range(global_num_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """[first, last) global env indices owned by `rank`."""
    if global_num_envs % world_size != 0:
        raise ValueError("num_instances must be divisible by world_size")
    n = global_num_envs // world_size
    return rank * n, (rank + 1) * n


def stats_to_sums(step_stats: torch.Tensor, local_num_envs: int) -> torch.Tensor:
    """Shard statistics hold means for the mean-type slots and counts for the rest; sums add up
    across shards, means do not."""
    w = torch.ones_like(step_stats)
    w[list(MEAN_SLOTS)] = float(local_num_envs)
    return step_stats * w


def all_reduce_stats(step_stats: torch.Tensor, local_num_envs: int, global_num_envs: int,
                     group=None, episode_stats: Optional[torch.Tensor] = None,
                     episode_term_stats: Optional[torch.Tensor] = None):
    """Job-wide statistics vector in the same layout (means / counts) from every rank's shard vector.
    With `episode_stats` (a shard's LG_NUM_EPISODE_STATS sums) both go through one all-reduce and the result is the
    pair (statistics vector, job-wide episode sums).  With `episode_term_stats` too (a shard's LG_NUM_EPISODE_TERMS
    per-term return sums) all three go through the one all-reduce and the result is the triple (statistics vector,
    episode sums, per-term return sums)."""
    if episode_term_stats is not None and episode_stats is None:
        raise ValueError("episode_term_stats is reduced together with episode_stats")
    sums = stats_to_sums(step_stats.to(torch.float64), local_num_envs)
    n = sums.numel()
    if episode_stats is not None:
        sums = torch.cat([sums, episode_stats.to(device=sums.device, dtype=torch.float64)])
    if episode_term_stats is not None:
        sums = torch.cat([sums, episode_term_stats.to(device=sums.device, dtype=torch.float64)])
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.all_reduce(sums, op=torch.distributed.ReduceOp.SUM, group=group)
    w = torch.ones(n, dtype=sums.dtype, device=sums.device)
    w[list(MEAN_SLOTS)] = 1.0 / float(global_num_envs)
    if episode_stats is None:
        return sums * w
    m = n + nat.LG_NUM_EPISODE_STATS
    if episode_term_stats is None:
        return sums[:n] * w, sums[n:]
    return sums[:n] * w, sums[n:m], sums[m:]


def stats_to_info(stats: torch.Tensor, active_terms, episode_stats: Optional[torch.Tensor] = None,
                  episode_term_stats: Optional[torch.Tensor] = None, episode_terms=None) -> Dict[str, float]:
    """The reference's `_step_info` keys from a statistics vector.  With `episode_stats` (LgEpisodeStat sums) also
    env/episodes/{count, return_sum, length_sum, successes} and, when episodes ended, env/episodes/{mean_return,
    mean_length, success_rate}.  With `episode_term_stats` (per-term return sums, nat.EPISODE_TERM_NAMES order) also
    env/episodes/return_sum/<name> and, when episodes ended, env/episodes/mean_return/<name>, for the names in
    `episode_terms` (default: all eight)."""
    if episode_term_stats is not None and episode_stats is None:
        raise ValueError("episode_term_stats is reported together with episode_stats")
    v = stats.detach().cpu().tolist()
    out = {}
    for i, name in enumerate(nat.TERM_NAMES):
        if name in active_terms:
            out[f"env/rewards/{name}"] = v[i]
    out["env/current_position_goal/count"] = v[nat.STAT_POSITION_GOAL]
    out["env/current_orientation_goal/count"] = v[nat.STAT_ORIENTATION_GOAL]
    out["env/average_consecutive_success"] = v[nat.STAT_SUCCESSES]
    if episode_stats is not None:
        count, ret, length, succ = episode_stats.detach().cpu().tolist()
        out.update({"env/episodes/count": count, "env/episodes/return_sum": ret, "env/episodes/length_sum": length,
                    "env/episodes/successes": succ})
        if count > 0:
            out.update({"env/episodes/mean_return": ret / count, "env/episodes/mean_length": length / count,
                        "env/episodes/success_rate": succ / count})
        if episode_term_stats is not None:
            t = episode_term_stats.detach().cpu().tolist()
            for i, name in enumerate(nat.EPISODE_TERM_NAMES):
                if episode_terms is None or name in episode_terms:
                    out[f"env/episodes/return_sum/{name}"] = t[i]
                    if count > 0:
                        out[f"env/episodes/mean_return/{name}"] = t[i] / count
    return out
