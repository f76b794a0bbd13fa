"""Torch restatement of the episode-statistics extension ("episode_statistics": {"activate": True}; no reference code).

The contract the kernels implement, in plain torch on the CPU:
  * every post-physics pass that computes rewards adds the env's final reward to its running return (fp32);
  * a reset of an env (timeout, forced or caller-set flag, `reset()`, `_reset_impl`; not a goal-only reset) with
    steps_count > 0 moves (return, steps_count, _successes) into the env's record and zeroes the return, then the
    counters are zeroed;
  * the first post-physics pass after such a reset sees steps_count == 0 with a record of length > 0 and reports the
    record once: episode_stats = (count, return sum, length sum, success count).
"""
from __future__ import annotations

from typing import List, Sequence

import torch


class EpisodeTracker:
    def __init__(self, n: int):
        self.episode_return = torch.zeros(n, dtype=torch.float32)
        self.last_episode_return = torch.zeros(n, dtype=torch.float32)
        self.last_episode_length = torch.zeros(n, dtype=torch.int64)
        self.last_episode_success = torch.zeros(n, dtype=torch.bool)
        self.steps = torch.zeros(n, dtype=torch.int64)
        self.successes = torch.zeros(n, dtype=torch.bool)

    def reset(self, ids) -> None:
        """The envs `ids` are reset (any route that ends an episode)."""
        ids = torch.as_tensor(ids, dtype=torch.int64).reshape(-1)
        ended = ids[self.steps[ids] > 0]
        self.last_episode_return[ended] = self.episode_return[ended]
        self.last_episode_length[ended] = self.steps[ended]
        self.last_episode_success[ended] = self.successes[ended]
        self.episode_return[ended] = 0.0
        self.steps[ids] = 0
        self.successes[ids] = False

    def post(self, reward: torch.Tensor, successes: torch.Tensor) -> torch.Tensor:
        """One post-physics pass with rewards: the step's final `reward` [N] and the `_successes` it left.  Returns
        this pass's episode_stats (float64 [4])."""
        self.episode_return = self.episode_return + reward.to(torch.float32)
        fresh = (self.steps == 0) & (self.last_episode_length > 0)
        stats = torch.tensor([float(fresh.sum()), float(self.last_episode_return[fresh].double().sum()),
                              float(self.last_episode_length[fresh].sum()),
                              float((self.last_episode_success & fresh).sum())], dtype=torch.float64)
        self.steps += 1
        self.successes = successes.to(torch.bool).clone()
        return stats


def episode_statistics(rewards: Sequence[torch.Tensor], reset_ids: Sequence, successes: Sequence[torch.Tensor]):
    """Fused steps t = 0..T-1 from a fresh env: `reset_ids[t]` are reset at the start of step t, then its post-physics
    pass produces `rewards[t]` and leaves `successes[t]`.  Returns (tracker after the last step, [episode_stats of
    every step])."""
    tr = EpisodeTracker(rewards[0].numel())
    stats: List[torch.Tensor] = []
    for r, ids, s in zip(rewards, reset_ids, successes):
        tr.reset(ids)
        stats.append(tr.post(r, s))
    return tr, stats
