"""Torch restatement of the per-term episode returns ("episode_term_returns": {"activate": True}; no reference code).

The contract the kernels implement, in plain torch on the CPU.  A row has 8 slots: the 7 reward terms in LgTerm order,
then the success bonus.
  * every post-physics pass that computes rewards adds, in fp32, the env's value of each ACTIVE term k to slot k (the
    value the reward took, what `term_rewards` shows) and, where success termination fired, the fp32 bonus to slot 7;
    inactive terms leave their slot at 0;
  * a reset that ends an episode (any route, steps_count > 0, not a goal-only reset) moves the running row into the
    env's record and zeroes it;
  * the first post-physics pass after such a reset (steps_count == 0, a record of length > 0) adds the record into
    episode_term_stats, once.
"""
from __future__ import annotations

import torch

NUM_SLOTS = 8
BONUS = 7


class EpisodeTermTracker:
    def __init__(self, n: int, active_terms, bonus: float):
        """`active_terms`: 7 bools (LgTerm order); `bonus`: the success bonus of the config (rounded to fp32)."""
        self.active = [bool(a) for a in active_terms]
        assert len(self.active) == NUM_SLOTS - 1
        self.bonus = torch.tensor(bonus, dtype=torch.float32)
        self.episode_term_return = torch.zeros(n, NUM_SLOTS, dtype=torch.float32)
        self.last_episode_term_return = torch.zeros(n, NUM_SLOTS, dtype=torch.float32)
        self.last_episode_length = torch.zeros(n, dtype=torch.int64)
        self.steps = torch.zeros(n, dtype=torch.int64)

    def reset(self, ids) -> None:
        """The envs `ids` are reset (any route that ends an episode)."""
        ids = torch.as_tensor(ids, dtype=torch.int64).reshape(-1)
        ended = ids[self.steps[ids] > 0]
        self.last_episode_term_return[ended] = self.episode_term_return[ended]
        self.last_episode_length[ended] = self.steps[ended]
        self.episode_term_return[ended] = 0.0
        self.steps[ids] = 0

    def post(self, terms: torch.Tensor, bonus_paid: torch.Tensor):
        """One post-physics pass with rewards: the step's per-term values `terms` [7, N] and where the success bonus was
        paid [N].  Returns (count of records reported, this pass's episode_term_stats float64 [8])."""
        run = self.episode_term_return
        for k, on in enumerate(self.active):
            if on:
                run[:, k] = run[:, k] + terms[k].to(torch.float32)
        paid = bonus_paid.to(torch.bool)
        run[paid, BONUS] = run[paid, BONUS] + self.bonus
        fresh = (self.steps == 0) & (self.last_episode_length > 0)
        stats = self.last_episode_term_return[fresh].double().sum(0)
        self.steps += 1
        return int(fresh.sum()), stats


def slot_sum_bound(abs_total: torch.Tensor, length: torch.Tensor) -> torch.Tensor:
    """Bound on |sum of a record's 8 slots - its episode return|.  Both are fp32 recursive sums of the same addends
    (at most 8 per step over `length` steps) in different orders: the return adds them step by step (at most 8 * length
    roundings on its chain), the slots add them term by term (length roundings) and then the 8 slots (8 more).  Each
    rounding errs by at most 2^-24 of a partial sum, and every partial sum is at most `abs_total`, the sum of the
    absolute contributions."""
    return abs_total.double() * ((NUM_SLOTS * length.double() + length.double() + NUM_SLOTS) * 2.0 ** -24)
