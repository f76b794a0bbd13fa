"""One CUDA env and the CPU oracle in lockstep, with injected reset draws, every output checked after every step
(tests/test_cuda_instantiations.py, tests/test_cuda_fuzz.py).  Needs a GPU.

Extensions the harness can switch on: the fused clamps of VecTaskPython, bf16 copies, the keypoint term, the moving
goal integrated on both sides, episode statistics, per-term episode returns and the per-episode DR offsets.  The
offsets go into the oracle as inputs (oracle/extensions.OffsetOracleEnv), the way the episode restatements take the
kernel's own rewards: the action offset rows read before the step perturb the oracle's action, the obs offset rows the
step's resets drew perturb its actor observation.  White DR noise stays off.

Checks after every step (`Lockstep.check`):
  bit-exact   reset / goal-reset ids, actor-index lists, flags, successes, step counters, reset joint rows, `_dones`
              (the oracle's reset & goal_reset), `_history` (a copy of simulator data), `action_buf`, bf16 copies
              (of the kernel's own fp32 / clipped outputs), closed schedule gates (term exactly 0)
  tolerances  obs, states, clipped copies, goal pose / movement, applied torque, the six terms, the keypoint term,
              reward (tests/tolerances.py, the angle allowance, the integrator drift with the moving goal), `_step_info`
  trackers    episode buffers / `_episode_stats` (tests/episode_reference.py) and per-term rows / records /
              `_episode_term_stats` (tests/episode_term_reference.py), fed the kernel's own rewards, terms and ids
"""
import copy

import numpy as np
import torch

from episode_reference import EpisodeTracker
from test_cuda_edges import _check, _check_info, _np
from test_cuda_episode_terms import _Checker as TermChecker
from test_cuda_episodes import _check_against_tracker
from tolerances import angle_slack, compare

DEV = "cuda:0"
KEYPOINT = {"activate": True, "weight": 1500, "scale": 30.0, "eps": 2.0}
CLIP_OBS, CLIP_ACTIONS = 5.0, 1.0
TERM_NAMES = ("finger_reach_object_rate", "finger_move_penalty", "object_dist", "object_rot", "object_rot_delta",
              "object_move")   # LgTerm order, the rows of `term_rewards` and of the oracle's `last_terms`
# LgTerm index -> (term, schedule kind) of the terms a schedule can switch off
GATED = {0: ("finger_reach_object_rate", "thresh"), 2: ("object_dist", "thresh"), 3: ("object_rot", "thresh"),
         4: ("object_rot_delta", "linear")}


def rf_same(a, b):
    a, b = _np(a), _np(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def angle_allowance(ora, goal, dt):
    """Per-env allowance of the six terms and of the reward for the angle's asin (tests/tolerances.angle_slack), with
    the goal the rewards saw; a NaN angle (NaN terms on both sides) adds none."""
    cur = np.nan_to_num(angle_slack(ora.obj_hist[0][:, 3:7], goal[:, 3:7]), nan=0.0)
    prev = np.nan_to_num(angle_slack(ora.obj_hist[1][:, 3:7], goal[:, 3:7]), nan=0.0)
    t = ora.terms
    rot = abs(t["object_rot"]["weight"]) * dt / t["object_rot"]["scale"] * cur
    delta = abs(t["object_rot_delta"]["weight"]) * (cur + prev)
    terms = np.zeros((6, len(cur)))
    terms[3], terms[4] = rot, delta
    return terms, rot * t["object_rot"]["activate"] + delta * t["object_rot_delta"]["activate"]


class Lockstep:
    """`cfg`: a user config (num_instances included); `seq`: its StateSequence (goal rows already planted where the
    case plants them); `masks` / `goal_masks`: [T, N] bool forced resets per step (None: none); `draw_seed`: seed of
    the injected reset draws.  Keyword flags switch the extensions on; `obs_bias` maps observation groups to sigmas,
    `action_bias` is the action offset's sigma."""

    def __init__(self, cfg, seq, masks=None, goal_masks=None, draw_seed=0, *, clip=False, bf16=False, keypoint=False,
                 goal_integration=False, episode_statistics=False, episode_term_returns=False, obs_bias=None,
                 action_bias=0.0):
        from leibnizgym_b200.config import resolve_config
        from leibnizgym_b200.env import TrifingerEnv
        from leibnizgym_b200.params import obs_group_columns
        from leibnizgym_b200.sim import SyntheticSim
        from leibnizgym_b200.wrappers import VecTaskPython
        from oracle.extensions import OffsetOracleEnv, integrate_goal_rows
        from oracle.trifinger_oracle import OracleSim
        cfg = copy.deepcopy(cfg)
        N, A = int(cfg["num_instances"]), seq.action.shape[-1]
        assert not goal_integration or cfg["goal_movement"]["rotation"]["activate"], "goal integration needs the moving goal"
        assert not episode_term_returns or episode_statistics, "per-term returns need the episode statistics"
        self.N, self.seq, self.masks, self.goal_masks = N, seq, masks, goal_masks
        self.clip, self.keypoint, self.integrate = clip, keypoint, goal_integration
        if episode_statistics:
            cfg["episode_statistics"] = {"activate": True}
        if episode_term_returns:
            cfg["episode_term_returns"] = {"activate": True}
        if obs_bias or action_bias:
            cfg["domain_randomization"] = {"activate": True, "obs_bias_std": dict(obs_bias or {}),
                                           "action_bias_std": float(action_bias)}
        ora_cfg = resolve_config(copy.deepcopy(cfg))
        if keypoint:
            cfg["reward_terms"]["keypoint"] = dict(KEYPOINT)
        self.dt = float(ora_cfg["sim"]["dt"])
        sim = SyntheticSim(seq.to(DEV), DEV)
        self.env = env = TrifingerEnv(cfg, device=DEV, verbose=False, sim=sim)
        env.enable_term_rewards(True)
        if goal_integration:
            sim.enable_goal_integration(env._P, self.dt)
        self.vec = None
        if clip:
            self.vec = VecTaskPython(env, rl_device=DEV, clip_obs=CLIP_OBS, clip_actions=CLIP_ACTIONS,
                                     obs_dtype=torch.bfloat16 if bf16 else torch.float32)
        elif bf16:
            env.enable_bf16_outputs()
        dt = self.dt

        class IntegratingOracleSim(OracleSim):
            def simulate(self):
                keep = self.root.view(N, 4, 13)[:, 3].clone()
                super().simulate()
                self.root.view(N, 4, 13)[:, 3] = torch.from_numpy(integrate_goal_rows(keep.numpy(), dt).astype(np.float32))

        self.ora = ora = OffsetOracleEnv(ora_cfg, (IntegratingOracleSim if goal_integration else OracleSim)(seq, N))
        cols = obs_group_columns(A)
        ora.bias_cols = [c for g, s in (obs_bias or {}).items() if s for c in range(*cols[g])]
        # the goal pose the rewards see: the moving goal's update (after the termination check) replaces it
        check_termination = ora._check_termination

        def snapshot():
            self.goal_rewarded = ora.goal_poses.clone()
            check_termination()
        ora._check_termination = snapshot
        self.episodes = EpisodeTracker(N) if episode_statistics else None
        self.term_returns = TermChecker(env, env.config) if episode_term_returns else None
        self.g = torch.Generator().manual_seed(draw_seed)

    def _draws(self, k):
        return (torch.rand(k, 24, generator=self.g).numpy(), torch.randn(k, 8, generator=self.g).numpy()) if k else None

    def _obs_bias(self):
        self.ora.obs_bias = None if self.env.obs_bias is None else self.env.obs_bias.cpu()

    def reset(self):
        d = self._draws(self.N)
        self.env.inject_draws(reset=d)
        self.ora.inject_draws(reset=d)
        (self.vec.reset if self.vec is not None else self.env.reset)()
        self._obs_bias()
        self.ora.reset()
        if self.episodes is not None:
            self.episodes.reset(torch.arange(self.N))

    def step(self, t):
        """Step t of the sequence on both sides; returns (any reset, any goal reset)."""
        env, ora = self.env, self.ora
        m = None if self.masks is None else self.masks[t]
        gm = None if self.goal_masks is None else self.goal_masks[t]
        if m is not None:
            ora.reset_buf |= m
        if gm is not None:
            ora.goal_reset_buf |= gm
        env.set_forced_resets(None if m is None else m.to(DEV).contiguous(),
                              None if gm is None else gm.to(DEV).contiguous())
        dr, dg = self._draws(int(ora.reset_buf.sum())), self._draws(int(ora.goal_reset_buf.sum()))
        env.inject_draws(reset=dr, goal=dg)
        ora.inject_draws(reset=dr, goal=dg)
        act = self.seq.action[t]
        want = act.clone()
        if env.action_bias is not None:   # the rows read before the step; envs the step resets store 0 on both sides
            want = want + env.action_bias.cpu()
        if self.clip:
            want = torch.clamp(want, -CLIP_ACTIONS, CLIP_ACTIONS)
        (self.vec.step if self.vec is not None else env.step)(act.to(DEV))
        self._obs_bias()   # the rows the step's resets drew
        self.dones = ora.step(want)[2].clone()
        return dr is not None, dg is not None

    def check(self, t, reset, goal_reset, where):
        from oracle.extensions import keypoint_reward
        from oracle.trifinger_oracle import _gate, _ramp
        env, ora, N = self.env, self.ora, self.N
        w = (where, "step", t)
        torch.cuda.synchronize()
        # bit-exact: ids, actor-index lists, flags, counters, reset joint rows, dones, history
        _check("reset_ids", env.reset_env_ids, ora.last_ids[0], w)
        _check("goal_reset_ids", env.goal_reset_env_ids, ora.last_ids[1], w)
        k, kg = int(env._counts[0]), int(env._counts[1])
        if reset:
            _check("dof_index_list", env._robot_indices[:k], ora.index_lists["dof"], w)
            _check("root_index_list0", env._reset_root_indices[:3 * k], ora.index_lists["root_reset"], w)
        if goal_reset:
            _check("root_index_list1", env._goal_root_indices[:kg], ora.index_lists["root_goal"], w)
        for key, got, exp in (("reset_buf", env._reset_buf, ora.reset_buf), ("goal_reset_buf", env._goal_reset_buf,
                              ora.goal_reset_buf), ("successes", env._successes, ora.successes),
                              ("steps_count", env._steps_count_buf, ora.steps_count_buf)):
            _check(key, got, exp, w)
        assert np.array_equal(_np(env._dof_state).reshape(N, 18), ora.sim.dof.numpy().reshape(N, 18)), (w, "joint rows")
        assert torch.equal(env._dones.cpu(), self.dones), (w, "dones")
        hist = torch.cat([ora.tip_hist[0][:, :, 0:3].reshape(N, 9), ora.obj_hist[0][:, 0:7]], dim=1)
        assert rf_same(env._history, hist), (w, "history")
        # within the tolerances: outputs, action row, torque, terms, reward
        drift = 2e-6 if self.integrate else None       # the moving goal: fp32 integrator against the fp64 oracle
        _check("goal_pose", env._object_goal_poses_buf, ora.goal_poses, w, drift)
        _check("goal_movement", env._object_goal_movement_buf, ora.goal_movement, w)
        clip = lambda x: torch.clamp(x, -CLIP_OBS, CLIP_OBS)  # noqa: E731
        outs = [("obs", env.obs_buf, ora.obs_buf, env._obs_clipped, env._obs_bf16)]
        if env.config["asymmetric_obs"]:
            outs.append(("states", env.states_buf, ora.states_buf, env._states_clipped, env._states_bf16))
        for key, raw, want, clipped, bf16 in outs:
            _check(key, raw, want, w, drift)
            if self.clip:
                _check(key, clipped, clip(want), w + ("clipped",), drift)
            if bf16 is not None:
                src = clipped if self.clip else raw
                assert torch.equal(bf16.view(torch.int16), src.to(torch.bfloat16).view(torch.int16)), (w, key, "bf16")
        assert rf_same(env.action_buf, ora.action_buf), (w, "action_buf")
        _check("applied_torque", env._applied_torque, ora.applied_torque, w)
        slack_terms, slack_reward = angle_allowance(ora, self.goal_rewarded, self.dt)
        if self.integrate:   # goal quaternions up to 2e-6 apart (drift above): ~17x the 2 ulp of |v| the allowance assumes
            slack_terms, slack_reward = 20 * slack_terms, 20 * slack_reward
        terms = env._term_rewards
        _check("terms", terms[:6], ora.last_terms, w, slack_terms)
        T = ora.env_steps_count
        for i, (name, kind) in GATED.items():
            p = ora.terms[name]
            if (_gate if kind == "thresh" else _ramp)(p["start"], p["end"], T) == 0.0:
                assert bool((terms[i] == 0).all()), (w, "closed schedule", name, T)
        want = ora.reward_buf
        if self.keypoint:
            kp = keypoint_reward(KEYPOINT["weight"], self.dt, ora.obj_hist[0][:, 0:7], self.goal_rewarded,
                                 KEYPOINT["scale"], KEYPOINT["eps"])
            ok, detail = compare("terms", _np(terms[6]), kp.numpy(), extra_atol=2e-5 * np.abs(kp.numpy()))
            assert ok, (w, "keypoint", detail)
            want = want + kp
            slack_reward = slack_reward + 5e-4
        _check("reward", env.reward_buf, want, w, slack_reward)
        # a term's mean may differ by the mean of its per-env allowance (the goal drift's, with the moving goal)
        means = {f"env/rewards/{name}": float(slack_terms[i].mean()) for i, name in enumerate(TERM_NAMES)}
        _check_info(env._step_info, ora.step_info, w, means)
        # the episode restatements, fed the kernel's own rewards, terms, reset ids and flags
        if self.episodes is not None:
            self.episodes.reset(env.reset_env_ids.cpu())
            stats = self.episodes.post(env._reward_buf.cpu(), env._successes.cpu())
            _check_against_tracker(env, self.episodes, stats, w)
        if self.term_returns is not None:
            self.term_returns.step(w)

    def run(self, steps, where):
        """reset() then steps 1 .. steps - 1, each checked."""
        self.reset()
        for t in range(1, steps):
            self.check(t, *self.step(t), where)
