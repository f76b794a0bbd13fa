#!/usr/bin/env python
"""Bit-level digests of the CUDA step with every extension on, for tests/test_cuda_instantiations.py (needs a GPU).

    LG_TILE_ENVS=24 python tests/instantiation_digest.py [scenario ...]

The launcher's switches (LG_TILE_ENVS, LG_PRE_TICKET, LG_PRE_DIRECT, LG_PDL) are read once per process, so every forced
setting runs in a process of its own and prints one JSON line per scenario: a sha256 per buffer group, the episode
statistics (step and episode), and the instantiations of the two fused kernels that ran (`launched`, parsed from torch.profiler).

Scenario "ext:<a|s>:<A>:<N>:<own|torch>:<route>": difficulty 4 with DR observation and action noise, per-episode DR
observation and action offsets, the keypoint term, the moving goal (integrated by the synthetic simulator), bf16
copies, the wrapper's fused clamps, success termination, episode statistics and per-term episode returns, 30 % forced
resets and 5 % forced goal resets, 4 steps after reset().  Routes:
  eager   VecTaskPython.step
  graph   GraphRunner with the device clock, captured and replayed (clamps off: the runner's buffers have none; env
          counts divisible by 4, so that every output slot is 16-byte aligned, and still ragged at every tile size)
  host    GraphRunner with the host clock, stepped eagerly through the same sequence as `graph`
  shards  two shards of N / 2 envs (world_size 2), outputs concatenated: equal to `eager` except ids and statistics
  fused / hooks   TrifingerEnv.step against IsaacEnvBase.step: no clamps, no action noise and no DR offsets (see config)
"""
import copy
import hashlib
import json
import os
import re
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

T = 4
SIGMA = {"robot_q": 0.01, "robot_u": 0.05, "object_q": 0.002, "object_q_des": 0.001, "command": 0.01}
BIAS = {"robot_q": 0.02, "robot_u": 0.1, "object_q": 0.005, "object_q_des": 0.003, "command": 0.03}
SUCCESS = {"success": {"activate": True, "bonus": 500.0, "position_tolerance": 0.05, "orientation_tolerance": 1.0}}
DEFAULT = ["ext:a:9:12343:own:eager", "ext:s:9:12343:own:eager", "ext:a:9:16381:own:eager", "ext:s:9:16381:own:eager",
           "ext:a:9:16384:own:eager", "ext:a:18:12343:own:eager", "ext:s:18:16381:own:eager",
           "ext:a:9:12343:torch:eager", "ext:s:18:16381:torch:eager",
           "ext:a:9:12344:own:graph", "ext:s:9:16376:own:graph", "ext:a:18:12344:own:graph",
           "ext:a:9:12344:own:host", "ext:s:9:16376:own:host", "ext:a:18:12344:own:host",
           "ext:a:9:8198:own:eager", "ext:a:9:8198:own:shards",
           "ext:a:9:12343:torch:fused", "ext:a:9:12343:torch:hooks"]


def kernel_args(name):
    """'lg::post_physics_kernel<(int)9, (bool)1, ...>' or '<9, true, ...>' -> ('post', (9, 1, ...)), else None."""
    m = re.search(r"lg::(post|pre)_physics_kernel<([^>]*)>", name)
    if not m:
        return None
    vals = []
    for a in m.group(2).split(","):
        a = re.sub(r"^\((int|bool)\)", "", a.strip())
        vals.append(1 if a == "true" else 0 if a == "false" else int(a))
    return m.group(1), tuple(vals)


def launched(fn):
    """Runs fn() under torch.profiler (CUDA activity) and returns {'post': {tuples}, 'pre': {tuples}}."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"post": set(), "pre": set()}
    for ev in prof.events():
        k = kernel_args(ev.name)
        if k:
            out[k[0]].add(k[1])
    return out


def config(N, asym, A, stream, action_noise=True):
    """`action_noise=False`: no action noise and no DR offsets, for the hook route.  It refuses the action noise and
    the action offsets, and its resets key their draws by an epoch of their own, so its offset rows differ."""
    from leibnizgym_b200.config import difficulty_config
    cfg = difficulty_config(4, N, asymmetric_obs=asym, seed=23, episode_length=3,
                            command_mode="torque" if A == 9 else "position_impedance",
                            termination_conditions=copy.deepcopy(SUCCESS),
                            goal_movement={"rotation": {"activate": True, "rate_magnitude": 0.5}})
    cfg["reward_terms"]["keypoint"] = {"activate": True, "weight": 1500, "scale": 30.0, "eps": 2.0}
    cfg["domain_randomization"] = {"activate": True, "action_noise_std": 0.03 if action_noise else 0.0,
                                   "obs_noise_std": dict(SIGMA), "obs_bias_std": dict(BIAS) if action_noise else {},
                                   "action_bias_std": 0.05 if action_noise else 0.0}
    cfg["episode_statistics"] = {"activate": True}
    cfg["episode_term_returns"] = {"activate": True}
    cfg["rng_stream"] = "philox" if stream == "own" else stream
    return cfg


def _sha(*tensors):
    h = hashlib.sha256()
    for t in tensors:
        if t is not None:
            h.update(t.detach().contiguous().view(torch.uint8).cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def groups(envs, obs=None, states=None):
    """sha256 per buffer group over one env or the shards of one (concatenated along the env axis: dim 0 of the
    [N, ...] buffers, dim 1 of the [7, N] term rewards)."""
    cat = lambda name: (torch.cat([getattr(e, name) for e in envs]) if getattr(envs[0], name) is not None  # noqa: E731
                        else None)
    out = {
        "obs": _sha(obs if obs is not None else cat("_obs_buf"), cat("_obs_clipped"), cat("_obs_bf16")),
        "states": _sha(states if states is not None else cat("_states_buf"), cat("_states_clipped"),
                       cat("_states_bf16")),
        "reward": _sha(cat("_reward_buf"), torch.cat([e._term_rewards for e in envs], dim=1).t().contiguous()),
        "flags": _sha(cat("_reset_buf"), cat("_goal_reset_buf"), cat("_successes")),
        "dones": _sha(cat("_dones")),
        "steps": _sha(cat("_steps_count_buf")),
        "goal": _sha(cat("_object_goal_poses_buf"), cat("_object_goal_movement_buf"), cat("_history")),
        "action": _sha(cat("_action_buf"), cat("_applied_torque")),
        "sim": _sha(torch.cat([e._sim.dof_state.reshape(e.num_instances, -1) for e in envs]),
                    torch.cat([e._sim.root_state.reshape(e.num_instances, -1) for e in envs])),
        "ids": _sha(*[torch.cat([e._reset_ids[: int(e._counts[0])], e._goal_reset_ids[: int(e._counts[1])]])
                      for e in envs]),
        "episodes": _sha(cat("_episode_return"), cat("_last_episode_return"), cat("_last_episode_length"),
                         cat("_last_episode_success"), cat("_episode_term_return"), cat("_last_episode_term_return")),
        "offsets": _sha(cat("_obs_bias"), cat("_action_bias")),
    }
    return out


def episode_stats(env):
    """The step's `_episode_stats` and `_episode_term_stats` (fp64 sums of the CTAs' fixed-point parts)."""
    return env._episode_stats.tolist() + env._episode_term_stats.tolist()


def run(name):
    from leibnizgym_b200.env import IsaacEnvBase, TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import StateSequence, bernoulli_masks, make_sequence
    from leibnizgym_b200.wrappers import VecTaskPython
    _, sa, sA, sN, stream, route = name.split(":")
    asym, A, N = sa == "a", int(sA), int(sN)
    cfg = config(N, asym, A, stream, action_noise=route not in ("fused", "hooks"))
    dev = "cuda:0"
    seq = make_sequence(40 + A, T + 1, N, action_dim=A)
    rm, gm = bernoulli_masks(41, T + 1, N, 0.3, device=dev), bernoulli_masks(42, T + 1, N, 0.05, device=dev)
    kernels = {"post": set(), "pre": set()}

    def note(k):
        for key in kernels:
            kernels[key] |= k[key]

    def make_env(sq, rank=0, world=1):
        sim = SyntheticSim(sq.to(dev), dev)
        env = TrifingerEnv(cfg, device=dev, verbose=False, sim=sim, rank=rank, world_size=world)
        sim.enable_goal_integration(env._P, 0.02)
        env.enable_term_rewards(True)
        return env

    if route in ("graph", "host"):
        ring = make_sequence(40 + A, T, N, device=dev, action_dim=A)
        env = TrifingerEnv(cfg, device=dev, verbose=False, sim=SyntheticSim(ring, dev))
        env.enable_bf16_outputs()
        env.enable_term_rewards(True)
        env.reset()
        runner = GraphRunner(env, ring, rotate_outputs=True, inject_reset_masks=rm[:T], inject_goal_masks=gm[:T],
                             device_clock=route == "graph")
        if route == "graph":   # no profiler around a capture: `host` runs (and records) the same instantiations
            runner.capture(T)
            runner.replay()
        else:   # the same launches as capture() + replay(): two warm-up steps, then ring slots 0 .. T-1 again
            note(launched(lambda: runner.step_eager(2)))
            runner.t, runner.t0 = 0, -2
            runner.step_eager(T)
        torch.cuda.synchronize()
        return groups([env], runner.obs_slots, runner.state_slots), env._step_stats.tolist(), episode_stats(env), kernels

    world = 2 if route == "shards" else 1
    n = N // world
    envs, vecs = [], []
    for r in range(world):
        lo, hi = r * n, (r + 1) * n
        sq = StateSequence(*(x.contiguous() for x in (seq.dof_state[:, lo:hi], seq.root_state[:, 4 * lo:4 * hi],
                                                      seq.rigid_body[:, lo:hi], seq.dof_force[:, lo:hi],
                                                      seq.ft_sensors[:, lo:hi], seq.action[:, lo:hi])))
        env = make_env(sq, r, world)
        envs.append(env)
        if route in ("fused", "hooks"):
            env.enable_bf16_outputs()
            vecs.append(None)
        else:
            vecs.append(VecTaskPython(env, rl_device=dev, clip_obs=5.0, clip_actions=1.0, obs_dtype=torch.bfloat16))
    for env, vec in zip(envs, vecs):
        note(launched(vec.reset if vec is not None else env.reset))
    for t in range(1, T + 1):
        for r, (env, vec) in enumerate(zip(envs, vecs)):
            act = seq.action[t, r * n:(r + 1) * n].to(dev)
            if route == "hooks":
                env._reset_buf |= rm[t]
                env._goal_reset_buf |= gm[t]
                IsaacEnvBase.step(env, act)
                continue
            env.set_forced_resets(rm[t, r * n:(r + 1) * n].contiguous(), gm[t, r * n:(r + 1) * n].contiguous())
            step = (lambda: vec.step(act)) if vec is not None else (lambda: env.step(act))
            if t == 1:
                note(launched(step))
            else:
                step()
    torch.cuda.synchronize()
    stats = [e._step_stats.tolist() for e in envs]
    episodes = [episode_stats(e) for e in envs]
    return groups(envs), stats[0] if world == 1 else stats, episodes[0] if world == 1 else episodes, kernels


def main(argv):
    for name in argv or DEFAULT:
        digests, stats, episodes, kernels = run(name)
        print(json.dumps({"scenario": name, "digests": digests, "stats": stats, "episode_stats": episodes,
                          "launched": {k: sorted(v) for k, v in kernels.items()}}), flush=True)


if __name__ == "__main__":
    main(sys.argv[1:])
