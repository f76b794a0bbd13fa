"""Cost of the per-episode DR offsets ("domain_randomization": obs_bias_std / action_bias_std) in CUDA-graph replay,
stepped by GraphRunner over a 32-slot ring, one graph of 128 steps per workload and variant, the variants' graphs
replayed alternately in one process:
  c3  bench.py's c3 (difficulty 3, 65 536 envs, DR white noise on obs and action, goal resampling forced on 5 %)
        a  white noise only        b  a plus object-pose offsets        c  a plus offsets on every group and the action
  c5  bench.py's c5 (difficulty 4, 16 384 envs, 30 % of the envs reset per step) with c3's white noise
        a  white noise only        c  a plus offsets on every group and the action
Prints the card's name and power limit with the numbers.
Usage: python scripts/dr_bias_cost.py [--replays 20] [--rounds 5]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

import episode_stats_cost as base  # noqa: E402  (graph set-up and timing)

WHITE = {"activate": True, "action_noise_std": 0.02,
         "obs_noise_std": {"robot_q": 0.005, "robot_u": 0.05, "object_q": 0.002, "object_q_des": 0.0, "command": 0.0}}
OBJECT = {"obs_bias_std": {"object_q": 0.005}}
EVERY = {"obs_bias_std": {"robot_q": 0.01, "robot_u": 0.05, "object_q": 0.005, "object_q_des": 0.005, "command": 0.02},
         "action_bias_std": 0.02}
VARIANTS = {"c3": {"a": {}, "b": OBJECT, "c": EVERY}, "c5": {"a": {}, "c": EVERY}}


def make(wl_name, offsets, R=32, C=128):
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence
    wl = base.bench.WORKLOADS[wl_name]
    N, dev = wl["envs"], "cuda:0"
    cfg = base.bench.workload_config(wl, N)
    cfg["domain_randomization"] = dict(WHITE, **offsets)
    ring = make_sequence(wl["seed"], R, N, device=dev)
    masks = bernoulli_masks(wl["seed"], R, N, wl["reset_p"], device=dev)
    goal = bernoulli_masks(wl["seed"] + 7, R, N, wl.get("goal_p", 0.0), device=dev) if wl.get("goal_p") else None
    env = TrifingerEnv(cfg, device=dev, verbose=False, sim=SyntheticSim(ring, dev))
    env.reset()
    runner = GraphRunner(env, ring, rotate_outputs=True, inject_reset_masks=masks, inject_goal_masks=goal)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        runner.capture(C)
        runner.replay(2)   # warm-up of the very graph that is timed
    torch.cuda.synchronize()
    return runner, s, C


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {}
    for wl, variants in VARIANTS.items():
        runs = {v: make(wl, off) for v, off in variants.items()}
        for _ in range(args.rounds):
            for v, (runner, s, C) in runs.items():
                res.setdefault(f"{wl}/{v}", []).append(round(base.time_replays(runner, s, C, args.replays), 2))
        del runs
        torch.cuda.empty_cache()
    med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
    diff = {k: round(med[k] - med[k.split("/")[0] + "/a"], 2) for k in med if not k.endswith("/a")}
    print(json.dumps({"gpu": smi, "us_per_step_graph_replay": res, "median": med, "median_minus_a": diff}))


if __name__ == "__main__":
    main()
