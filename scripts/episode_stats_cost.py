"""Cost of "episode_statistics" in CUDA-graph replay: bench.py's c2 (difficulty 2, 16 384 envs, no forced resets) and c5
(difficulty 4, 16 384 envs, 30 % of the envs reset per step) stepped by GraphRunner over a 32-slot ring, one graph of
128 steps per workload and variant, the variants' graphs replayed alternately in one process:
  a  default (the non-EXT post-physics instantiation)
  b  bf16 copies of obs / states on (the EXT instantiation, without episode statistics)
  c  b plus episode statistics
c - b is the cost of the feature itself (8 B/env-step more traffic: the running return read and written); a is the
baseline bench.py's c2 measures.  Prints the card's name and power limit with the numbers.
Usage: python scripts/episode_stats_cost.py [--replays 20] [--rounds 5]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

import bench  # noqa: E402  (workload definitions only)

VARIANTS = {"a": (False, False), "b": (True, False), "c": (True, True)}   # (bf16 outputs, episode statistics)


def make(wl_name, variant, R=32, C=128):
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence
    bf16, episodes = VARIANTS[variant]
    wl = bench.WORKLOADS[wl_name]
    N, dev = wl["envs"], "cuda:0"
    cfg = bench.workload_config(wl, N)
    cfg["episode_statistics"] = {"activate": episodes}
    ring = make_sequence(wl["seed"], R, N, device=dev)
    masks = bernoulli_masks(wl["seed"], R, N, wl["reset_p"], device=dev)
    env = TrifingerEnv(cfg, device=dev, verbose=False, sim=SyntheticSim(ring, dev))
    if bf16:
        env.enable_bf16_outputs()
    env.reset()
    runner = GraphRunner(env, ring, rotate_outputs=True, inject_reset_masks=masks)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        runner.capture(C)
        runner.replay(2)   # warm-up of the very graph that is timed
    torch.cuda.synchronize()
    return runner, s, C


def time_replays(runner, s, C, replays):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s):
        runner.replay(1)
        a.record()
        runner.replay(replays)
        b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / (replays * C)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {}
    for wl in ("c2", "c5"):
        runs = {v: make(wl, v) for v in VARIANTS}
        for _ in range(args.rounds):
            for v, (runner, s, C) in runs.items():
                res.setdefault(f"{wl}/{v}", []).append(round(time_replays(runner, s, C, args.replays), 2))
        del runs
        torch.cuda.empty_cache()
    med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
    diff = {wl: round(med[f"{wl}/c"] - med[f"{wl}/b"], 2) for wl in ("c2", "c5")}
    print(json.dumps({"gpu": smi, "us_per_step_graph_replay": res, "median": med, "median_c_minus_b": diff}))


if __name__ == "__main__":
    main()
