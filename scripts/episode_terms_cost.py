"""Cost of "episode_term_returns" in CUDA-graph replay: bench.py's c2 (difficulty 2, 16 384 envs, no forced resets) and c5
(difficulty 4, 16 384 envs, 30 % of the envs reset per step) stepped by GraphRunner over a 32-slot ring, one graph of
128 steps per workload and variant, the variants' graphs replayed alternately in one process:
  a  bf16 copies of obs / states on (the EXT instantiation, nothing else)
  b  a plus episode statistics
  c  b plus per-term episode returns
c - b is the cost of the feature itself (64 B/env-step more traffic: the 32-byte running row read and written).
Prints the card's name and power limit with the numbers.
Usage: python scripts/episode_terms_cost.py [--replays 20] [--rounds 5]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

import episode_stats_cost as base  # noqa: E402  (graph set-up and timing)

VARIANTS = {"a": (False, False), "b": (True, False), "c": (True, True)}   # (episode statistics, per-term returns)


def make(wl_name, variant, R=32, C=128):
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence
    episodes, terms = VARIANTS[variant]
    wl = base.bench.WORKLOADS[wl_name]
    N, dev = wl["envs"], "cuda:0"
    cfg = base.bench.workload_config(wl, N)
    cfg["episode_statistics"] = {"activate": episodes}
    cfg["episode_term_returns"] = {"activate": terms}
    ring = make_sequence(wl["seed"], R, N, device=dev)
    masks = bernoulli_masks(wl["seed"], R, N, wl["reset_p"], device=dev)
    env = TrifingerEnv(cfg, device=dev, verbose=False, sim=SyntheticSim(ring, dev))
    env.enable_bf16_outputs()
    env.reset()
    runner = GraphRunner(env, ring, rotate_outputs=True, inject_reset_masks=masks)
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
    for wl in ("c2", "c5"):
        runs = {v: make(wl, v) for v in VARIANTS}
        for _ in range(args.rounds):
            for v, (runner, s, C) in runs.items():
                res.setdefault(f"{wl}/{v}", []).append(round(base.time_replays(runner, s, C, args.replays), 2))
        del runs
        torch.cuda.empty_cache()
    med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
    diff = {wl: round(med[f"{wl}/c"] - med[f"{wl}/b"], 2) for wl in ("c2", "c5")}
    print(json.dumps({"gpu": smi, "us_per_step_graph_replay": res, "median": med, "median_c_minus_b": diff}))


if __name__ == "__main__":
    main()
