#!/usr/bin/env python
"""Benchmark of the TriFinger MDP hot path (reward + obs/states + reset), BASELINE.json metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c1|c2|c3|c4|c5] [--all-workloads] [--impl reference]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (N > 1, one rank per GPU)

A "step" is one pass of the hot path over all envs of the workload: lg_pre_physics (action store,
ordered reset compaction, reset / goal sampling, action->torque) + lg_post_physics (obs, states,
six reward terms, termination, counters, episode statistics).  PhysX is replaced by a ring of
synthetic simulator states resident in HBM (leibnizgym_b200/synthetic.py).

One JSON line is printed by rank 0:
  value      env-steps/s over all GPUs, inputs resident in HBM: after the warm-up, exactly K steps are
             replayed from CUDA graphs and timed with CUDA events (max over ranks) in steady state;
             value = K * envs / region time (`timing` also holds the cold-start figure).  The window is
             one sample: at small K it is short (K = 20 is ~0.2 ms at c2) and the figure is noisy, ~1 %
             from run to run; compare builds at K of about 2048 (the default)
  e2e        the same metric through the public API (VecTaskPython.step + get_state) with the
             simulator state and the action in pinned HOST memory and obs/states/reward/dones
             read back to the host every step
  roofline   dominant kernel (post_physics) alone: algorithmic bytes / measured launch duration
             against the measured HBM copy bandwidth of MEASURED_PEAKS.json
  cpu_baseline  the oracle port of the reference's torch CPU path on the host cores (N = 1 only)
`--impl reference` times that CPU path alone and prints the same line shape.

The inputs are generated from the workload's seed, so two runs with the same arguments execute the same steps on the
same data: `--dump-outputs DIR` writes what the last timed step computed, to compare two builds output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from leibnizgym_b200.config import difficulty_config, resolve_config  # noqa: E402
from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence  # noqa: E402

METRIC = "env-steps/sec reward+obs+reset"
UNIT = "env-steps/s"
FALLBACK_HBM_GBS = 6650.0

# BASELINE.json configs -> concrete runs (SURVEY.md §8d).  envs are PER GPU (weak scaling).
WORKLOADS = {
    # BASELINE.json configs[0] (SURVEY.md 8d C1): the reference's own CPU-runnable case
    "c1": dict(desc="trifinger_difficulty_1, asymmetric obs+states, 1024 envs/GPU", difficulty=1, envs=1024, asym=True,
               seed=1001, reset_p=0.0),
    "c1sym": dict(desc="trifinger_difficulty_1, symmetric obs only, 1024 envs/GPU", difficulty=1, envs=1024, asym=False,
                  seed=1001, reset_p=0.0),
    "c2": dict(desc="trifinger_difficulty_2, asymmetric obs+states, 16384 envs/GPU", difficulty=2, envs=16384,
               asym=True, seed=1002, reset_p=0.0),
    # SURVEY.md 8d C3: DR noise (extension, no reference code) + goal resampling forced on 5 % of the envs per step
    "c3": dict(desc="trifinger_difficulty_3, asymmetric, 65536 envs/GPU, DR obs/action noise (extension), goal "
                    "resampling forced on 5% of envs/step", difficulty=3, envs=65536, asym=True, seed=1003, reset_p=0.0,
               goal_p=0.05, dr=True),
    "c3ref": dict(desc="trifinger_difficulty_3, asymmetric, 65536 envs/GPU, goal resampling forced on 5% of envs/step "
                       "(reference features only)", difficulty=3, envs=65536, asym=True, seed=1003, reset_p=0.0, goal_p=0.05),
    "c3reset": dict(desc="trifinger_difficulty_3, asymmetric, 65536 envs/GPU, 5% forced resets/step", difficulty=3,
                    envs=65536, asym=True, seed=1003, reset_p=0.05),
    # SURVEY.md 8d C2: the keypoint pose reward is an extension term, reported separately from the headline
    "c2kp": dict(desc="trifinger_difficulty_2 + keypoint pose reward (extension), asymmetric, 16384 envs/GPU", difficulty=2,
                 envs=16384, asym=True, seed=1002, reset_p=0.0, keypoint=True),
    "c4": dict(desc="trifinger_difficulty_4, asymmetric obs+states, 32768 envs/GPU (262144 over 8)", difficulty=4,
               envs=32768, asym=True, seed=1004, reset_p=0.0),
    "c5": dict(desc="reset-heavy: difficulty 4, asymmetric, 16384 envs/GPU, 30% envs reset per step", difficulty=4,
               envs=16384, asym=True, seed=1005, reset_p=0.3),
    "c2sym": dict(desc="trifinger_difficulty_2, symmetric obs only, 16384 envs/GPU", difficulty=2, envs=16384,
                  asym=False, seed=1002, reset_p=0.0),
}

# one line per BASELINE.json config for --all-workloads (c3 with the reference's features only; the DR-noise and
# keypoint extensions have no reference implementation and stay out of every headline)
ALL_WORKLOADS = ("c1", "c1sym", "c2", "c3ref", "c4", "c5")


def workload_config(wl, num_envs, extensions=True):
    """Env config of a workload; `extensions=False` drops what the reference does not implement (CPU legs)."""
    over = {}
    if extensions and wl.get("dr"):
        over["domain_randomization"] = {"activate": True, "action_noise_std": 0.02,
                                        "obs_noise_std": {"robot_q": 0.005, "robot_u": 0.05, "object_q": 0.002,
                                                          "object_q_des": 0.0, "command": 0.0}}
    cfg = difficulty_config(wl["difficulty"], num_envs, asymmetric_obs=wl["asym"], seed=wl["seed"], **over)
    if extensions and wl.get("keypoint"):
        from leibnizgym_b200.config import KEYPOINT_TERM_DEFAULT
        cfg["reward_terms"]["keypoint"] = dict(KEYPOINT_TERM_DEFAULT, activate=True)
    return cfg


# algorithmic bytes per env-step (SURVEY.md §8d; derivation in DESIGN.md §5)
POST_BYTES = {True: 526 + 695, False: 298 + 243}
PRE_BYTES = 2 + 36 + 36 + 72 + 36          # flags, action in, action out, dof_state (safety damping), torque out
RESET_BYTES = 300                           # extra per resetting env


def measured_traffic(envs: int, asym: bool):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (or None)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)["post_physics_kernel"]
        if t["workload_envs"] == envs and bool(t["asymmetric"]) == bool(asym):
            return t["bytes_per_launch"]
    except Exception:
        pass
    return None


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled every few ms while the GPU is under load (NVML)."""

    def __init__(self, index: int, period_s: float = 0.004):
        self.index, self.period = index, period_s
        self.samples, self.reasons = [], set()
        self._stop = threading.Event()
        self._thread = None
        self.max_mhz = None
        self.enabled = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.enabled = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if mask & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.enabled and self._thread is None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join()
            self._thread = None

    def __enter__(self):
        self.start()
        return self

    def __exit__(self, *exc):
        self.stop()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


class NumaBinding:
    """Run the enclosed block on the CPUs NVML reports as local to the GPU, so that the pinned host buffers allocated
    inside it (first touch) and the thread issuing the copies sit on the GPU's NUMA node.  Matters when several ranks
    share a multi-socket host: without it a rank's staging memory can land on the far socket.  Restores the previous
    affinity on exit (the CPU baseline afterwards uses every core); a no-op when NVML or the mask is unavailable."""

    def __init__(self, gpu_index: int):
        self.gpu_index, self.prev, self.info = gpu_index, None, "unbound"

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
            self.prev = os.sched_getaffinity(0)
            use = (cpus & self.prev) or cpus
            if use and os.environ.get("LG_NO_NUMA_BIND") is None:
                os.sched_setaffinity(0, use)
                self.info = f"{len(use)} of {len(self.prev)} cpus local to gpu {self.gpu_index}"
        except Exception as ex:  # noqa: BLE001 - best effort
            self.info = f"unbound ({type(ex).__name__})"
        return self

    def __exit__(self, *exc):
        if self.prev is not None:
            try:
                os.sched_setaffinity(0, self.prev)
            except Exception:  # noqa: BLE001
                pass
        return False


# ------------------------------------------------------------------------------------------------
# CPU path (oracle port of the reference) — cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------------------
def time_cpu_path(wl: dict, envs: int, steps: int, warmup: int, max_seconds: float):
    """Times the hot path only (simulator playback excluded) of the oracle port on host cores."""
    from oracle.trifinger_oracle import OracleEnv, OracleSim

    class TimedSim(OracleSim):
        sim_seconds = 0.0

        def simulate(self):
            t0 = time.perf_counter()
            super().simulate()
            TimedSim.sim_seconds += time.perf_counter() - t0

    # all host cores, also under torchrun (which exports OMP_NUM_THREADS=1)
    torch.set_num_threads(int(os.environ.get("LG_CPU_THREADS", os.cpu_count() or 1)))
    cfg = resolve_config(workload_config(wl, envs, extensions=False))   # the reference has no DR noise / keypoint term
    T = 4
    seq = make_sequence(wl["seed"], T, envs)
    masks = bernoulli_masks(wl["seed"], T, envs, wl["reset_p"])
    gmasks = bernoulli_masks(wl["seed"] + 7, T, envs, wl.get("goal_p", 0.0))
    env = OracleEnv(cfg, TimedSim(seq, envs))
    env.reset()
    for t in range(warmup):
        env.step(seq.action[t % T])
    done = 0
    TimedSim.sim_seconds = 0.0
    t0 = time.perf_counter()
    while done < steps:
        if masks is not None:
            env.reset_buf |= masks[done % T]
        if gmasks is not None:
            env.goal_reset_buf |= gmasks[done % T]
        env.step(seq.action[done % T])
        done += 1
        if time.perf_counter() - t0 > max_seconds:
            break
    wall = time.perf_counter() - t0
    hot = wall - TimedSim.sim_seconds
    return dict(env_steps_per_s=done * envs / hot, ms_per_step=1e3 * hot / done, steps=done, envs=envs,
                cores=torch.get_num_threads())


def ring_slots(args, envs: int) -> int:
    """Distinct simulator states (and output slots) resident in HBM: enough that one pass over the ring moves several
    times the 126 MB L2, capped so that the largest workloads stay within a few GB."""
    if args.ring:
        return args.ring
    per_slot = envs * (1724 + 616)          # bytes of simulator state + obs/states outputs per env and slot
    return int(max(4, min(32, -(-(1280 << 20) // per_slot))))


def make_config(wl: dict, world: int, ring: int, ring_mib: float) -> dict:
    """The `config` object of the JSON line — the same dict from the B200 arm and from `--impl reference`."""
    N = wl["envs"]
    return {"workload": wl["desc"], "envs_per_gpu": N, "global_envs": N * world, "parallelism": f"dp{world}",
            "l2_policy": f"inputs larger than L2: ring of {ring} distinct simulator states ({ring_mib:.0f} MiB) and "
                         f"{ring} output slots per GPU",
            "reset_fraction_per_step": wl["reset_p"], "goal_reset_fraction_per_step": wl.get("goal_p", 0.0),
            "extensions": [k for k in ("dr", "keypoint") if wl.get(k)]}


def ring_mib_of(envs: int, ring: int) -> float:
    return ring * envs * 1464 / 2**20   # 18+52+260+9+18+9 floats of simulator state and action per env and slot


def run_reference(args, wl):
    """`--impl reference`: the reference's CPU implementation of the path (oracle port; the reference tree does not
    travel to the GPU box) on all host cores.  Same metric / unit / config as the B200 arm; every step is a bounded
    sample of the workload (at most the workload's envs per GPU — at N > 1 the CPU arm still runs ONE shard's envs,
    on rank 0 only; env-steps/s of a CPU path does not depend on how many GPUs the other arm uses)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    # bounded sample: each step covers a slice of the workload's envs so K steps end within ~1 min
    budget_env_steps = 4.0e7
    envs = int(min(wl["envs"], max(256, 2 ** int(math.log2(max(budget_env_steps / max(args.steps, 1), 256))))))
    r = time_cpu_path(wl, envs, args.steps, max(args.warmup, 3) if args.warmup < 16 else 16, max_seconds=150.0)
    sample = (f"{r['steps']} steps x {envs} envs per step (one shard of the workload: {wl['envs']} envs per GPU; the CPU arm "
              f"runs one shard at every N), oracle port of the reference's torch CPU path, {r['cores']} torch threads, "
              f"simulator playback excluded")
    R = ring_slots(args, wl["envs"])
    line = {
        "impl": "reference", "metric": METRIC, "value": r["env_steps_per_s"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(wl, world, R, ring_mib_of(wl["envs"], R)),
        "cpu_baseline": {"value": r["env_steps_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["env_steps_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def pctl(xs, q):
    xs = sorted(xs)
    if not xs:
        return None
    i = (len(xs) - 1) * q
    lo, hi = int(math.floor(i)), int(math.ceil(i))
    return xs[lo] + (xs[hi] - xs[lo]) * (i - lo)


class DeviceTimer:
    """Steady-state timing of replayed graphs with CUDA events, max over ranks.

    `steps` times the K steps of the workload once: barrier + synchronize | lead-in replays | event | the K-step region
    (+ the statistics all-reduce when sharded) | event | synchronize.  The lead-in keeps the GPU busy while the host
    enqueues the timed replays, so the events bracket K steps of a running pipeline, not the launch latency of the first
    graph of an idle stream nor a host-side stall; its first replay starts on an idle stream and is reported as the
    cold-start figure.  Exactly K steps are timed, so the steps a run executes, and with them its outputs, depend on the
    arguments only, never on how fast the device is.

    `run` times a single graph (one kernel alone) over repeats until `min_ms` of device time is covered; the result is
    every repeat's time, for the median and p10 / p90."""

    def __init__(self, world: int, dev: str):
        self.world, self.dev = world, dev

    def barrier(self):
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def agree(self, x: float, op="max") -> float:
        import torch.distributed as dist
        if self.world == 1:
            return x
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.MIN)
        return float(t.item())

    def once(self, region, lead_in=None) -> float:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        if lead_in is not None:
            lead_in()
        e0.record()
        region()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def steps(self, region, lead_in, lead_in_reps):
        """Returns (ms of the first lead-in replay, from an idle stream; region ms), each the max over ranks."""
        c0, c1, e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        self.barrier()
        c0.record()
        lead_in()
        c1.record()
        for _ in range(lead_in_reps - 1):
            lead_in()
        e0.record()
        region()
        e1.record()
        torch.cuda.synchronize()
        return self.agree(c0.elapsed_time(c1)), self.agree(e0.elapsed_time(e1))

    def run(self, region, lead_in, min_ms: float = 50.0, min_rep: int = 7, max_rep: int = 400):
        est = self.agree(self.once(region, lead_in))
        reps = int(max(min_rep, min(max_rep, math.ceil(min_ms / max(est, 1e-3)))))
        ms = [self.once(region, lead_in) for _ in range(reps)]
        if self.world > 1:
            import torch.distributed as dist
            t = torch.tensor(ms, device=self.dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)      # per repeat: the slowest rank
            ms = t.tolist()
        return ms


LEAD_IN_STEPS = 4096    # untimed steps right before the timed ones: ~40 ms of device time at 16384 envs


def measure_device(args, wl, rank, world, local_rank, sampler=None, dump_dir=None):
    """Device-resident throughput of one workload: K steps replayed from CUDA graphs over a ring of simulator states
    larger than L2, plus the two kernels alone.  Returns a dict of measurements (all times max over ranks).
    `dump_dir`: rank 0 writes what the last timed step computed there (dump_outputs)."""
    import torch.distributed as dist

    from leibnizgym_b200.distributed import stats_to_sums
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim

    dev = f"cuda:{local_rank}"
    N, K, W = wl["envs"], args.steps, max(args.warmup, 3)
    R = ring_slots(args, N)
    asym = wl["asym"]
    cfg = workload_config(wl, N * world)
    ring = make_sequence(wl["seed"], R, N, device=dev, first_env=rank * N)
    masks = bernoulli_masks(wl["seed"] + rank, R, N, wl["reset_p"], device=dev)
    gmasks = bernoulli_masks(wl["seed"] + 7 + rank, R, N, wl.get("goal_p", 0.0), device=dev)
    env = TrifingerEnv(cfg, device=dev, verbose=False, sim=SyntheticSim(ring, dev), rank=rank, world_size=world)
    env.reset()
    runner = GraphRunner(env, ring, rotate_outputs=True, inject_reset_masks=masks, inject_goal_masks=gmasks,
                         chain_pre=not getattr(args, "no_chain", False))
    timer = DeviceTimer(world, dev)
    stream = torch.cuda.Stream()
    side = torch.cuda.Stream() if world > 1 else None
    out = {}
    with torch.cuda.stream(stream):
        # ---- graphs: K <= 1024 steps are ONE graph; longer regions replay a 128-step graph q times + a tail --------
        if K <= 1024:
            C, q, rem = K, 1, 0
        else:
            C = R * max(1, 128 // R)
            q, rem = divmod(K, C)
        main_graph = runner.capture(C)
        tail_graph = runner.capture(rem) if rem else None
        reduced = []

        # shard sums = statistics vector x (local env count for the mean-type slots): one multiply per snapshot
        sum_weights = stats_to_sums(torch.ones_like(env._step_stats), N) if side is not None else None

        def region():
            # Episode statistics are the path's only collective (SURVEY.md 8e).  EVERY timed region carries one: the
            # shard sums of the step that just finished are snapshotted on the step stream and all-reduced over NCCL
            # on a side stream while the region's steps run — the way a logger consumes them, the steps never wait for
            # another rank — and the region is over only when that reduction has completed.
            if side is not None:
                side.wait_stream(stream)
                with torch.cuda.stream(side):
                    snap = env._step_stats * sum_weights
                    dist.all_reduce(snap, op=dist.ReduceOp.SUM)
                reduced[:] = [snap]
            for _ in range(q):
                main_graph.replay()
            if tail_graph is not None:
                tail_graph.replay()
            if side is not None:
                stream.wait_stream(side)

        def lead_in():
            main_graph.replay()

        # ---- warm-up: at least W steps of exactly what is timed (every graph of the region replayed) ---------------
        for _ in range(max(1, math.ceil(W / K))):
            region()
        timer.barrier()
        if sampler is not None:
            sampler.start()
        # The lead-in is counted in steps, so the steps before the timed ones are fixed too.  With a single replay
        # (0.2 ms at K = 20) a host-side stall, such as the clock sampler's thread starting, could leave the device idle
        # inside the timed region; LEAD_IN_STEPS of queued work absorb it.
        cold_ms, region_ms = timer.steps(region, lead_in, max(1, math.ceil(LEAD_IN_STEPS / C)))
        if dump_dir is not None and rank == 0:
            # every graph starts at ring slot 0: the last timed step wrote output slot (steps in the last graph - 1) % R
            slot = ((rem or C) - 1) % R
            per_env = {"obs": runner.obs_slots[slot], "reward": env._reward_buf, "dones": env._dones,
                       "reset": env._reset_buf, "applied_torque": env._applied_torque}
            if runner.state_slots is not None:
                per_env["states"] = runner.state_slots[slot]
            dump_outputs(dump_dir, per_env, {"step_stats": env._step_stats})
        # ---- the two kernels alone, back to back over the same ring (per-kernel roofline) --------------------------
        Ck = R * max(1, 128 // R)
        post_graph = runner.capture(Ck, post_only=True)
        post_graph.replay()
        post_ms = timer.run(post_graph.replay, post_graph.replay, min_ms=args.min_timed_ms, min_rep=9, max_rep=60)
        pre_graph = runner.capture(Ck, pre_only=True)
        pre_graph.replay()
        pre_ms = timer.run(pre_graph.replay, pre_graph.replay, min_ms=args.min_timed_ms / 2, min_rep=9, max_rep=60)
        # ---- what a plain device copy of the same number of bytes achieves at this size: R distinct source /
        # destination buffers of half the post kernel's algorithmic bytes each (read + write = the same traffic),
        # copied back to back from a graph like the kernels above.  The roofline peak is measured on a 4 GB copy; a
        # 20 MB launch is in the launch-latency regime for a memcpy too, and this is the honest yardstick for it.
        half = POST_BYTES[asym] * N // 2 // 4 * 4
        src = torch.empty((R, half // 4), device=dev, dtype=torch.float32).normal_()
        dst = torch.empty_like(src)
        for t in range(2):
            dst[t].copy_(src[t])
        torch.cuda.synchronize()
        copy_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(copy_graph):
            for t in range(Ck):
                dst[t % R].copy_(src[t % R])
        copy_graph.replay()
        copy_ms = timer.run(copy_graph.replay, copy_graph.replay, min_ms=args.min_timed_ms / 2, min_rep=9, max_rep=60)
        del src, dst
        if sampler is not None:
            sampler.stop()
        # ---- sharded statistics: the NCCL all-reduce against a gather + host sum of the same vectors ----------------
        if world > 1:
            torch.cuda.synchronize()
            mine = stats_to_sums(env._step_stats, N)    # what the next region snapshots and reduces
            region()
            torch.cuda.synchronize()
            parts = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(parts, mine)
            want = torch.stack(parts).cpu().sum(dim=0)
            got = reduced[0].cpu()
            err = float(((got - want).abs() / want.abs().clamp_min(1e-300)).max())
            count_slots = [7, 8, 11, 12]   # position / orientation goal counts, resets, dones: integers, exact in fp64
            counts_equal = bool(torch.equal(got[count_slots], want[count_slots]))
            out["stats_allreduce_check"] = {"max_rel_err_vs_gathered_sum": err, "count_slots_equal": counts_equal,
                                            "ok": bool(err < 1e-12 and counts_equal), "ranks": world}
            if not out["stats_allreduce_check"]["ok"]:
                raise RuntimeError(f"all-reduced statistics differ from the gathered per-rank sums: {out}")
    out.update(
        env=env, cfg=cfg, ring=R, ring_mib=ring.nbytes() / 2**20, steps_per_graph=C,
        region_ms=region_ms, us_per_step=1e3 * region_ms / K, cold_us_per_step=1e3 * cold_ms / C,
        post_us=1e3 * statistics.median(post_ms) / Ck, post_us_p10=1e3 * pctl(post_ms, 0.1) / Ck,
        post_us_p90=1e3 * pctl(post_ms, 0.9) / Ck, pre_us=1e3 * statistics.median(pre_ms) / Ck,
        copy_us=1e3 * statistics.median(copy_ms) / Ck,
        value=float(K) * N * world / (region_ms * 1e-3))
    return out


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, per_env, other):
    """Writes each device tensor as <out_dir>/<name>.npy: `per_env` ([N, ...], one row per env; booleans as 0 / 1) in
    float32, `other` in float64.  When the rows of everything would exceed DUMP_BYTES, a fixed seeded sample of envs is
    kept, the same rows of every array; env_index.npy lists them."""
    import numpy as np
    per_env = {k: v.cpu().numpy() for k, v in per_env.items()}
    other = {k: v.cpu().numpy().astype(np.float64) for k, v in other.items()}
    n = len(next(iter(per_env.values())))
    row_bytes = 8 + sum(4 * (a.size // n) for a in per_env.values())        # + env_index (float64)
    keep = min(n, (DUMP_BYTES - 4096 * (len(per_env) + len(other) + 1)     # .npy headers
                   - sum(a.nbytes for a in other.values())) // row_bytes)
    rows = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in per_env.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[rows].astype(np.float32))
    np.save(os.path.join(out_dir, "env_index.npy"), rows.astype(np.float64))
    for name, a in other.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def summarize_workload(wl, m):
    """Short record of one workload for `--all-workloads`."""
    asym = wl["asym"]
    N = wl["envs"]
    peak, _ = hbm_peak()
    post_gbs = POST_BYTES[asym] * N / (m["post_us"] * 1e-6) / 1e9
    step_bytes = (POST_BYTES[asym] + PRE_BYTES + (wl["reset_p"] + wl.get("goal_p", 0.0) / 3) * RESET_BYTES) * N
    return {"workload": wl["desc"], "envs_per_gpu": N, "value": m["value"], "us_per_step": m["us_per_step"],
            "post_us": m["post_us"], "pre_us": m["pre_us"],
            "post_frac_of_hbm_peak": post_gbs / peak,
            "whole_step_frac_of_hbm_peak": step_bytes / (m["us_per_step"] * 1e-6) / 1e9 / peak,
            "ring": m["ring"]}


def run_gpu(args, wl):
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        # The path's one collective moves 128 bytes: one NCCL CTA is plenty, and it leaves the SMs to the step kernels,
        # whose grids are sized to exactly one wave (2 GPUs, K = 20: 11.7 against 12.1 us/step with NCCL's default).
        os.environ.setdefault("NCCL_MAX_CTAS", "1")
        os.environ.setdefault("NCCL_MIN_CTAS", "1")
        dist.init_process_group("nccl", device_id=torch.device(dev))
    if args.l2_fetch:
        from leibnizgym_b200 import _native as nat
        nat.check(nat.load().lg_set_l2_fetch_granularity(args.l2_fetch), "lg_set_l2_fetch_granularity")
    N, K, W = wl["envs"], args.steps, max(args.warmup, 3)
    asym = wl["asym"]
    # clocks are sampled on rank 0 only (one NVML thread per box, 20 ms period), while the timed repeats run
    sampler = ClockSampler(physical_gpu_index(local_rank), period_s=0.02) if rank == 0 else None
    m = measure_device(args, wl, rank, world, local_rank, sampler, dump_dir=args.dump_outputs)
    m.pop("env")
    cfg = m.pop("cfg")
    clocks = sampler.summary() if sampler is not None else None

    # ---- end to end through the public API with host buffers (rank-local, then max over ranks) ----
    if args.no_e2e:
        e2e = None
    else:
        with NumaBinding(physical_gpu_index(local_rank)) as numa:
            e2e = run_e2e(args, wl, cfg, dev, rank, world)
        e2e["host_numa"] = numa.info

    peak, peak_src = hbm_peak()
    post_bytes = POST_BYTES[asym] * N
    post_us = m["post_us"]
    achieved = post_bytes / (post_us * 1e-6) / 1e9
    step_bytes = (POST_BYTES[asym] + PRE_BYTES + (wl["reset_p"] + wl.get("goal_p", 0.0) / 3) * RESET_BYTES) * N
    step_s = m["us_per_step"] * 1e-6
    config = make_config(wl, world, m["ring"], m["ring_mib"])
    line = {
        "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": m["us_per_step"] * 1e-3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config,
        "timing": {"method": f"CUDA events around the K steps, replayed from CUDA graphs once, after an untimed lead-in "
                             f"of >= {LEAD_IN_STEPS} steps (steady state); the max over ranks; value = K steps / region "
                             f"time; cold start = the first lead-in replay (steps_per_graph steps), from an idle stream",
                   "steps_per_graph": m["steps_per_graph"], "region_ms": m["region_ms"], "us_per_step": m["us_per_step"],
                   "cold_start_us_per_step": m["cold_us_per_step"],
                   "statistics_allreduce_in_region": world > 1,
                   "pre_launch": "stream order (lg_pre_physics)" if args.no_chain else
                                 "chained to the preceding post-physics pass (lg_pre_physics_chained: actions and joint "
                                 "states are resident in the ring long before they are used)"},
        "roofline": {"bound": "hbm", "kernel": "post_physics_kernel", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": achieved / peak, "traffic": measured_traffic(N, asym), "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": post_bytes, "launch_us": post_us,
                     "launch_us_p10": m["post_us_p10"], "launch_us_p90": m["post_us_p90"],
                     "pre_us": m["pre_us"], "pre_algorithmic_bytes_per_launch": PRE_BYTES * N,
                     "device_copy_same_bytes_us": m["copy_us"],
                     "device_copy_same_bytes_frac": post_bytes / (m["copy_us"] * 1e-6) / 1e9 / peak,
                     "step_us": m["us_per_step"], "whole_step_gbs": step_bytes / step_s / 1e9,
                     "whole_step_frac": step_bytes / step_s / 1e9 / peak},
        "clocks": clocks,
        "gpu_launches": 2 * K * world,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if "stats_allreduce_check" in m:
        line["stats_allreduce_check"] = m["stats_allreduce_check"]
    if args.all_workloads:
        per = {args.workload: summarize_workload(wl, m)}
        for name in ALL_WORKLOADS:
            if name == args.workload:
                continue
            w2 = dict(WORKLOADS[name])
            torch.cuda.empty_cache()
            m2 = measure_device(args, w2, rank, world, local_rank)
            m2.pop("env"), m2.pop("cfg")
            per[name] = summarize_workload(w2, m2)
        line["workloads"] = per
    if rank == 0 and world == 1 and not args.no_cpu:
        r = time_cpu_path(wl, N, steps=10_000, warmup=3, max_seconds=args.cpu_seconds)
        line["cpu_baseline"] = {
            "value": r["env_steps_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port",
            "sample": f"{r['steps']} steps x {N} envs (~{args.cpu_seconds:.0f} s), oracle port of the reference's torch CPU "
                      f"path, simulator playback excluded"}
        if args.all_workloads:   # BASELINE config 1 is the reference's own CPU-runnable case: time it on the CPU too
            for name in ("c1", "c1sym"):
                w1 = WORKLOADS[name]
                r1 = time_cpu_path(w1, w1["envs"], steps=10_000, warmup=3, max_seconds=min(args.cpu_seconds, 6.0))
                line["workloads"][name]["cpu_env_steps_per_s"] = r1["env_steps_per_s"]
                line["workloads"][name]["cpu_ms_per_step"] = r1["ms_per_step"]
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(args, wl, cfg, dev, rank, world):
    """Public-API step (VecTaskPython.step + get_state) with HOST-resident simulator state, action and
    results, every step.  Three transports (--e2e-mode):
      zc      zero copy: the simulator tensors and the action sit in pinned host memory and the
              fused kernels read the rows they need — and write obs/states/reward/dones — over PCIe themselves;
      zc_out  inputs staged by host->device copies of the five simulator tensors, results written to the host
              by the kernels;
      copy    (default) inputs staged by host->device copies (of root_state / rigid_body only the object and
              fingertip rows), results copied back with four device->host copies."""
    import torch.distributed as dist

    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import HostZeroCopySim, SyntheticSim
    from leibnizgym_b200.wrappers import VecTaskPython

    N = wl["envs"]
    T = 4
    mode = args.e2e_mode
    asym = wl["asym"]
    host = make_sequence(wl["seed"], T, N, first_env=rank * N).to("cpu", pin=True)
    sim = HostZeroCopySim(host) if mode == "zc" else SyntheticSim(host, dev)
    env = TrifingerEnv(cfg, device=dev, verbose=False, sim=sim, rank=rank, world_size=world)
    if mode != "zc" and not args.e2e_full_upload:
        sim.use_sparse_upload(env._P)
    chunks = args.e2e_chunks if mode == "copy" else 0
    vec = VecTaskPython(env, rl_device=dev if (mode == "copy" and not chunks) else "cpu", clip_obs=5.0, clip_actions=1.0,
                        host_pipeline_chunks=chunks)
    vec.reset()
    obs_dim, st_dim = env.get_obs_dim(), env.get_state_dim()
    if mode == "copy":
        pin = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt).pin_memory()  # noqa: E731
        h_obs, h_rew, h_done = pin(N, obs_dim), pin(N), pin(N, dt=torch.bool)
        h_states = pin(N, st_dim) if asym else None
    steps = max(8, min(args.e2e_steps, args.steps))
    sink = torch.zeros(1)

    def one(t):
        obs, rew, done, _ = vec.step(host.action[t % T])   # pinned host action
        states = vec.get_state() if asym else None
        if mode == "copy" and not chunks:
            h_obs.copy_(obs, non_blocking=True)
            h_rew.copy_(rew, non_blocking=True)
            h_done.copy_(done, non_blocking=True)
            if asym:
                h_states.copy_(states, non_blocking=True)
        torch.cuda.synchronize()                           # the caller consumes the results every step
        return obs if (mode != "copy" or chunks) else h_obs

    for t in range(3):
        one(t)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(steps):
        o = one(t)
    e1.record()
    torch.cuda.synchronize()
    sink += float(o[0, 0])                                 # the host really reads the result
    ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    # rows staged per env: everything with --e2e-full-upload, else the object actor's root row and the 3 fingertip bodies
    root_rows, body_rows = (4, 20) if args.e2e_full_upload else (1, 3)
    full_h2d = 4 * N * (18 + root_rows * 13 + body_rows * 13 + (9 + 18 if asym else 0) + 9)
    # zero copy: bytes the kernels fetch from host memory = the rows the path reads (dof_state twice: torque + obs)
    zc_h2d = 4 * N * (9 + 18 + 18 + 13 + 39 + (9 + 18 if asym else 0))
    shared_obs = bool(chunks) and vec._pipeline.shared_obs   # obs = first columns of the downloaded states
    d2h = 4 * N * ((0 if shared_obs else obs_dim) + st_dim + 1 + (0 if mode == "copy" else 9)) + N   # zero-copy modes also return the torque
    return {"value": steps * N * world / (ms * 1e-3), "unit": UNIT,
            "h2d_bytes_per_step": zc_h2d if mode == "zc" else full_h2d, "d2h_bytes_per_step": d2h,
            "steps": steps, "ms_per_step": ms / steps, "mode": mode, "pipeline_chunks": chunks, "obs_is_view_of_states": shared_obs,
            "api": "VecTaskPython.step + get_state; simulator state, action and results in pinned host memory"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2048)
    ap.add_argument("--warmup", type=int, default=256)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=None, help="override envs per GPU")
    ap.add_argument("--ring", type=int, default=0, help="distinct simulator states in HBM (0: sized to several times L2)")
    ap.add_argument("--all-workloads", action="store_true",
                    help="also measure one line per BASELINE.json config (c1, c1sym, c2, c3ref, c4, c5) into `workloads`")
    ap.add_argument("--min-timed-ms", type=float, default=20.0,
                    help="device time the kernel-alone roofline timings repeat for: the post-physics kernel this long, "
                         "the pre-physics kernel and the device copy half of it (the K timed steps are not repeated)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0's envs: obs, states, reward, dones, reset, "
                         "applied_torque, step_stats) as DIR/<name>.npy, float32 / float64; at most 64 MB, a seeded "
                         "sample of envs (env_index.npy) when larger")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-chain", action="store_true",
                    help="launch the pre-physics pass in stream order (lg_pre_physics) instead of chained to the preceding "
                         "post-physics pass (lg_pre_physics_chained)")
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--e2e-mode", default="copy", choices=["zc", "zc_out", "copy"])
    ap.add_argument("--e2e-chunks", type=int, default=1, help="env ranges of the host pipeline (0 = un-chunked copies)")
    ap.add_argument("--e2e-full-upload", action="store_true", help="upload all 20 rigid bodies, not just the fingertip run")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--l2-fetch", type=int, default=0, help="cudaLimitMaxL2FetchGranularity hint (32/64/128); 0 = leave")
    args = ap.parse_args()
    wl = dict(WORKLOADS[args.workload])
    if args.envs:
        wl["envs"] = args.envs
        wl["desc"] += f" [envs/GPU overridden to {args.envs}]"
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the outputs of the B200 path; it does not apply to --impl reference")
        run_reference(args, wl)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU path")
    run_gpu(args, wl)


if __name__ == "__main__":
    main()
