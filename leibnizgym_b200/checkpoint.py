"""Env-state checkpoint: everything the MDP carries from one step to the next, on disk.

The reference has no resume path for the environment (SURVEY.md §5; `dump_config`, ref
envs/env_base.py:295-309, only writes the config).  A run of this build can stop after any step
and continue bit-identically: the file holds the goal poses and movement, step counters, reset /
goal-reset / success flags, the one-deep history, the last action / outputs, the per-step
statistics (and, with "episode_statistics" on, the running returns and last-episode records; with
"episode_term_returns" on, their per-term rows too; with per-episode DR offsets on, each env's offsets), the device control block (RNG epoch of the kernel's Philox stream, frame counter,
compaction epoch) and the state of the torch CUDA stream (`rng_stream` "torch": seed, offset) — plus, for `SyntheticSim`, the simulator tensors and its clock, because the
pre-physics pass of the next step reads (and the resets wrote) simulator memory.

Format: one uncompressed `.npz`; `meta` is a JSON string (format version, shard geometry, config),
`env/<name>` and `sim/<name>` are the arrays.  Shards checkpoint independently (one file per rank).
"""
from __future__ import annotations

import json
import os
from typing import Dict

import numpy as np
import torch

from .params import dr_bias_sigmas

FORMAT_VERSION = 1

# name -> attribute of TrifingerEnv (device tensors, restored in place: the pointers the C ABI holds stay valid)
_ENV_TENSORS = {
    "obs": "_obs_buf", "states": "_states_buf", "obs_clipped": "_obs_clipped", "states_clipped": "_states_clipped",
    "action": "_action_buf", "reward": "_reward_buf", "reset": "_reset_buf", "goal_reset": "_goal_reset_buf",
    "successes": "_successes", "dones": "_dones", "steps_count": "_steps_count_buf",
    "goal_pose": "_object_goal_poses_buf", "goal_movement": "_object_goal_movement_buf", "history": "_history",
    "applied_torque": "_applied_torque", "step_stats": "_step_stats", "control": "_control",
    "scan_status": "_scan_status", "counts": "_counts", "reset_ids": "_reset_ids", "goal_reset_ids": "_goal_reset_ids",
    "reward_coef": "_reward_coef", "torch_rng": "_torch_rng",
    # episode statistics (absent when the extension is off)
    "episode_return": "_episode_return", "last_episode_return": "_last_episode_return",
    "last_episode_length": "_last_episode_length", "last_episode_success": "_last_episode_success",
    "episode_stats": "_episode_stats",
    # per-term episode returns (absent when that extension is off)
    "episode_term_return": "_episode_term_return", "last_episode_term_return": "_last_episode_term_return",
    "episode_term_stats": "_episode_term_stats",
    # per-episode DR offsets (each absent when its sigmas are all zero)
    "obs_bias": "_obs_bias", "action_bias": "_action_bias",
}
_SIM_TENSORS = ("dof_state", "root_state", "rigid_body", "dof_force", "ft_sensors")


def env_state_dict(env) -> Dict[str, object]:
    """Snapshot as host numpy arrays (synchronises the device)."""
    out: Dict[str, object] = {}
    for name, attr in _ENV_TENSORS.items():
        t = getattr(env, attr, None)
        if t is not None and t.numel():
            out[f"env/{name}"] = t.detach().cpu().numpy()
    sim = env._sim
    sim_meta = {"frame_count": int(sim.get_frame_count()), "cursor": int(getattr(sim, "cursor", 0)),
                "kind": type(sim).__name__}
    if not getattr(sim, "rebinds_tensors", False):   # simulators that own device tensors we can read back
        for name in _SIM_TENSORS:
            t = getattr(sim, name, None)
            if t is not None:
                out[f"sim/{name}"] = t.detach().cpu().numpy()
    out["meta"] = {
        "format": FORMAT_VERSION, "num_instances": int(env.num_instances), "global_num_instances": int(env._global_N),
        "env_offset": int(env._env_offset), "obs_dim": int(env.get_obs_dim()), "state_dim": int(env.get_state_dim()),
        "action_dim": int(env.get_action_dim()), "episode_statistics": _episode_statistics(env.config),
        "episode_term_returns": _activated(env.config, "episode_term_returns"),
        "dr_bias": _dr_bias(env.config), "sim": sim_meta, "config": json.loads(json.dumps(env.config, default=str)),
    }
    return out


def load_env_state_dict(env, state: Dict[str, object]) -> None:
    meta = state["meta"]
    if isinstance(meta, (str, bytes, np.ndarray)):
        meta = json.loads(str(meta))
    if meta.get("format") != FORMAT_VERSION:
        raise ValueError(f"checkpoint format {meta.get('format')} != {FORMAT_VERSION}")
    for key, have in (("num_instances", env.num_instances), ("global_num_instances", env._global_N),
                      ("env_offset", env._env_offset), ("obs_dim", env.get_obs_dim()),
                      ("state_dim", env.get_state_dim()), ("action_dim", env.get_action_dim())):
        if int(meta[key]) != int(have):
            raise ValueError(f"checkpoint was written for {key}={meta[key]}, this env has {have}")
    # the two streams are different random sequences (and "torch" carries generator state): never mix them
    have_stream = env.config.get("rng_stream", "philox")
    ck_stream = meta.get("config", {}).get("rng_stream", "philox")
    if ck_stream != have_stream:
        raise ValueError(f"checkpoint was written with rng_stream={ck_stream!r}, this env has {have_stream!r}")
    # with the setting on, the running returns and records are part of the state: never drop or invent them
    have_ep = _episode_statistics(env.config)
    ck_ep = bool(meta.get("episode_statistics", _episode_statistics(meta.get("config", {}))))
    if ck_ep != have_ep:
        raise ValueError(f"checkpoint was written with episode_statistics.activate={ck_ep}, this env has {have_ep}")
    have_terms = _activated(env.config, "episode_term_returns")
    ck_terms = bool(meta.get("episode_term_returns", _activated(meta.get("config", {}), "episode_term_returns")))
    if ck_terms != have_terms:
        raise ValueError(f"checkpoint was written with episode_term_returns.activate={ck_terms}, this env has {have_terms}")
    have_bias = _dr_bias(env.config)
    ck_bias = list(meta.get("dr_bias", _dr_bias(meta.get("config", {}))))
    if ck_bias != have_bias:
        raise ValueError(f"checkpoint was written with per-episode DR offsets (domain_randomization obs_bias_std / "
                         f"action_bias_std) on for [obs, action] = {ck_bias}, this env has {have_bias}")
    for name, attr in _ENV_TENSORS.items():
        t = getattr(env, attr, None)
        arr = state.get(f"env/{name}")
        if t is None or not t.numel():
            continue
        if arr is None:
            if name in ("obs_clipped", "states_clipped"):
                continue          # the writer had no wrapper attached; the next step refills them
            if name == "torch_rng":
                continue          # written before the torch stream existed: the env keeps its seeded state
            raise ValueError(f"checkpoint lacks env/{name}")
        src = torch.from_numpy(np.ascontiguousarray(arr))
        if tuple(src.shape) != tuple(t.shape) or src.dtype != t.dtype:
            raise ValueError(f"env/{name}: checkpoint {tuple(src.shape)} {src.dtype} != env {tuple(t.shape)} {t.dtype}")
        t.copy_(src)
    sim = env._sim
    if any(k.startswith("sim/") for k in state):
        for name in _SIM_TENSORS:
            arr, t = state.get(f"sim/{name}"), getattr(sim, name, None)
            if arr is not None and t is not None:
                t.copy_(torch.from_numpy(np.ascontiguousarray(arr)).view(t.shape))
    if hasattr(sim, "frame_count"):
        sim.frame_count = int(meta["sim"]["frame_count"])
    if hasattr(sim, "cursor"):
        sim.cursor = int(meta["sim"]["cursor"])
    env._clear_injection()
    env._step_info = env._make_info()
    torch.cuda.synchronize(env._torch_device)


def _episode_statistics(config: dict) -> bool:
    return _activated(config, "episode_statistics")


def _dr_bias(config: dict) -> list:
    """[obs offsets on, action offsets on]: which offset arrays the env keeps."""
    obs, act = dr_bias_sigmas(config)
    return [any(v != 0.0 for v in obs.values()), act != 0.0]


def _activated(config: dict, key: str) -> bool:
    return bool((config.get(key) or {}).get("activate", False))


def save_env_state(env, path: str) -> str:
    if not path.endswith(".npz"):
        path += ".npz"
    os.makedirs(os.path.dirname(path) or ".", exist_ok=True)
    state = env_state_dict(env)
    state["meta"] = np.array(json.dumps(state["meta"]))
    tmp = path + ".tmp.npz"
    np.savez(tmp, **state)
    os.replace(tmp, path)      # a crash mid-write never leaves a truncated checkpoint under the final name
    return path


def load_env_state(env, path: str) -> None:
    if not path.endswith(".npz"):
        path += ".npz"
    with np.load(path) as z:
        load_env_state_dict(env, {k: z[k] for k in z.files})
