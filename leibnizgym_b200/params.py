"""Config dict -> `LgParams` (the flattened parameter block of SURVEY.md §A.6).

Constants are the reference's (ref envs/trifinger/trifinger_env.py:143-224,
envs/trifinger/utils.py:54-131).  Scale tables are assembled in the reference's
order (ref trifinger_env.py:630-710) and reduced to centre/span in float32 with
the same two operations `scale_transform` performs (ref utils/torch_utils.py:33-36).
"""
from __future__ import annotations

import math
from typing import Dict, Tuple

import numpy as np

from . import _native as nat

F = np.float32

CUBE_SIZE = 0.065
ARENA_RADIUS = 0.195
MAX_TORQUE_NM = 0.36
MAX_VELOCITY_RADPS = 10

JOINT_POS_LOW = np.array([-0.33, 0.0, -2.7] * 3, dtype=F)
JOINT_POS_HIGH = np.array([1.0, 1.57, 0.0] * 3, dtype=F)
JOINT_POS_DEFAULT = np.array([0.0, 0.9, -1.7] * 3, dtype=F)
JOINT_STIFFNESS_LOW = np.array([1.0] * 9, dtype=F)
JOINT_STIFFNESS_HIGH = np.array([50.0] * 9, dtype=F)
GAIN_KP = np.array([10.0, 10.0, 10.0] * 3, dtype=F)
GAIN_KD = np.array([0.1, 0.3, 0.001] * 3, dtype=F)
GAIN_SAFETY_KD = np.array([0.08, 0.08, 0.04] * 3, dtype=F)

VALID_DIFFICULTIES = (-1, 1, 2, 3, 4, 5, 6)


def cube_geometry(size: float = CUBE_SIZE) -> Dict[str, float]:
    """ref envs/trifinger/utils.py:119-131 (python/NumPy double arithmetic)."""
    radius_3d = size * np.sqrt(3) / 2
    return {"half_size": size / 2, "radius_3d": float(radius_3d), "max_height": 0.1,
            "max_com_distance": float(ARENA_RADIUS - radius_3d)}


def action_dim_of(command_mode: str) -> int:
    return 18 if command_mode == "position_impedance" else 9


def action_scale(command_mode: str) -> Tuple[np.ndarray, np.ndarray]:
    """ref trifinger_env.py:636-651"""
    tq = np.full(9, MAX_TORQUE_NM, dtype=F)
    if command_mode == "position":
        return JOINT_POS_LOW.copy(), JOINT_POS_HIGH.copy()
    if command_mode == "torque":
        return -tq, tq
    if command_mode == "position_impedance":
        return (np.concatenate([JOINT_POS_LOW, JOINT_STIFFNESS_LOW]),
                np.concatenate([JOINT_POS_HIGH, JOINT_STIFFNESS_HIGH]))
    raise ValueError(f"Invalid command mode. Input: {command_mode} not in ['torque', 'position'].")


def observation_scale(cfg: dict) -> Tuple[np.ndarray, np.ndarray]:
    """ref trifinger_env.py:655-680"""
    A = action_dim_of(cfg["command_mode"])
    if cfg["normalize_action"]:
        a_lo, a_hi = np.full(A, -1, dtype=F), np.full(A, 1, dtype=F)
    else:
        a_lo, a_hi = action_scale(cfg["command_mode"])
    vel = np.full(9, MAX_VELOCITY_RADPS, dtype=F)
    pos_lo, pos_hi = np.array([-0.3, -0.3, 0], dtype=F), np.array([0.3, 0.3, 0.3], dtype=F)
    one4 = np.ones(4, dtype=F)
    lo = np.concatenate([JOINT_POS_LOW, -vel, pos_lo, -one4, pos_lo, -one4, a_lo])
    hi = np.concatenate([JOINT_POS_HIGH, vel, pos_hi, one4, pos_hi, one4, a_hi])
    return lo, hi


def state_scale(cfg: dict) -> Tuple[np.ndarray, np.ndarray]:
    """ref trifinger_env.py:682-710"""
    o_lo, o_hi = observation_scale(cfg)
    one4 = np.ones(4, dtype=F)
    tip_lo = np.concatenate([np.array([-0.4, -0.4, 0], dtype=F), -one4, np.full(6, -0.2, dtype=F)])
    tip_hi = np.concatenate([np.array([0.4, 0.4, 0.5], dtype=F), one4, np.full(6, 0.2, dtype=F)])
    ov = np.full(6, 0.5, dtype=F)
    tq = np.full(9, MAX_TORQUE_NM, dtype=F)
    wr = np.full(6, 1.0, dtype=F)
    lo = np.concatenate([o_lo, -ov, np.tile(tip_lo, 3), -tq, np.tile(-wr, 3)])
    hi = np.concatenate([o_hi, ov, np.tile(tip_hi, 3), tq, np.tile(wr, 3)])
    return lo, hi


_TERM_DEFAULT_WEIGHT = {  # constructor defaults, ref rewards.py:44, :71, :107, :155, :195, :244
    "finger_reach_object_rate": -250, "finger_move_penalty": -1.0e-4, "object_dist": 2000,
    "object_rot": 100, "object_rot_delta": 100, "object_move": -750, "keypoint": 2000,
}


def _fill_terms(p: nat.LgParams, cfg_terms: dict) -> None:
    for i, name in enumerate(nat.TERM_NAMES):
        t = p.terms[i]
        c = cfg_terms.get(name)
        if c is None:
            if name != "keypoint":
                # the reference indexes all six terms unconditionally (trifinger_env.py:513-550)
                raise KeyError(name)
            t.activate = 0
            continue
        t.activate = int(bool(c["activate"]))
        t.weight = float(c.get("weight", _TERM_DEFAULT_WEIGHT[name]))
        if name == "object_rot_delta":  # ref rewards.py:158-159
            t.sched_start = float(c.get("linear_schedule_start", 0))
            t.sched_end = float(c.get("linear_schedule_end", 0))
        else:                           # ref rewards.py:46-47, :112-113, :197-198
            t.sched_start = float(c.get("thresh_sched_start", 0))
            t.sched_end = float(c.get("thresh_sched_end", 0))
        t.scale = float(c.get("scale", 30.0 if name == "keypoint" else 1.0))
        t.eps = float(c.get("eps", 2.0))
        if name == "finger_reach_object_rate" and c.get("norm_p", 2) != 2:
            raise ValueError("finger_reach_object_rate.norm_p: only the 2-norm is built")


OBS_GROUPS = ("robot_q", "robot_u", "object_q", "object_q_des", "command")


def obs_group_columns(action_dim: int) -> Dict[str, Tuple[int, int]]:
    """Raw actor observation columns [a, b) of each obs_spec group (trifinger_env.py:280-286)."""
    return {"robot_q": (0, 9), "robot_u": (9, 18), "object_q": (18, 25), "object_q_des": (25, 32),
            "command": (32, 32 + action_dim)}


def _sigma(value, key: str) -> float:
    try:
        s = float(value)
    except (TypeError, ValueError):
        raise ValueError(f"{key} must be a number, got {value!r}") from None
    if not math.isfinite(s) or s < 0.0:
        raise ValueError(f"{key} must be finite and >= 0, got {value!r}")
    return s


def dr_bias_sigmas(cfg: dict) -> Tuple[Dict[str, float], float]:
    """Per-episode offsets of "domain_randomization" (extension): (sigma per obs group, sigma of the action offset),
    all zero unless `activate`.  Raises ValueError naming the key for a negative or non-finite sigma or an unknown
    group."""
    dr = cfg.get("domain_randomization") or {}
    groups = {name: 0.0 for name in OBS_GROUPS}
    if not dr.get("activate", False):
        return groups, 0.0
    obs = dr.get("obs_bias_std") or {}
    for name, value in obs.items():
        if name not in groups:
            raise ValueError(f"domain_randomization.obs_bias_std: unknown observation group {name!r} "
                             f"(groups: {list(OBS_GROUPS)})")
        groups[name] = _sigma(value, f"domain_randomization.obs_bias_std.{name}")
    return groups, _sigma(dr.get("action_bias_std", 0.0), "domain_randomization.action_bias_std")


def build_params(cfg: dict, num_local_envs: int, env_offset: int = 0, global_num_envs: int | None = None,
                 fingertip_bodies=(6, 11, 16), bodies_per_env: int = 20, actors_per_env: int = 4,
                 slots=(0, 2, 3), sm_count: int = 0, threads_per_sm: int = 0) -> nat.LgParams:
    """Flattens a resolved config (config.resolve_config) into the kernel parameter block.  `sm_count` /
    `threads_per_sm`: the device's, which fix torch's launch grid and so its stream ("rng_stream": "torch")."""
    mode = cfg["command_mode"]
    if mode not in nat.CMD_MODES:
        raise ValueError(f"Invalid command mode. Input: {mode} not in ['torque', 'position'].")
    d = cfg["task_difficulty"]
    if d not in VALID_DIFFICULTIES:
        raise ValueError(f"Invalid difficulty index for task: {d}.")
    rd = cfg["reset_distribution"]
    r_kind, o_kind = rd["robot_initial_state"]["type"], rd["object_initial_state"]["type"]
    if r_kind not in nat.RESET_KINDS:
        raise ValueError(f"Invalid robot initial state distribution. Input: {r_kind} not in [`default`, `random`].")
    if o_kind not in nat.RESET_KINDS:
        raise ValueError(f"Invalid object initial state distribution. Input: {o_kind} "
                         "not in [`default`, `random`, `none`].")

    stream = cfg.get("rng_stream", "philox")
    if stream not in nat.RNG_STREAMS:
        raise ValueError(f"Invalid rng_stream. Input: {stream!r} not in {list(nat.RNG_STREAMS)}.")

    p = nat.LgParams()
    p.num_envs = int(num_local_envs)
    p.env_offset = int(env_offset)
    p.global_num_envs = int(global_num_envs if global_num_envs is not None else num_local_envs)
    ep = cfg["episode_length"]
    p.episode_length = -1 if ep is None else int(ep)
    A = action_dim_of(mode)
    p.action_dim = A
    p.asymmetric_obs = int(bool(cfg["asymmetric_obs"]))
    p.normalize_obs = int(bool(cfg["normalize_obs"]))
    p.normalize_action = int(bool(cfg["normalize_action"]))
    p.command_mode = nat.CMD_MODES[mode]
    p.apply_safety_damping = int(bool(cfg["apply_safety_damping"]))
    p.task_difficulty = int(d)
    p.robot_reset, p.object_reset = nat.RESET_KINDS[r_kind], nat.RESET_KINDS[o_kind]
    rot = cfg["goal_movement"]["rotation"]
    p.goal_rotation = int(bool(rot["activate"]))
    p.goal_rate_magnitude = float(rot["rate_magnitude"])
    succ = cfg["termination_conditions"]["success"]
    p.success_activate = int(bool(succ["activate"]))
    p.success_bonus = float(succ["bonus"])
    p.position_tolerance = float(succ["position_tolerance"])
    p.orientation_tolerance = float(succ["orientation_tolerance"])
    p.control_decimation = int(cfg["control_decimation"])
    p.dt = float(cfg["sim"]["dt"])
    p.dof_pos_stddev = float(rd["robot_initial_state"].get("dof_pos_stddev", 0.0))
    p.dof_vel_stddev = float(rd["robot_initial_state"].get("dof_vel_stddev", 0.0))
    _fill_terms(p, cfg["reward_terms"])
    p.term_active_mask = sum((1 << i) for i in range(nat.LG_NUM_TERMS) if p.terms[i].activate)

    lo, hi = state_scale(cfg) if cfg["asymmetric_obs"] else observation_scale(cfg)
    centre = ((lo + hi) * F(0.5)).astype(F)   # torch: (lower + upper) * 0.5 in fp32
    span = (hi - lo).astype(F)                # torch: upper - lower in fp32
    rcp = (F(1.0) / span).astype(F)           # IEEE fp32 division: the correctly rounded reciprocal
    for i in range(len(lo)):
        p.scale_centre[i], p.scale_span[i], p.scale_rcp[i] = centre[i], span[i], rcp[i]
    a_lo, a_hi = action_scale(mode)
    for i in range(A):
        p.action_low[i], p.action_high[i] = a_lo[i], a_hi[i]
    for i in range(9):
        p.kp[i], p.kd[i], p.safety_kd[i] = GAIN_KP[i], GAIN_KD[i], GAIN_SAFETY_KD[i]
        p.torque_low[i], p.torque_high[i] = -F(MAX_TORQUE_NM), F(MAX_TORQUE_NM)
        p.dof_default_pos[i], p.dof_default_vel[i] = JOINT_POS_DEFAULT[i], 0.0
    g = cube_geometry()
    p.cube_half_size, p.cube_radius_3d = g["half_size"], g["radius_3d"]
    p.cube_max_height, p.max_com_distance = g["max_height"], g["max_com_distance"]
    p.bodies_per_env, p.actors_per_env = int(bodies_per_env), int(actors_per_env)
    for i in range(3):
        p.fingertip_body[i] = int(fingertip_bodies[i])
    p.robot_slot, p.object_slot, p.goal_slot = (int(s) for s in slots)
    p.clip_obs, p.clip_actions, p.clip_input_actions = 5.0, 1.0, 0
    dr = cfg.get("domain_randomization", {})
    p.dr_activate = int(bool(dr.get("activate", False)))
    p.dr_action_sigma = float(dr.get("action_noise_std", 0.0)) if p.dr_activate else 0.0
    if p.dr_activate:  # sigma per RAW observation column, by the obs_spec groups (trifinger_env.py:280-286)
        std = dr.get("obs_noise_std", {})
        for name, (a, b) in obs_group_columns(A).items():
            for c in range(a, b):
                p.dr_sigma[c] = float(std.get(name, 0.0))
    obs_bias, p.dr_action_bias_sigma = dr_bias_sigmas(cfg)   # per-episode offsets (zero unless activate)
    for name, (a, b) in obs_group_columns(A).items():
        for c in range(a, b):
            p.dr_bias_sigma[c] = obs_bias[name]
            if p.dr_bias_sigma[c] != 0.0:
                p.dr_bias_mask |= 1 << c
    p.seed = int(cfg["seed"]) & 0xFFFFFFFFFFFFFFFF
    p.rng_stream = nat.RNG_STREAMS[stream]
    p.sm_count, p.threads_per_sm = int(sm_count), int(threads_per_sm)
    p.inject_draws = 0
    p.use_device_clock = 0
    p.fuse_bookkeeping = 1
    return p


TWO_PI = 2.0 * math.pi
