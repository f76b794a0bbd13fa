"""Configuration of the TriFinger MDP hot path.

The key names are the reference's (a user's config dict works unchanged):
simulator-level keys follow `ISAACGYM_DEFAULT_CONFIG_DICT` (ref
leibnizgym/envs/env_base.py:30-77), task-level keys follow
`TRIFINGER_DEFAULT_CONFIG_DICT` (ref leibnizgym/envs/trifinger/trifinger_env.py:28-115).
Unlike the reference, defaults are rebuilt per call — the reference mutates its
module-level dicts in place (SURVEY.md §C5), which leaks settings between envs.
"""
from __future__ import annotations

import copy
from collections.abc import Mapping
from typing import Any, Dict


def merge_config(base: dict, override: Mapping) -> dict:
    """Nested dict update with the semantics of the reference's `update_dict`
    (ref leibnizgym/utils/helpers.py:25-45): mappings merge, leaves overwrite.
    Operates on, and returns, `base`."""
    for key, val in override.items():
        if isinstance(val, Mapping):
            base[key] = merge_config(base.get(key, {}), val)
        else:
            base[key] = val
    return base


def default_sim_config() -> Dict[str, Any]:
    """Simulator-level defaults (ref env_base.py:30-77)."""
    return {
        "seed": 0,
        "num_instances": 1,
        "spacing": 1.0,
        "control_decimation": 1,
        "episode_length": None,
        "aggregate_mode": True,
        "physics_engine": "physx",
        "sim": {
            "dt": 0.02,
            "substeps": 2,
            "up_axis": "z",
            "gravity": [0.0, 0.0, -9.81],
            "num_client_threads": 0,
            "use_gpu_pipeline": False,
            "physx": {
                "solver_type": 1,
                "num_position_iterations": 4,
                "num_velocity_iterations": 0,
                "num_threads": 4,
                "use_gpu": False,
                "num_subscenes": 0,
                "max_gpu_contact_pairs": 8 * 1024 * 1024,
            },
            "flex": {
                "shape_collision_margin": 0.01,
                "num_outer_iterations": 4,
                "num_inner_iterations": 10,
            },
        },
    }


def default_trifinger_config() -> Dict[str, Any]:
    """Task-level defaults (ref trifinger_env.py:28-115): every reward term on,
    success termination on, position control."""
    return {
        "episode_length": 750,
        "task_difficulty": 1,
        "enable_ft_sensors": False,
        "command_mode": "position",
        "apply_safety_damping": True,
        "asymmetric_obs": False,
        "normalize_obs": True,
        "normalize_action": True,
        "reset_distribution": {
            "robot_initial_state": {"type": "default", "dof_pos_stddev": 0.4, "dof_vel_stddev": 0.2},
            "object_initial_state": {"type": "random"},
        },
        "goal_movement": {"rotation": {"activate": False, "rate_magnitude": 0.5}},
        "reward_terms": {
            "finger_reach_object_rate": {"activate": True, "weight": -750, "norm_p": 2},
            "finger_move_penalty": {"activate": True, "weight": -0.1},
            "object_dist": {"activate": True, "weight": 2000},
            "object_rot": {"activate": True, "weight": 300},
            "object_rot_delta": {"activate": True, "weight": -250},
            "object_move": {"activate": True, "weight": -750},
        },
        "termination_conditions": {
            "success": {
                "activate": True,
                "bonus": 5000.0,
                "position_tolerance": 0.01,
                "orientation_tolerance": 0.2,
            }
        },
        # ---- extensions of this build (absent from the reference; all default OFF so
        # ---- the default path is the reference's; SURVEY.md §8c "parity unpinned")
        "domain_randomization": {
            "activate": False,
            # additive Gaussian on the RAW actor observation groups, before scale_transform (the TODO of
            # trifinger_env.py:979); the critic's states stay clean
            "obs_noise_std": {"robot_q": 0.0, "robot_u": 0.0, "object_q": 0.0, "object_q_des": 0.0, "command": 0.0},
            "action_noise_std": 0.0,  # additive Gaussian on the action before clipping
            # per-episode offsets, drawn N(0, sigma^2) per env and column whenever the env is reset (not by a goal-only
            # reset) and held for the whole episode: a calibration error of the cube pose, an encoder bias, an action
            # offset.  Added to the raw actor observation before the noise above, and to the action before the noise
            # and the clip; env.obs_bias / env.action_bias hold them
            "obs_bias_std": {"robot_q": 0.0, "robot_u": 0.0, "object_q": 0.0, "object_q_des": 0.0, "command": 0.0},
            "action_bias_std": 0.0,
        },
        # where reset / goal samples come from: "philox" = this build's own counter stream, keyed by (seed, global env
        # id), the same for any sharding; "torch" = the numbers the reference's own torch.rand / torch.randn calls on
        # the CUDA device return after the same seed (one process only; env.sync_torch_generator / load_torch_generator)
        "rng_stream": "philox",
        # per-env running return and the record of each env's last finished episode (return, length, success), and
        # per step the count / return sum / length sum / successes of the episodes that ended, in `info`
        "episode_statistics": {"activate": False},
        # with "episode_statistics" on: each episode's return split by reward term plus the success bonus (running
        # and last finished, per env), and per step the per-term sums of the episodes that ended, in `info`
        "episode_term_returns": {"activate": False},
    }


# extension reward term (no reference code, SURVEY.md 8c(i)); add as reward_terms["keypoint"] to enable
KEYPOINT_TERM_DEFAULT = {"activate": False, "weight": 2000, "scale": 30.0, "eps": 2.0}


def difficulty_config(difficulty: int, num_instances: int, asymmetric_obs: bool = True,
                      seed: int = 0, **overrides) -> Dict[str, Any]:
    """The per-difficulty training configs the reference ships through Hydra
    (ref scripts/rlg_hydra.py:58-182, flattened; SURVEY.md §A.6).

    Difficulties 1-3: torque control; finger_move_penalty -0.1, finger_reach_object_rate
    -750, object_dist 2000 active; success termination off (tolerances 0.01 m / 0.1 rad).
    Difficulty 4: finger_reach_object_rate -250 gated [0, 1e7]; object_dist 2000 gated
    [0, 1e11]; object_rot 2000 (scale 3) gated [1e7, 1e10]; tolerances 0.02 m / 0.25 rad.
    """
    cfg: Dict[str, Any] = {
        "num_instances": int(num_instances),
        "seed": int(seed),
        "episode_length": 750,
        "task_difficulty": int(difficulty),
        "enable_ft_sensors": False,
        "asymmetric_obs": bool(asymmetric_obs),
        "normalize_obs": True,
        "apply_safety_damping": True,
        "command_mode": "torque",
        "normalize_action": True,
        "reset_distribution": {
            "object_initial_state": {"type": "random"},
            "robot_initial_state": {"dof_pos_stddev": 0.4, "dof_vel_stddev": 0.2, "type": "default"},
        },
        "sim": {"dt": 0.02},
    }
    if difficulty == 4:
        cfg["reward_terms"] = {
            "finger_move_penalty": {"activate": True, "weight": -0.1},
            "finger_reach_object_rate": {"activate": True, "norm_p": 2, "weight": -250,
                                         "thresh_sched_start": 0, "thresh_sched_end": 1e7},
            "object_dist": {"activate": True, "weight": 2000,
                            "thresh_sched_start": 0, "thresh_sched_end": 10e10},
            "object_rot": {"activate": True, "weight": 2000, "epsilon": 0.01, "scale": 3.0,
                           "thresh_sched_start": 1e7, "thresh_sched_end": 1e10},
            "object_rot_delta": {"activate": False, "weight": -250},
            "object_move": {"activate": False, "weight": -750},
        }
        cfg["termination_conditions"] = {"success": {
            "activate": False, "bonus": 5000.0,
            "orientation_tolerance": 0.25, "position_tolerance": 0.02}}
    else:
        cfg["reward_terms"] = {
            "finger_move_penalty": {"activate": True, "weight": -0.1},
            "finger_reach_object_rate": {"activate": True, "norm_p": 2, "weight": -750},
            "object_dist": {"activate": True, "weight": 2000},
            "object_rot": {"activate": False, "weight": 300},
            "object_rot_delta": {"activate": False, "weight": -250},
            "object_move": {"activate": False, "weight": -750},
        }
        cfg["termination_conditions"] = {"success": {
            "activate": False, "bonus": 5000.0,
            "orientation_tolerance": 0.1, "position_tolerance": 0.01}}
    return merge_config(cfg, overrides)


def resolve_config(user: Mapping | None) -> Dict[str, Any]:
    """Full config = sim defaults <- task defaults <- user dict (ref
    trifinger_env.py:268-273 then env_base.py:134-136).  Asymmetric observations
    force the force-torque sensors on (ref :272-273)."""
    cfg = default_sim_config()
    merge_config(cfg, default_trifinger_config())
    if user is not None:
        merge_config(cfg, copy.deepcopy(dict(user)))
    if cfg["asymmetric_obs"]:
        cfg["enable_ft_sensors"] = True
    return cfg
