"""ctypes binding of the C ABI in include/leibniz_b200.h.

The shared library is built in-tree (`python -m leibnizgym_b200.build` or
`__graft_entry__.build()`) as `leibnizgym_b200/libleibniz_b200.so`.  There is no
CPU fallback: if the library is missing or its struct layout disagrees with this
file, importing the native layer raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LG_LIB_PATH: development hook for same-box A/B runs of two builds of this library (scripts/ab_bench.sh)
LIB_PATH = os.environ.get("LG_LIB_PATH") or os.path.join(_HERE, "libleibniz_b200.so")

LG_MAX_ACTION_DIM = 18
LG_MAX_STATE_DIM = 122
LG_NUM_TERMS = 7
LG_NUM_STATS = 16
LG_INJECT_U_COLS = 24
LG_INJECT_N_COLS = 8
LG_HISTORY_COLS = 16
LG_NUM_COEF = 20

TERM_NAMES = ("finger_reach_object_rate", "finger_move_penalty", "object_dist", "object_rot",
              "object_rot_delta", "object_move", "keypoint")
CMD_MODES = {"position": 0, "torque": 1, "position_impedance": 2}
RESET_KINDS = {"none": 0, "default": 1, "random": 2}
RNG_STREAMS = {"philox": 0, "torch": 1}
STAT_POSITION_GOAL, STAT_ORIENTATION_GOAL, STAT_SUCCESSES, STAT_REWARD, STAT_RESETS, STAT_DONES = 7, 8, 9, 10, 11, 12
LG_NUM_EPISODE_STATS = 4
EPISODE_COUNT, EPISODE_RETURN_SUM, EPISODE_LENGTH_SUM, EPISODE_SUCCESSES = 0, 1, 2, 3   # LgEpisodeStat
LG_NUM_EPISODE_TERMS = 8
LG_EPISODE_TERM_BONUS = 7
EPISODE_TERM_NAMES = TERM_NAMES + ("success_bonus",)   # slots of the per-term episode return rows

c_float_p = C.POINTER(C.c_float)


class LgRewardTerm(C.Structure):
    _fields_ = [("activate", C.c_int32), ("_pad", C.c_int32), ("weight", C.c_double),
                ("sched_start", C.c_double), ("sched_end", C.c_double), ("scale", C.c_double),
                ("eps", C.c_double)]


class LgParams(C.Structure):
    _fields_ = [
        ("num_envs", C.c_int64), ("env_offset", C.c_int64), ("global_num_envs", C.c_int64),
        ("episode_length", C.c_int64),
        ("action_dim", C.c_int32), ("asymmetric_obs", C.c_int32), ("normalize_obs", C.c_int32),
        ("normalize_action", C.c_int32), ("command_mode", C.c_int32), ("apply_safety_damping", C.c_int32),
        ("task_difficulty", C.c_int32), ("robot_reset", C.c_int32), ("object_reset", C.c_int32),
        ("goal_rotation", C.c_int32), ("success_activate", C.c_int32), ("control_decimation", C.c_int32),
        ("bodies_per_env", C.c_int32), ("actors_per_env", C.c_int32), ("fingertip_body", C.c_int32 * 3),
        ("robot_slot", C.c_int32), ("object_slot", C.c_int32), ("goal_slot", C.c_int32),
        ("clip_obs", C.c_float), ("clip_actions", C.c_float), ("clip_input_actions", C.c_int32),
        ("dr_activate", C.c_int32), ("inject_draws", C.c_int32), ("use_device_clock", C.c_int32),
        ("fuse_bookkeeping", C.c_int32), ("term_active_mask", C.c_int32), ("seed", C.c_uint64),
        ("stats_num_envs", C.c_int64),
        ("dt", C.c_double), ("success_bonus", C.c_double), ("position_tolerance", C.c_double),
        ("orientation_tolerance", C.c_double), ("dof_pos_stddev", C.c_double), ("dof_vel_stddev", C.c_double),
        ("goal_rate_magnitude", C.c_double),
        ("terms", LgRewardTerm * LG_NUM_TERMS),
        ("scale_centre", C.c_float * LG_MAX_STATE_DIM), ("scale_span", C.c_float * LG_MAX_STATE_DIM),
        ("scale_rcp", C.c_float * LG_MAX_STATE_DIM),
        ("action_low", C.c_float * LG_MAX_ACTION_DIM), ("action_high", C.c_float * LG_MAX_ACTION_DIM),
        ("kp", C.c_float * 9), ("kd", C.c_float * 9), ("safety_kd", C.c_float * 9),
        ("torque_low", C.c_float * 9), ("torque_high", C.c_float * 9),
        ("dof_default_pos", C.c_float * 9), ("dof_default_vel", C.c_float * 9),
        ("cube_half_size", C.c_double), ("cube_radius_3d", C.c_double), ("cube_max_height", C.c_double),
        ("max_com_distance", C.c_double),
        ("dr_action_sigma", C.c_float), ("dr_sigma", C.c_float * LG_MAX_STATE_DIM), ("_pad_tail", C.c_int32),
        ("rng_stream", C.c_int32), ("sm_count", C.c_int32), ("threads_per_sm", C.c_int32), ("_pad_tail2", C.c_int32),
        ("dr_bias_sigma", C.c_float * 64), ("dr_bias_mask", C.c_uint64),
        ("dr_action_bias_sigma", C.c_float), ("_pad_tail3", C.c_int32),
    ]


class LgControl(C.Structure):
    _fields_ = [("rng_epoch", C.c_uint64), ("frame_count", C.c_int64), ("scan_ticket", C.c_uint32),
                ("scan_epoch", C.c_uint32), ("scan_readers", C.c_uint32), ("scan_exits", C.c_uint32)]


class LgTorchRng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("offset", C.c_uint64), ("launch_base", C.c_uint64),
                ("launch_counts", C.c_int32 * 2), ("acc", C.c_uint32 * 2), ("ticket", C.c_uint32), ("_pad", C.c_uint32)]


class LgSimState(C.Structure):
    _fields_ = [("dof_state", C.c_void_p), ("root_state", C.c_void_p), ("rigid_body", C.c_void_p),
                ("dof_force", C.c_void_p), ("ft_sensors", C.c_void_p)]


class LgBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "obs", "states", "obs_clipped", "states_clipped", "action", "reward", "reset", "goal_reset",
        "successes", "dones", "steps_count", "goal_pose", "goal_movement", "history", "applied_torque",
        "term_rewards", "step_stats", "reset_ids", "goal_reset_ids", "counts",
        "robot_indices", "reset_root_indices", "goal_root_indices", "scan_status", "control", "reward_coef", "scale_table",
        "inject_reset_u", "inject_reset_n", "inject_goal_u", "inject_goal_n", "obs_bf16", "states_bf16",
        "force_reset", "force_goal_reset",
        "episode_return", "last_episode_return", "last_episode_length", "last_episode_success", "episode_stats",
        "episode_term_return", "last_episode_term_return", "episode_term_stats",
        "obs_bias", "action_bias",
        "torch_rng")]


class LgHostStep(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "dof_state_host", "root_state_host", "rigid_body_host", "dof_force_host", "ft_sensors_host",
        "action_host", "obs_host", "states_host", "reward_host", "dones_host", "action_staging")]


# every symbol include/leibniz_b200.h declares: name -> (restype, argtypes)
_P, _S, _B = C.POINTER(LgParams), C.POINTER(LgSimState), C.POINTER(LgBuffers)
_vp, _i64, _i32 = C.c_void_p, C.c_int64, C.c_int32
SYMBOLS = {
    "lg_version": (C.c_int, []),
    "lg_last_error": (C.c_char_p, []),
    "lg_struct_size": (C.c_size_t, [C.c_int]),
    "lg_scan_tiles": (_i64, [_i64]),
    "lg_pre_resident_tiles": (_i64, []),
    "lg_set_l2_fetch_granularity": (C.c_int, [C.c_int]),
    "lg_pre_physics": (C.c_int, [_P, _S, _B, _vp, _vp]),
    "lg_pre_physics_chained": (C.c_int, [_P, _S, _B, _vp, C.c_int, _vp]),
    "lg_post_physics": (C.c_int, [_P, _S, _B, C.c_double, _vp]),
    "lg_fill_observations": (C.c_int, [_P, _S, _B, _vp]),
    "lg_init_history": (C.c_int, [_P, _S, _B, _vp]),
    "lg_compact": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "lg_reset_envs": (C.c_int, [_P, _S, _B, _vp, _i64, _vp]),
    "lg_goal_reset_envs": (C.c_int, [_P, _S, _B, _vp, _i64, _vp]),
    "lg_pre_step": (C.c_int, [_P, _S, _B, _vp]),
    "lg_quat_mul": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "lg_quat_diff_rad": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "lg_scale_transform": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "lg_unscale_transform": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "lg_saturate": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "lg_lgsk_kernel": (C.c_int, [_vp, C.c_float, _vp, _i64, _vp]),
    "lg_cube_keypoints": (C.c_int, [_vp, C.c_float, _vp, _i64, _vp]),
    "lg_integrate_goal": (C.c_int, [_P, _S, C.c_float, _vp]),
    "lg_selftest_division": (C.c_int, [C.c_float, C.c_float, _vp, _vp]),
    "lg_upload_sim_state": (C.c_int, [_P, _S, C.POINTER(LgHostStep), _vp]),
    "lg_step_host_pipelined": (C.c_int, [_P, _S, _B, C.POINTER(LgHostStep), C.c_double, C.c_int, _vp, _vp, _vp]),
    "lg_step_host": (C.c_int, [_P, _S, _B, C.POINTER(LgHostStep), C.c_double, _vp]),
    "lg_torch_philox": (C.c_int, [C.c_uint64, C.c_uint64, _i64, C.c_int, _vp, _vp]),
    "lg_torch_philox_advance": (C.c_uint64, [_i64, _i32, _i32]),
}


class NativeError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """Loads the library once; raises if it is missing or mismatched (no fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            f"{LIB_PATH} not found. leibnizgym_b200 has no CPU or PyTorch fallback: build the CUDA "
            "library first (`python -m leibnizgym_b200.build`).")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype, fn.argtypes = res, args
    for which, struct in enumerate((LgParams, LgSimState, LgBuffers, LgControl, LgRewardTerm, LgHostStep, LgTorchRng)):
        native = lib.lg_struct_size(which)
        if native != C.sizeof(struct):
            raise NativeError(f"ABI mismatch: sizeof({struct.__name__}) is {native} in the library, "
                              f"{C.sizeof(struct)} in the binding")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().lg_last_error().decode()
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise NativeError(f"{what}: error {rc}: {msg}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None stays None)."""
    return None if t is None else t.data_ptr()
