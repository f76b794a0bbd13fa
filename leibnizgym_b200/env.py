"""Drop-in `IsaacEnvBase` / `TrifingerEnv` whose MDP hot path runs in sm_100a kernels.

Interface mirrored from the reference (same constructor arguments, hooks, buffer
properties, getters, return values and exceptions):
    IsaacEnvBase   ref leibnizgym/envs/env_base.py:79-614
    TrifingerEnv   ref leibnizgym/envs/trifinger/trifinger_env.py:118-1284
What differs by design:
  * the simulator is an object passed in (`sim=`; default `SyntheticSim`) instead of the
    closed-source isaacgym module — PhysX is out of scope (BASELINE.json);
  * buffers are persistent and written in place (the reference re-binds `_obs_buf` /
    `_states_buf` each step, SURVEY.md §C4) and `step()` never synchronises the host
    (the reference does, 4x per step: `nonzero`, `len`, `unique`, `.cpu()`);
  * `step()` issues two fused launches (lg_pre_physics / lg_post_physics) instead of
    ~350-550 ATen ops; the individual hooks stay callable and do the same work;
  * CUDA only: there is no CPU path (`device='cpu'` raises).
"""
from __future__ import annotations

import os
import random
from types import SimpleNamespace
from typing import Dict, Optional, Tuple, Union

import numpy as np
import torch
import yaml

from . import _native as nat
from .config import resolve_config
from .params import action_dim_of, action_scale, build_params, dr_bias_sigmas, observation_scale, state_scale
from .sim import LazyCount, SyntheticSim
from .synthetic import make_sequence

# `info` keys of the episode statistics, in LgEpisodeStat order
EPISODE_KEYS = ("env/episodes/count", "env/episodes/return_sum", "env/episodes/length_sum", "env/episodes/successes")


class IsaacEnvBase:
    """Template-method env runtime: buffers, step sequencing, timeout bookkeeping
    (ref leibnizgym/envs/env_base.py).  Sub-classes implement the five hooks."""

    def __init__(self, obs_spec: Dict[str, int], action_spec: Dict[str, int], state_spec: Dict[str, int],
                 config: dict = None, device: str = "cuda:0", verbose: bool = True, visualize: bool = False):
        self.obs_spec, self.action_spec, self.state_spec = obs_spec, action_spec, state_spec
        self.device = device
        self.verbose = verbose
        self.visualize = visualize
        self.config = config
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError(f"leibnizgym_b200 is CUDA-only (sm_100a kernels, no CPU fallback); got device={device!r}")
        if not torch.cuda.is_available():
            raise RuntimeError("leibnizgym_b200 needs a CUDA device")
        self._torch_device = dev
        nat.load()  # fail now, loudly, if the CUDA library is not built
        self.num_instances = self.config["num_instances"]
        self.control_decimation = self.config["control_decimation"]
        self.episode_length = self.config["episode_length"]
        if self.config["physics_engine"] not in ("physx", "flex"):  # ref env_base.py:579-587
            raise ValueError(f"Invalid physics engine backend: {self.config['physics_engine']}")
        if self.config["sim"]["up_axis"] not in ("z", "y"):         # ref env_base.py:504-507
            raise ValueError(f"Invalid physics up-axis: {self.config['sim']['up_axis']}")
        self._observations_scale = SimpleNamespace(low=None, high=None)
        self._states_scale = SimpleNamespace(low=None, high=None)
        self._action_scale = SimpleNamespace(low=None, high=None)
        self._step_info: Dict[str, torch.Tensor] = {}
        self._allocate_buffers()
        self._setup_sim()
        self.seed(self.config["seed"])

    def _allocate_buffers(self):
        """ref env_base.py:533-572"""
        N, dev = self.num_instances, self._torch_device
        sd, od, ad = sum(self.state_spec.values()), sum(self.obs_spec.values()), sum(self.action_spec.values())
        self._states_buf = torch.zeros((N, sd), device=dev, dtype=torch.float)
        self._obs_buf = torch.zeros((N, od), device=dev, dtype=torch.float)
        self._action_buf = torch.zeros((N, ad), device=dev, dtype=torch.float)
        self._reset_buf = torch.zeros(N, device=dev, dtype=torch.bool)
        self._goal_reset_buf = torch.zeros(N, device=dev, dtype=torch.bool)
        self._reward_buf = torch.zeros(N, device=dev, dtype=torch.float)
        self._steps_count_buf = torch.zeros(N, device=dev, dtype=torch.long)

    # -- getters (ref env_base.py:222-255) ---------------------------------------------
    def get_state_shape(self) -> torch.Size:
        return self._states_buf.size()

    def get_obs_shape(self) -> torch.Size:
        return self._obs_buf.size()

    def get_action_shape(self) -> torch.Size:
        return self._action_buf.size()

    def get_num_instances(self) -> int:
        return self.num_instances

    def get_state_dim(self) -> int:
        return self.get_state_shape()[1]

    def get_obs_dim(self) -> int:
        return self.get_obs_shape()[1]

    def get_action_dim(self) -> int:
        return self.get_action_shape()[1]

    # -- buffer access (ref env_base.py:261-289) -----------------------------------------
    @property
    def states_buf(self) -> torch.Tensor:
        return self._states_buf

    @property
    def obs_buf(self) -> torch.Tensor:
        return self._obs_buf

    @property
    def action_buf(self) -> torch.Tensor:
        return self._action_buf

    @property
    def reward_buf(self) -> torch.Tensor:
        return self._reward_buf

    @property
    def dones_buf(self) -> torch.Tensor:
        return self._reset_buf

    @property
    def env_steps_count(self) -> int:
        """frames x env count over the WHOLE job, so schedules are invariant to sharding."""
        return self._frame_count() * self._global_num_instances()

    def _frame_count(self) -> int:
        raise NotImplementedError

    def _global_num_instances(self) -> int:
        return self.num_instances

    # -- operations (ref env_base.py:295-401) ----------------------------------------------
    def dump_config(self, filename: str):
        if not filename.endswith(".yaml"):
            filename += ".yaml"
        os.makedirs(os.path.dirname(filename) or ".", exist_ok=True)
        with open(filename, "w") as f:
            yaml.dump(self.config, f)

    @staticmethod
    def seed(seed: int = None):
        random.seed(seed)
        np.random.seed(seed)
        if seed is not None:
            torch.manual_seed(seed)

    def reset(self) -> torch.Tensor:
        """ref env_base.py:322-343"""
        self._reset_impl(torch.arange(0, self.num_instances, device=self._torch_device))
        self._pre_step()
        self._simulate()
        self._fill_observations_and_states()
        return self._obs_buf.clone().detach()

    def _check_action(self, action) -> torch.Tensor:
        if isinstance(action, np.ndarray):
            action = torch.tensor(action, dtype=torch.float, device=self._torch_device)
        shape = (self.num_instances, self.get_action_dim())
        if tuple(action.size()) != shape:
            raise ValueError(f"Invalid shape for tensor `action`. Input: {tuple(action.size())} != {shape}.")
        if getattr(self, "_host_io", False) and action.device.type == "cpu" and action.is_pinned() \
                and action.dtype == torch.float and action.is_contiguous():
            return action  # pinned host memory is addressable from the kernel (UVA): no staging copy
        action = action.to(self._torch_device, dtype=torch.float, non_blocking=True).contiguous()
        if action.data_ptr() % 16:   # an offset view (e.g. a slice of a larger rollout buffer): the bulk copies need 16 B
            action = action.clone()
        return action

    def step(self, action: Union[np.ndarray, torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, dict]:
        """Generic hook-by-hook sequencing (ref env_base.py:345-401); TrifingerEnv overrides it
        with the fused two-launch version."""
        dr = self.config.get("domain_randomization") or {}
        for key in ("action_noise_std", "action_bias_std"):
            if dr.get("activate") and float(dr.get(key, 0.0)) != 0.0:
                # the action noise is keyed by the compaction epoch, which only the fused pre-physics pass advances:
                # hook steps would store the raw action and, if they drew at all, draw the same noise every step.  The
                # action offset is added by that pass too
                raise ValueError(f"domain_randomization.{key} > 0 is applied by the fused step only: "
                                 "step with TrifingerEnv.step, not the hook-by-hook IsaacEnvBase.step")
        self._step_info = {}
        action = self._check_action(action)
        self._action_buf.copy_(action)
        env_ids = torch.nonzero(self._reset_buf).view(-1)
        if len(env_ids) > 0:
            self._reset_impl(env_ids)
        goal_env_ids = torch.nonzero(self._goal_reset_buf).view(-1)
        if len(goal_env_ids) > 0:
            self._goal_reset_impl(goal_env_ids)
        self._pre_step()
        for _ in range(self.control_decimation):
            self._simulate()
        self._post_step()
        self._steps_count_buf += 1
        if self.episode_length is not None:
            self._reset_buf.logical_or_(torch.greater_equal(self._steps_count_buf, self.episode_length))
        dones = torch.logical_and(self._reset_buf, self._goal_reset_buf)
        return self._obs_buf, self._reward_buf, dones, self._step_info

    def render(self):
        print("[WARN] The function `render()` called without visualization enabled.")

    def close(self):
        pass

    # -- hooks (ref env_base.py:444-490) -----------------------------------------------------
    def _setup_sim(self):
        raise NotImplementedError

    def _simulate(self):
        raise NotImplementedError

    def _fill_observations_and_states(self):
        raise NotImplementedError

    def _reset_impl(self, instances: torch.Tensor):
        raise NotImplementedError

    def _goal_reset_impl(self, instances: torch.Tensor):
        raise NotImplementedError

    def _pre_step(self):
        raise NotImplementedError

    def _post_step(self):
        raise NotImplementedError


class TrifingerEnv(IsaacEnvBase):
    """TriFinger cube-manipulation MDP (ref leibnizgym/envs/trifinger/trifinger_env.py).

    Args:
        config: the reference's config dict (merged over its defaults, config.resolve_config).
        device: CUDA device string.
        sim: simulator object owning the state tensors (default: SyntheticSim over a seeded
            64-step sequence).  Needs: dof_state, root_state, rigid_body, dof_force,
            ft_sensors, fingertip_bodies, bodies_per_env, actors_per_env, slots, simulate(),
            get_frame_count(), set_dof_actuation_force_tensor(), set_*_tensor_indexed().
        rank / world_size: this process' shard of `config["num_instances"]` envs
            (contiguous blocks of global env index, SURVEY.md §8e).
    """

    def __init__(self, config: dict = None, device: str = "cuda:0", verbose: bool = True, visualize: bool = False,
                 sim=None, rank: int = 0, world_size: int = 1):
        if config is None or "command_mode" not in config:
            # the reference reads config['command_mode'] of the CALLER's dict (trifinger_env.py:277)
            raise KeyError("command_mode")
        cfg = resolve_config(config)
        self._global_N = int(cfg["num_instances"])
        self.rank, self.world_size = int(rank), int(world_size)
        if self._global_N % self.world_size != 0:
            raise ValueError("num_instances must be divisible by world_size")
        if cfg.get("rng_stream", "philox") == "torch" and self.world_size > 1:
            # the reference is one process drawing for all envs: a per-shard copy of its stream is no run of it
            raise ValueError('rng_stream "torch" draws the stream of one process over all envs: world_size must be 1')
        local_n = self._global_N // self.world_size
        self._env_offset = self.rank * local_n
        cfg["num_instances"] = local_n  # buffers hold the local shard; config['global_num_instances'] keeps the total
        cfg["global_num_instances"] = self._global_N
        A = action_dim_of(cfg["command_mode"])
        if cfg["command_mode"] not in nat.CMD_MODES:
            raise ValueError(f"Invalid command mode. Input: {cfg['command_mode']} not in ['torque', 'position'].")
        if cfg["episode_term_returns"]["activate"] and not cfg["episode_statistics"]["activate"]:
            raise ValueError('"episode_term_returns" needs "episode_statistics": {"activate": True}: the per-term '
                             "returns are kept and reported with the episode statistics")
        dr_bias_sigmas(cfg)   # a bad sigma or group of the per-episode DR offsets raises here, before any device work
        obs_spec = {"robot_q": 9, "robot_u": 9, "object_q": 7, "object_q_des": 7, "command": A}
        if cfg["asymmetric_obs"]:
            state_spec = dict(obs_spec, object_u=6, fingertip_state=39, robot_a=9, fingertip_wrench=18)
        else:
            state_spec = {}
        self._sim = sim
        self._lib = nat.load()
        super().__init__(obs_spec, {"command": A}, state_spec, cfg, device=device, verbose=verbose, visualize=visualize)
        self._configure_mdp_spaces()
        self._bind()
        if verbose:
            terms = {k: v for k, v in self.config["reward_terms"].items()}
            print(f"[INFO] TrifingerEnv(B200): {self.num_instances} envs on {device} "
                  f"(global {self._global_N}, rank {self.rank}/{self.world_size}); reward terms: {terms}")

    # -- construction --------------------------------------------------------------------------
    def _setup_sim(self):
        """ref trifinger_env.py:356-371 builds the PhysX scene; here: adopt / create the synthetic sim."""
        N, dev = self.num_instances, self._torch_device
        if self._sim is None:
            seq = make_sequence(self.config["seed"], 64, N, device=str(dev), first_env=self._env_offset)
            self._sim = SyntheticSim(seq, device=str(dev))
        s = self._sim
        # zero-copy views of simulator memory (ref trifinger_env.py:602-617)
        self._dof_state = s.dof_state.view(N, 9, 2)
        self._dof_position = self._dof_state[..., 0]
        self._dof_velocity = self._dof_state[..., 1]
        self._rigid_body_state = s.rigid_body.view(N, s.bodies_per_env, 13)
        self._actors_root_state = s.root_state.view(-1, 13)
        self._dof_torque = s.dof_force.view(N, 9) if self.config["enable_ft_sensors"] else None
        self._ft_sensors_values = s.ft_sensors.view(N, 18) if self.config["enable_ft_sensors"] else None
        e = torch.arange(N, device=dev, dtype=torch.long) * s.actors_per_env
        self._gym_indices = {"robot": e + s.slots[0], "stage": e + 1, "object": e + s.slots[1],
                             "goal_object": e + s.slots[2]}
        i32 = dict(device=dev, dtype=torch.int32)
        self._object_goal_poses_buf = torch.zeros((N, 7), device=dev, dtype=torch.float)
        self._object_goal_movement_buf = torch.zeros((N, 6), device=dev, dtype=torch.float)
        self._successes = torch.zeros(N, device=dev, dtype=torch.bool)
        self._dones = torch.zeros(N, device=dev, dtype=torch.bool)
        self._history = torch.zeros((N, nat.LG_HISTORY_COLS), device=dev, dtype=torch.float)
        self._applied_torque = torch.zeros((N, 9), device=dev, dtype=torch.float)
        self._term_rewards = None
        self._obs_clipped = self._states_clipped = None
        self._obs_bf16 = self._states_bf16 = None
        self._step_stats = torch.zeros(nat.LG_NUM_STATS, device=dev, dtype=torch.float64)
        # extension: episode statistics (all five buffers or none; the kernels check)
        self._episode_return = self._last_episode_return = self._last_episode_length = None
        self._last_episode_success = self._episode_stats = None
        if self.config["episode_statistics"]["activate"]:
            self._episode_return = torch.zeros(N, device=dev, dtype=torch.float)
            self._last_episode_return = torch.zeros(N, device=dev, dtype=torch.float)
            self._last_episode_length = torch.zeros(N, device=dev, dtype=torch.long)
            self._last_episode_success = torch.zeros(N, device=dev, dtype=torch.bool)
            self._episode_stats = torch.zeros(nat.LG_NUM_EPISODE_STATS, device=dev, dtype=torch.float64)
        # extension: per-term episode returns (all three or none, on top of the five above)
        self._episode_term_return = self._last_episode_term_return = self._episode_term_stats = None
        if self.config["episode_term_returns"]["activate"]:
            T = nat.LG_NUM_EPISODE_TERMS
            self._episode_term_return = torch.zeros((N, T), device=dev, dtype=torch.float)
            self._last_episode_term_return = torch.zeros((N, T), device=dev, dtype=torch.float)
            self._episode_term_stats = torch.zeros(T, device=dev, dtype=torch.float64)
        # extension: per-episode DR offsets, each allocated only when one of its sigmas is nonzero
        obs_sig, act_sig = dr_bias_sigmas(self.config)
        A = action_dim_of(self.config["command_mode"])
        self._obs_bias = (torch.zeros((N, 32 + A), device=dev, dtype=torch.float)
                          if any(v != 0.0 for v in obs_sig.values()) else None)
        self._action_bias = torch.zeros((N, A), device=dev, dtype=torch.float) if act_sig != 0.0 else None
        self._reset_ids = torch.zeros(N, device=dev, dtype=torch.long)
        self._goal_reset_ids = torch.zeros(N, device=dev, dtype=torch.long)
        self._counts = torch.zeros(2, **i32)
        self._robot_indices = torch.zeros(N, **i32)
        self._reset_root_indices = torch.zeros(3 * N, **i32)
        self._goal_root_indices = torch.zeros(N, **i32)
        self._reward_coef = torch.zeros(nat.LG_NUM_COEF, device=dev, dtype=torch.float)
        self._scan_status = torch.zeros(int(self._lib.lg_scan_tiles(N)), device=dev, dtype=torch.int64)
        self._control = torch.zeros(4, device=dev, dtype=torch.int64)  # LgControl, 32 bytes
        self._inject = {}
        # LgTorchRng, 48 bytes: torch's CUDA generator state (seed, offset) for "rng_stream": "torch", and workspace
        self._torch_rng = torch.zeros(6, device=dev, dtype=torch.int64)
        props = torch.cuda.get_device_properties(dev)
        self._P = build_params(self.config, N, env_offset=self._env_offset, global_num_envs=self._global_N,
                               fingertip_bodies=s.fingertip_bodies, bodies_per_env=s.bodies_per_env,
                               actors_per_env=s.actors_per_env, slots=s.slots, sm_count=props.multi_processor_count,
                               threads_per_sm=props.max_threads_per_multi_processor)
        tab = np.zeros((4, nat.LG_MAX_STATE_DIM), np.float32)
        tab[0], tab[1], tab[2] = self._P.scale_centre, self._P.scale_span, self._P.scale_rcp
        tab[3] = self._P.dr_sigma
        tab[1][tab[1] == 0] = 1.0
        self._scale_table = torch.as_tensor(tab, device=dev).contiguous()

    def _configure_mdp_spaces(self):
        """Scale vectors as tensors, for callers that read them (ref trifinger_env.py:630-748)."""
        dev = self._torch_device
        lo, hi = action_scale(self.config["command_mode"])
        self._action_scale.low, self._action_scale.high = torch.tensor(lo, device=dev), torch.tensor(hi, device=dev)
        lo, hi = observation_scale(self.config)
        self._observations_scale.low, self._observations_scale.high = torch.tensor(lo, device=dev), torch.tensor(hi, device=dev)
        if self.config["asymmetric_obs"]:
            lo, hi = state_scale(self.config)
            self._states_scale.low, self._states_scale.high = torch.tensor(lo, device=dev), torch.tensor(hi, device=dev)
        else:
            self._states_scale.low = self._states_scale.high = torch.zeros(0, device=dev)
        obs_dim, st_dim, a_dim = sum(self.obs_spec.values()), sum(self.state_spec.values()), sum(self.action_spec.values())
        if self._observations_scale.low.shape[0] != obs_dim:
            raise AssertionError(f"Observation scaling dimensions mismatch. \tExpected: {obs_dim}.")
        if self._states_scale.low.shape[0] != st_dim:
            raise AssertionError(f"States scaling dimensions mismatch. \tExpected: {st_dim}.")
        if self._action_scale.low.shape[0] != a_dim:
            raise AssertionError(f"Actions scaling dimensions mismatch. \tExpected: {a_dim}.")

    def _bind(self):
        """(Re)builds the pointer structs handed to the C ABI and seeds the history."""
        s, p = self._sim, nat.ptr
        self._S = nat.LgSimState(p(s.dof_state), p(s.root_state), p(s.rigid_body), p(s.dof_force), p(s.ft_sensors))
        b = nat.LgBuffers()
        b.obs, b.states = p(self._obs_buf), (p(self._states_buf) if self.config["asymmetric_obs"] else None)
        b.obs_clipped, b.states_clipped = p(self._obs_clipped), p(self._states_clipped)
        b.action, b.reward = p(self._action_buf), p(self._reward_buf)
        b.reset, b.goal_reset, b.successes, b.dones = p(self._reset_buf), p(self._goal_reset_buf), p(self._successes), p(self._dones)
        b.steps_count = p(self._steps_count_buf)
        b.goal_pose, b.goal_movement, b.history = p(self._object_goal_poses_buf), p(self._object_goal_movement_buf), p(self._history)
        b.applied_torque, b.term_rewards = p(self._applied_torque), p(self._term_rewards)
        b.step_stats = p(self._step_stats)
        b.obs_bf16, b.states_bf16 = p(self._obs_bf16), p(self._states_bf16)
        fr, fg = getattr(self, "_force_masks", (None, None))
        b.force_reset, b.force_goal_reset = p(fr), p(fg)
        b.reset_ids, b.goal_reset_ids, b.counts = p(self._reset_ids), p(self._goal_reset_ids), p(self._counts)
        b.robot_indices, b.reset_root_indices, b.goal_root_indices = p(self._robot_indices), p(self._reset_root_indices), p(self._goal_root_indices)
        b.scan_status, b.control = p(self._scan_status), p(self._control)
        b.torch_rng = p(self._torch_rng)
        b.scale_table = p(self._scale_table)
        b.reward_coef = p(self._reward_coef)
        b.episode_return, b.last_episode_return = p(self._episode_return), p(self._last_episode_return)
        b.last_episode_length, b.last_episode_success = p(self._last_episode_length), p(self._last_episode_success)
        b.episode_stats = p(self._episode_stats)
        b.episode_term_return, b.last_episode_term_return = p(self._episode_term_return), p(self._last_episode_term_return)
        b.episode_term_stats = p(self._episode_term_stats)
        b.obs_bias, b.action_bias = p(self._obs_bias), p(self._action_bias)
        self._B = b
        if not getattr(self, "_history_seeded", False):
            self._call("lg_init_history", self._P, self._S, self._B)  # ref trifinger_env.py:619-628
            self._history_seeded = True

    def _stream(self) -> int:
        return torch.cuda.current_stream(self._torch_device).cuda_stream

    def _call(self, name, P, S, B, *extra):
        fn = getattr(self._lib, name)
        nat.check(fn(P, S, B, *extra, self._stream()), name)

    # -- optional outputs ---------------------------------------------------------------------
    def enable_term_rewards(self, on: bool = True):
        """Also emit each reward term per env ([7, N]) — used by the parity tests."""
        self._term_rewards = (torch.zeros((nat.LG_NUM_TERMS, self.num_instances), device=self._torch_device)
                              if on else None)
        self._bind()
        return self._term_rewards

    def enable_clipped_outputs(self, clip_obs: float = 5.0, clip_actions: Optional[float] = None):
        """Let the fused pass also write clamp(obs/states, +-clip_obs) and clamp the incoming action:
        what VecTaskPython does with three extra ATen passes (ref wrappers/vec_task.py:146-170)."""
        dev = self._torch_device
        self._obs_clipped = torch.zeros_like(self._obs_buf)
        self._states_clipped = torch.zeros_like(self._states_buf) if self.config["asymmetric_obs"] else None
        self._P.clip_obs = float(clip_obs)
        if clip_actions is not None:
            self._P.clip_actions, self._P.clip_input_actions = float(clip_actions), 1
        self._bind()

    def set_forced_resets(self, reset_mask: Optional[torch.Tensor] = None, goal_reset_mask: Optional[torch.Tensor] = None):
        """Masks OR-ed into `_reset_buf` / `_goal_reset_buf` at the start of every following step, inside the
        pre-physics pass itself — what `env._reset_buf |= mask` between steps does (tests, reset-heavy workloads),
        without a separate pass over the flags.  [N] bool device tensors, kept alive here; None switches one off."""
        for m in (reset_mask, goal_reset_mask):
            if m is not None and (m.dtype != torch.bool or m.device != self._torch_device or m.numel() != self.num_instances
                                  or not m.is_contiguous()):
                raise ValueError("forced-reset masks must be contiguous [num_instances] bool tensors on the env's device")
        self._force_masks = (reset_mask, goal_reset_mask)
        self._B.force_reset = nat.ptr(reset_mask)
        self._B.force_goal_reset = nat.ptr(goal_reset_mask)

    def enable_bf16_outputs(self):
        """Also emit bfloat16 copies of the (clipped, when enabled) observations and states from the same pass, for
        policy / value networks that run in bf16 (SURVEY.md §8 f2): round-to-nearest-even, i.e. bit-identical to
        `.to(torch.bfloat16)` of the fp32 outputs, without the extra read-convert-write pass."""
        self._obs_bf16 = torch.zeros(self._obs_buf.shape, device=self._torch_device, dtype=torch.bfloat16)
        self._states_bf16 = (torch.zeros(self._states_buf.shape, device=self._torch_device, dtype=torch.bfloat16)
                             if self.config["asymmetric_obs"] else None)
        self._bind()
        return self._obs_bf16, self._states_bf16

    def enable_host_outputs(self, clip_obs: Optional[float] = None, clip_actions: Optional[float] = None):
        """Zero-copy result path for a HOST-side learner or simulator: the fused kernels store what the
        caller reads every step — (clipped) obs and states, reward, dones, applied torque — straight into
        pinned host memory over PCIe, as part of the same pass, instead of a device buffer plus a
        device-to-host copy.  The returned tensors are then pinned CPU tensors, valid once the stream is
        synchronised.  Un-clipped obs/states stay device resident when clipping is on."""
        pin = lambda t: torch.zeros(t.shape, dtype=t.dtype).pin_memory()  # noqa: E731
        if clip_obs is not None:
            self._P.clip_obs = float(clip_obs)
            self._obs_clipped = pin(self._obs_buf)
            self._states_clipped = pin(self._states_buf) if self.config["asymmetric_obs"] else None
        else:
            self._obs_buf = pin(self._obs_buf)
            self._states_buf = pin(self._states_buf)
        if clip_actions is not None:
            self._P.clip_actions, self._P.clip_input_actions = float(clip_actions), 1
        self._reward_buf = pin(self._reward_buf)
        self._dones = pin(self._dones)
        self._applied_torque = pin(self._applied_torque)
        self._host_io = True
        self._bind()

    def inject_draws(self, reset=None, goal=None):
        """Test hook: the next reset / goal reset reads these (uniforms [k,24], normals [k,8])
        instead of the Philox stream; rows are indexed by ascending-id rank."""
        if self.config["rng_stream"] == "torch" and (reset is not None or goal is not None):
            raise ValueError('inject_draws: with rng_stream "torch" the resets draw torch\'s stream, not injected arrays')
        dev = self._torch_device
        self._inject = {}
        for kind, pair in (("reset", reset), ("goal", goal)):
            if pair is not None:
                def up(a, cols):
                    a = np.nan_to_num(np.asarray(a, dtype=np.float32)).reshape(-1, cols)
                    if a.shape[0] == 0:  # an empty list still needs a valid device pointer
                        a = np.zeros((1, cols), np.float32)
                    return torch.as_tensor(a, device=dev).contiguous()
                self._inject[kind] = (up(pair[0], nat.LG_INJECT_U_COLS), up(pair[1], nat.LG_INJECT_N_COLS))
        self._apply_injection()

    def _apply_injection(self):
        b = self._B
        r, g = self._inject.get("reset"), self._inject.get("goal")
        b.inject_reset_u, b.inject_reset_n = (nat.ptr(r[0]), nat.ptr(r[1])) if r else (None, None)
        b.inject_goal_u, b.inject_goal_n = (nat.ptr(g[0]), nat.ptr(g[1])) if g else (None, None)
        self._P.inject_draws = int(bool(self._inject))

    def _clear_injection(self, kind=None):
        if not self._inject:
            return
        if kind is None:
            self._inject = {}
        else:
            self._inject.pop(kind, None)
        self._apply_injection()

    # -- torch's CUDA generator ("rng_stream": "torch") ------------------------------------------------
    def seed(self, seed: int = None):
        """ref env_base.py:312-320; with "rng_stream": "torch" the env's copy of torch's CUDA generator starts where
        `torch.manual_seed(seed)` leaves the real one: that seed, offset 0.  Without a seed it takes the real one's state."""
        IsaacEnvBase.seed(seed)
        if getattr(self, "_torch_rng", None) is None:
            return
        if seed is None:
            self.load_torch_generator()
        else:
            self._set_torch_rng(int(seed) & 0xFFFFFFFFFFFFFFFF, 0)

    def _torch_generator(self) -> torch.Generator:
        return torch.cuda.default_generators[self._torch_device.index if self._torch_device.index is not None
                                             else torch.cuda.current_device()]

    def _set_torch_rng(self, seed: int, offset: int):
        """Two fill launches with the values as kernel arguments: stream-ordered, no host synchronisation."""
        as_i64 = lambda v: v - (1 << 64) if v >= (1 << 63) else v  # noqa: E731  (uint64 bits in an int64 tensor)
        self._torch_rng[0].fill_(as_i64(seed))
        self._torch_rng[1].fill_(as_i64(offset))

    def torch_rng_state(self) -> Tuple[int, int]:
        """(seed, Philox offset) of the env's stream; synchronises the host."""
        seed, offset = (int(v) & 0xFFFFFFFFFFFFFFFF for v in self._torch_rng[:2].tolist())
        return seed, offset

    def sync_torch_generator(self):
        """Writes the env's stream state into torch's default CUDA generator of the env's device (one host sync): a
        loop that draws its own numbers from that generator between steps then continues the reference's stream."""
        seed, offset = self.torch_rng_state()
        g = self._torch_generator()
        g.manual_seed(seed)
        g.set_offset(offset)

    def load_torch_generator(self):
        """The other way: the env's stream continues from torch's default CUDA generator (no device sync)."""
        g = self._torch_generator()
        self._set_torch_rng(int(g.initial_seed()), int(g.get_offset()))

    # -- public surface -------------------------------------------------------------------------
    def _frame_count(self) -> int:
        return self._sim.get_frame_count()

    def _global_num_instances(self) -> int:
        return self._global_N

    def _simulate(self):
        self._sim.simulate()
        if getattr(self._sim, "rebinds_tensors", False):  # zero-copy simulators hand out a new set of tensors
            s, p = self._sim, nat.ptr
            self._S = nat.LgSimState(p(s.dof_state), p(s.root_state), p(s.rigid_body), p(s.dof_force), p(s.ft_sensors))
            N = self.num_instances
            self._dof_state = s.dof_state.view(N, 9, 2)
            self._rigid_body_state = s.rigid_body.view(N, s.bodies_per_env, 13)
            self._actors_root_state = s.root_state.view(-1, 13)

    @property
    def reset_env_ids(self) -> torch.Tensor:
        """Ascending ids reset by the last step (what `torch.nonzero(_reset_buf)` gave the reference,
        env_base.py:374).  Reading it synchronises the host; the step itself does not."""
        return self._reset_ids[: int(self._counts[0])]

    @property
    def goal_reset_env_ids(self) -> torch.Tensor:
        return self._goal_reset_ids[: int(self._counts[1])]

    def step(self, action):
        """Fused step: lg_pre_physics -> simulator -> lg_post_physics; no host synchronisation."""
        action = self._check_action(action)
        self._P.fuse_bookkeeping = 1
        nat.check(self._lib.lg_pre_physics(self._P, self._S, self._B, action.data_ptr(), self._stream()), "lg_pre_physics")
        self._clear_injection()
        self._notify_resets()
        self._sim.set_dof_actuation_force_tensor(self._applied_torque)
        self._notify_goal_movement()
        for _ in range(self.control_decimation):
            self._simulate()
        self._call("lg_post_physics", self._P, self._S, self._B, float(self.env_steps_count))
        self._step_info = self._make_info()
        return self._obs_buf, self._reward_buf, self._dones, self._step_info

    # -- episode statistics (extension, "episode_statistics": {"activate": True}; None when off) --------------------
    # An episode ends when the env is reset by any route: timeout, a flag set between steps or a forced mask, `reset()`,
    # `_reset_impl`.  A goal reset (success termination) does not end it.  The reset moves the running return, the
    # step count and `_successes` into the env's record; the first step after it reports the episode in `info`
    # (env/episodes/*).  The reset happens at the start of the next step, so an episode that times out at step t is
    # reported by step t + 1.
    @property
    def episode_return(self) -> Optional[torch.Tensor]:
        """[N] fp32: sum of the rewards of each env's running episode, success bonus included."""
        return self._episode_return

    @property
    def last_episode_return(self) -> Optional[torch.Tensor]:
        """[N] fp32: return of each env's last finished episode."""
        return self._last_episode_return

    @property
    def last_episode_length(self) -> Optional[torch.Tensor]:
        """[N] int64: its length in steps; 0 while the env has finished none."""
        return self._last_episode_length

    @property
    def last_episode_success(self) -> Optional[torch.Tensor]:
        """[N] bool: `_successes` at the moment it ended."""
        return self._last_episode_success

    # -- per-term episode returns (extension, "episode_term_returns": {"activate": True}; None when off) -----------
    # Column k < 7 of a row is reward term k (nat.TERM_NAMES), column 7 the success bonus (EPISODE_TERM_NAMES).  Each
    # step adds what the reward added: the value of every active term (what `term_rewards` shows) and the bonus when
    # success termination pays it; inactive terms stay 0.  The same resets that end an episode move the row into the
    # record, and the step that reports the episode adds the record into env/episodes/return_sum/<term>.
    EPISODE_TERM_NAMES = nat.EPISODE_TERM_NAMES

    @property
    def episode_term_return(self) -> Optional[torch.Tensor]:
        """[N, 8] fp32: each env's running episode return split by term (EPISODE_TERM_NAMES)."""
        return self._episode_term_return

    @property
    def last_episode_term_return(self) -> Optional[torch.Tensor]:
        """[N, 8] fp32: the same for each env's last finished episode."""
        return self._last_episode_term_return

    def _episode_term_slots(self) -> list:
        """Names of the slots that can be nonzero: the active reward terms and, with success termination, the bonus."""
        names = [n for n in nat.TERM_NAMES if self.config["reward_terms"].get(n, {}).get("activate")]
        if self.config["termination_conditions"]["success"]["activate"]:
            names.append("success_bonus")
        return names

    # -- per-episode DR offsets (extension, "domain_randomization": obs_bias_std / action_bias_std; None when off) --
    # Every reset of an env but a goal-only one (a timeout, a flag or forced mask, `reset()`, `_reset_impl`) draws its
    # rows anew: sigma x N(0, 1) per column from this build's Philox stream, whatever "rng_stream" says, and 0 where
    # sigma is 0.  An env never reset holds zeros; `reset()` draws every row.  The actor observation sees
    # scale_transform((raw + obs_bias) + noise); states, rewards and statistics see the clean values.  The stored
    # action is clamp((action + action_bias) + noise).
    @property
    def obs_bias(self) -> Optional[torch.Tensor]:
        """[N, obs_dim] fp32: each env's offset of the raw observation columns for its running episode."""
        return self._obs_bias

    @property
    def action_bias(self) -> Optional[torch.Tensor]:
        """[N, action_dim] fp32: each env's offset of the (normalised) action for its running episode."""
        return self._action_bias

    # -- checkpoint / resume (SURVEY.md §8 f4; the reference only dumps its config, env_base.py:295-309) ------
    def state_dict(self) -> dict:
        from .checkpoint import env_state_dict
        return env_state_dict(self)

    def load_state_dict(self, state: dict) -> None:
        from .checkpoint import load_env_state_dict
        load_env_state_dict(self, state)

    def save_checkpoint(self, path: str) -> str:
        """Everything the MDP carries between steps (and SyntheticSim's tensors) into one .npz; returns the path."""
        from .checkpoint import save_env_state
        return save_env_state(self, path)

    def load_checkpoint(self, path: str) -> None:
        """Continue bit-identically from `save_checkpoint` (same config, shard geometry and simulator sequence)."""
        from .checkpoint import load_env_state
        load_env_state(self, path)

    def _make_info(self) -> Dict[str, torch.Tensor]:
        """`_step_info` of the reference (trifinger_env.py:554, :1068, :1076, :1099) as 0-d fp64 views
        of the per-step statistics buffer: valid until the next step overwrites them; values are
        this shard's (see global_step_info)."""
        views = getattr(self, "_info_views", None)
        if views is None or views[0] is not self._step_stats:   # the views never change: build them once
            buf, info = self._step_stats, {}
            for i, name in enumerate(nat.TERM_NAMES):
                if self.config["reward_terms"].get(name, {}).get("activate"):
                    info[f"env/rewards/{name}"] = buf[i]
            info["env/current_position_goal/count"] = buf[nat.STAT_POSITION_GOAL]
            info["env/current_orientation_goal/count"] = buf[nat.STAT_ORIENTATION_GOAL]
            info["env/average_consecutive_success"] = buf[nat.STAT_SUCCESSES]
            ep = self._episode_stats
            if ep is not None:   # episodes reported by this step (sums over this shard)
                for i, key in enumerate(EPISODE_KEYS):
                    info[key] = ep[i]
            ts = self._episode_term_stats
            if ts is not None:   # ... and their returns, split by term
                for name in self._episode_term_slots():
                    info[f"env/episodes/return_sum/{name}"] = ts[nat.EPISODE_TERM_NAMES.index(name)]
            views = self._info_views = (buf, info)
        return dict(views[1])

    def global_step_info(self) -> Dict[str, float]:
        """Whole-job statistics: all-reduces the 16 shard sums (the only cross-GPU traffic of the
        path, SURVEY.md §8e) and divides by the global env count.  With episode statistics on, their four
        sums (and, with per-term returns on, their eight) go in the same all-reduce.  Synchronises the host."""
        from .distributed import all_reduce_stats, stats_to_info
        active = [k for k, v in self.config["reward_terms"].items() if v["activate"]]
        if self._episode_stats is None:
            stats = all_reduce_stats(self._step_stats, self.num_instances, self._global_N)
            return stats_to_info(stats, active)
        # one all-reduce for both vectors; adds the job-wide episode sums and, when episodes ended, their means
        if self._episode_term_stats is None:
            stats, episodes = all_reduce_stats(self._step_stats, self.num_instances, self._global_N,
                                               episode_stats=self._episode_stats)
            return stats_to_info(stats, active, episode_stats=episodes)
        stats, episodes, terms = all_reduce_stats(self._step_stats, self.num_instances, self._global_N,
                                                  episode_stats=self._episode_stats,
                                                  episode_term_stats=self._episode_term_stats)
        return stats_to_info(stats, active, episode_stats=episodes, episode_term_stats=terms,
                             episode_terms=self._episode_term_slots())

    # -- hooks, individually callable (ref trifinger_env.py:373-559, :959-994) ---------------------
    def _reset_impl(self, instances: torch.Tensor):
        ids = instances.to(self._torch_device, dtype=torch.long).contiguous()
        nat.check(self._lib.lg_reset_envs(self._P, self._S, self._B, ids.data_ptr(), ids.numel(), self._stream()),
                  "lg_reset_envs")
        self._clear_injection("reset")
        k = ids.numel()
        self._sim.set_dof_state_tensor_indexed(self._robot_indices[:k], k)
        self._sim.set_actor_root_state_tensor_indexed(self._reset_root_indices[:3 * k], 3 * k)

    def _goal_reset_impl(self, instances: torch.Tensor):
        ids = instances.to(self._torch_device, dtype=torch.long).contiguous()
        nat.check(self._lib.lg_goal_reset_envs(self._P, self._S, self._B, ids.data_ptr(), ids.numel(), self._stream()),
                  "lg_goal_reset_envs")
        self._clear_injection("goal")
        k = ids.numel()
        self._sim.set_actor_root_state_tensor_indexed(self._goal_root_indices[:k], k)

    def _pre_step(self):
        self._call("lg_pre_step", self._P, self._S, self._B)
        self._sim.set_dof_actuation_force_tensor(self._applied_torque)
        self._notify_goal_movement()

    def _notify_resets(self):
        """Tell the simulator which rows the pre-physics pass rewrote — what `_reset_impl` / `_goal_reset_impl` end
        with in the reference (`set_dof_state_tensor_indexed`, `set_actor_root_state_tensor_indexed`,
        trifinger_env.py:413-423, :435-440), in the same order.  The index lists and their lengths stay on the
        device (`LazyCount`): the step itself never synchronises; an adapter that needs a host integer calls
        `int(count)`.  Unlike the reference the calls are made every step, also when nothing was reset (count 0)."""
        n_reset = LazyCount(self._counts[0])
        self._sim.set_dof_state_tensor_indexed(self._robot_indices, n_reset)
        self._sim.set_actor_root_state_tensor_indexed(self._reset_root_indices, LazyCount(self._counts[0], 3))
        self._sim.set_actor_root_state_tensor_indexed(self._goal_root_indices, LazyCount(self._counts[1]))

    def _notify_goal_movement(self):
        """Moving goal (ref trifinger_env.py:1267-1277): the kernels re-imposed every goal body's angular velocity;
        tell the simulator which root rows changed (all goal actors, every step)."""
        if self._P.goal_rotation:
            if getattr(self, "_all_goal_indices", None) is None:
                apa, slot = self._sim.actors_per_env, self._sim.slots[2]
                self._all_goal_indices = (torch.arange(self.num_instances, device=self._torch_device, dtype=torch.int32)
                                          * apa + slot)
            self._sim.set_actor_root_state_tensor_indexed(self._all_goal_indices, self.num_instances)

    def _post_step(self):
        self._P.fuse_bookkeeping = 0
        try:
            self._call("lg_post_physics", self._P, self._S, self._B, float(self.env_steps_count))
        finally:
            self._P.fuse_bookkeeping = 1
        self._step_info = self._make_info()

    def _fill_observations_and_states(self):
        self._call("lg_fill_observations", self._P, self._S, self._B)
