"""The torch-stream extension ("rng_stream": "torch") on the GPU: the primitive equals torch.rand / torch.randn on
this device bit for bit, the hooks sample what the oracle samples when it makes the reference's calls on the CUDA
generator, the fused step equals the hook-by-hook step, and checkpoints carry the stream."""
import numpy as np
import pytest
import torch

from tolerances import compare

pytestmark = pytest.mark.gpu

SIZES = [1, 3, 4, 255, 256, 257, 4099, 16384, 18 * 16384, 303104, 303105, 18 * 65536, 1212416, 1212417, 18 * 262144]


def _bits(t):
    return t.contiguous().view(torch.int32).cpu()


@pytest.mark.parametrize("offset", [0, 4, (1 << 34) + 8])
@pytest.mark.parametrize("normal", [0, 1])
def test_primitive_equals_torch(offset, normal):
    from leibnizgym_b200 import _native
    lib = _native.load()
    props = torch.cuda.get_device_properties(0)
    seed = 0x1234_5678_9ABC
    stream = torch.cuda.current_stream().cuda_stream
    for n in SIZES:
        g = torch.Generator(device="cuda")
        g.manual_seed(seed)
        g.set_offset(offset)
        ref = (torch.randn if normal else torch.rand)(n, device="cuda", generator=g)
        out = torch.empty(n, device="cuda")
        _native.check(lib.lg_torch_philox(seed, offset, n, normal, out.data_ptr(), stream), "lg_torch_philox")
        assert torch.equal(_bits(out), _bits(ref)), (n, offset, normal)
        adv = lib.lg_torch_philox_advance(n, props.multi_processor_count, props.max_threads_per_multi_processor)
        assert g.get_offset() - offset == adv, (n, offset)


def _gpu_draws():
    from oracle.trifinger_oracle import Draws, F32

    class GpuDraws(Draws):
        """The reference's calls made on the CUDA device (use_gpu_pipeline), results moved to the CPU."""

        def uniform(self, k, cols):
            if self.u is not None:
                return super().uniform(k, cols)
            return torch.rand(k if isinstance(cols, int) else (k, len(cols)), dtype=F32, device="cuda").cpu()

        def normal(self, k, cols):
            if self.n is not None:
                return super().normal(k, cols)
            return torch.randn((k, len(cols)), dtype=F32, device="cuda").cpu()

    return GpuDraws()


def _cfg(N, difficulty=4, robot="random", obj="random", rot=True, seed=11, asym=False):
    return {"command_mode": "torque", "num_instances": N, "seed": seed, "rng_stream": "torch", "asymmetric_obs": asym,
            "task_difficulty": difficulty, "episode_length": 1000,
            "reset_distribution": {"robot_initial_state": {"type": robot, "dof_pos_stddev": 0.4, "dof_vel_stddev": 0.2},
                                   "object_initial_state": {"type": obj}},
            "goal_movement": {"rotation": {"activate": rot, "rate_magnitude": 0.5}}}


def _env(cfg, seq_seed=3, T=4):
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    seq = make_sequence(seq_seed, T, cfg["num_instances"])
    return TrifingerEnv(cfg, device="cuda:0", verbose=False, sim=SyntheticSim(seq.to("cuda:0"), "cuda:0")), seq


def _close(key, got, exp, where):
    ok, detail = compare(key, got.cpu().numpy(), exp.numpy())
    assert ok, (where, key, detail)


CONFIGS = [(-1, "random", "random", False), (1, "default", "random", False), (2, "random", "none", True),
           (3, "random", "default", False), (4, "random", "random", True), (5, "default", "random", False),
           (6, "none", "none", True), (6, "random", "random", False)]


@pytest.mark.parametrize("difficulty, robot, obj, rot, policy_draws",
                         [c + (False,) for c in CONFIGS] + [CONFIGS[0] + (True,), CONFIGS[4] + (True,)])
def test_hooks_match_oracle_drawing_on_gpu(difficulty, robot, obj, rot, policy_draws):
    """No injection: both sides draw torch's CUDA stream from the same seed.  Joint rows bit-exact, poses within the
    parity tolerances, the stream offset equal after every round (also with a policy drawing in between)."""
    from leibnizgym_b200.config import resolve_config
    from oracle.trifinger_oracle import OracleEnv, OracleSim
    N = 384
    cfg = _cfg(N, difficulty, robot, obj, rot)
    env, seq = _env(cfg)
    ora = OracleEnv(resolve_config(cfg), OracleSim(seq, N))   # torch.manual_seed(seed), like the env's seed()
    ora.draw = _gpu_draws()
    gen = torch.cuda.default_generators[0]
    rng = np.random.default_rng(difficulty + 10)
    apa = env._sim.actors_per_env
    for rnd in range(21):
        ids = np.arange(N) if rnd == 0 else np.flatnonzero(rng.random(N) < 0.3)
        gids = np.array([], np.int64) if rnd == 0 else np.flatnonzero(rng.random(N) < 0.05)
        for hook_env, hook_ora, lst in ((env._reset_impl, ora.reset_impl, ids), (env._goal_reset_impl, ora.goal_reset_impl, gids)):
            if len(lst):   # the reference calls a hook only for a non-empty list (env_base.py:374-379)
                hook_env(torch.as_tensor(lst, device="cuda"))
                hook_ora(torch.as_tensor(lst))
        w = (difficulty, robot, obj, rot, rnd)
        if len(ids):   # reset kind "none" leaves the rows alone (and the two simulators start from different rows)
            t = torch.as_tensor(ids)
            if robot != "none":
                assert torch.equal(_bits(env._dof_state[t.cuda()]), _bits(ora.sim.dof[t])), w
            if obj != "none":
                _close("pre_sim_obj_root", env._actors_root_state[(t * apa + 2).cuda()], ora.sim.root[t * apa + 2], w)
        _close("goal_pose", env._object_goal_poses_buf, ora.goal_poses, w)
        _close("goal_movement", env._object_goal_movement_buf, ora.goal_movement, w)
        assert env.torch_rng_state() == (cfg["seed"], gen.get_offset()), w
        if policy_draws:
            env.sync_torch_generator()
            torch.randn(N, 9, device="cuda")       # the policy's noise from the global generator
            env.load_torch_generator()


def _masks(N, T, p, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.rand(N, generator=g) < p).cuda() for _ in range(T)]


def _compare_envs(a, b, where):
    for name in ("_dof_state", "_applied_torque", "_object_goal_poses_buf", "_object_goal_movement_buf", "_history",
                 "_obs_buf", "_states_buf", "_reward_buf", "_reset_buf", "_goal_reset_buf", "_steps_count_buf"):
        x, y = getattr(a, name), getattr(b, name)
        assert torch.equal(x.contiguous().view(torch.uint8), y.contiguous().view(torch.uint8)), (where, name)
    assert a.torch_rng_state() == b.torch_rng_state(), where


@pytest.mark.parametrize("N, p", [(1024, 0.3), (12336, 0.3), (16384, 0.3), (262144, 0.3), (65536, 1.0), (262144, 1.0)])
def test_fused_step_equals_hooks(N, p):
    """Look-back (1024), direct prefix (16384, ragged 12336) and ticket (262144) grids; p = 1: every env resets, where
    rand(k, 18) leaves the one-round regime."""
    from leibnizgym_b200.env import IsaacEnvBase
    cfg = _cfg(N, difficulty=4, rot=True, asym=True)
    fused, seq = _env(cfg)
    hooks, _ = _env(cfg)
    T = 3
    rmask, gmask = _masks(N, T, p, 5), _masks(N, T, 0.05, 6)
    for t in range(T):
        fused._reset_buf |= rmask[t]
        fused._goal_reset_buf |= gmask[t]
        hooks._reset_buf |= rmask[t]
        hooks._goal_reset_buf |= gmask[t]
        a = seq.action[t].cuda()
        k_r, k_g = int(hooks._reset_buf.sum()), int(hooks._goal_reset_buf.sum())
        r_ids = torch.nonzero(hooks._reset_buf).view(-1)
        fused.step(a)
        IsaacEnvBase.step(hooks, a)
        assert torch.equal(fused.reset_env_ids, r_ids), (N, t)
        assert int(fused._counts[1]) == k_g
        assert torch.equal(fused._robot_indices[:k_r], hooks._robot_indices[:k_r]), (N, t)
        assert torch.equal(fused._reset_root_indices[:3 * k_r], hooks._reset_root_indices[:3 * k_r]), (N, t)
        assert torch.equal(fused._goal_root_indices[:k_g], hooks._goal_root_indices[:k_g]), (N, t)
        _compare_envs(fused, hooks, (N, t))


def test_checkpoint_carries_the_stream(tmp_path):
    N = 2048
    cfg = _cfg(N, difficulty=5)
    env, seq = _env(cfg)
    masks = _masks(N, 6, 0.3, 9)
    for t in range(3):
        env._reset_buf |= masks[t]
        env.step(seq.action[t % 4].cuda())
    path = env.save_checkpoint(str(tmp_path / "ck"))
    state = env.torch_rng_state()
    assert state[1] > 0
    resumed, _ = _env(cfg)
    resumed.load_checkpoint(path)
    assert resumed.torch_rng_state() == state
    for t in range(3, 6):
        for e in (env, resumed):
            e._reset_buf |= masks[t]
            e.step(seq.action[t % 4].cuda())
        _compare_envs(env, resumed, t)


def _runner_pair(N, R, chain, reset_p):
    """Two envs on their own copies of one ring: `fused` stepped by GraphRunner (captured graph, replayed), `hooks` stepped
    on the same per-slot buffers by the hook-by-hook sequence of env_base.py:369-381 (action store, lg_reset_envs,
    lg_goal_reset_envs, lg_pre_step), then the same lg_post_physics."""
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence
    cfg = _cfg(N, difficulty=4, rot=True, asym=True)
    cfg["episode_length"] = 5   # timeouts raise flags inside the run as well
    rm = bernoulli_masks(31, R, N, reset_p, device="cuda:0")
    gm = bernoulli_masks(32, R, N, 0.05, device="cuda:0")
    out = []
    for forced in (True, False):
        ring = make_sequence(30, R, N, device="cuda:0")
        env = TrifingerEnv(cfg, device="cuda:0", verbose=False, sim=SyntheticSim(ring, "cuda:0"))
        env.reset()
        runner = GraphRunner(env, ring, rotate_outputs=True, device_clock=False, chain_pre=chain,
                             inject_reset_masks=rm if forced else None, inject_goal_masks=gm if forced else None)
        out.append((env, runner, ring))
    return out, rm, gm


def _hook_step(env, runner, t, rm, gm):
    lib, st = env._lib, torch.cuda.current_stream().cuda_stream
    s, prev = t % runner.R, (t - 1) % runner.R
    P, S, B = runner.P, runner._S[prev], runner._B[prev]
    env._reset_buf |= rm[s]
    env._goal_reset_buf |= gm[s]
    env._action_buf.copy_(runner.ring.action[s])
    ids = torch.nonzero(env._reset_buf).view(-1)
    gids = torch.nonzero(env._goal_reset_buf).view(-1)
    for fn, lst in (("lg_reset_envs", ids), ("lg_goal_reset_envs", gids)):
        if len(lst):
            nat_check(getattr(lib, fn)(P, S, B, lst.data_ptr(), lst.numel(), st), fn)
    nat_check(lib.lg_pre_step(P, S, B, st), "lg_pre_step")
    sched = float((runner.frame0 + (t - runner.t0) + 1) * env._global_N)
    nat_check(lib.lg_post_physics(P, runner._S[s], runner._B[s], sched, st), "lg_post_physics")
    return ids, gids


def nat_check(rc, what):
    from leibnizgym_b200 import _native
    _native.check(rc, what)


@pytest.mark.parametrize("N, chain", [(1024, True), (16384, True), (16384, False), (262144, False)])
def test_graph_replay_equals_hooks(N, chain):
    """GraphRunner capture + replay in torch mode (counting launch captured, chained pre-physics falling back to stream
    order, per-slot force masks, the counting workspace re-armed across replays) against the hook-by-hook sequence on
    the same buffers: ids, index lists, joint rows, goal poses, obs / states / reward and the stream offset."""
    R = 4
    pair, rm, gm = _runner_pair(N, R, chain, 0.3)
    (fe, fr, fring), (he, hr, hring) = pair
    fr.capture(R)                 # two eager warm-up steps (t = 0, 1), then steps 0..R-1 captured
    fr.replay(2)
    order = [0, 1] + list(range(R)) * 2
    for t in order:
        ids, gids = _hook_step(he, hr, t, rm, gm)
    torch.cuda.synchronize()
    k, kg = int(fe._counts[0]), int(fe._counts[1])
    assert (k, kg) == (len(ids), len(gids)) and k > 0
    assert torch.equal(fe._reset_ids[:k], ids) and torch.equal(fe._goal_reset_ids[:kg], gids)
    assert torch.equal(fe._robot_indices[:k], he._robot_indices[:k])
    assert torch.equal(fe._reset_root_indices[:3 * k], he._reset_root_indices[:3 * k])
    assert torch.equal(fe._goal_root_indices[:kg], he._goal_root_indices[:kg])
    for a, b, what in ((fr.obs_slots, hr.obs_slots, "obs"), (fr.state_slots, hr.state_slots, "states"),
                       (fring.dof_state, hring.dof_state, "joint rows"), (fring.root_state, hring.root_state, "root rows"),
                       (fe._object_goal_poses_buf, he._object_goal_poses_buf, "goal poses"),
                       (fe._object_goal_movement_buf, he._object_goal_movement_buf, "goal movement"),
                       (fe._reward_buf, he._reward_buf, "reward"), (fe._history, he._history, "history"),
                       (fe._applied_torque, he._applied_torque, "torque"), (fe._reset_buf, he._reset_buf, "flags"),
                       (fe._goal_reset_buf, he._goal_reset_buf, "goal flags"), (fe._action_buf, he._action_buf, "action")):
        assert torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8)), (N, chain, what)
    assert fe.torch_rng_state() == he.torch_rng_state() and fe.torch_rng_state()[1] > 0
    assert int(fe._torch_rng[4]) == 0 and int(fe._torch_rng[5]) & 0xFFFFFFFF == 0   # counting workspace re-armed


def test_host_buffer_step_equals_eager_step():
    """lg_step_host (simulator state and outputs in pinned host memory) in torch mode against env.step."""
    from leibnizgym_b200 import _native
    N, T = 4096, 3
    cfg = _cfg(N, difficulty=5, rot=False, asym=True)
    ref, seq = _env(cfg)
    host, _ = _env(cfg)
    masks = _masks(N, T, 0.3, 12)
    pin = lambda x: x.cpu().contiguous().pin_memory()  # noqa: E731
    lib, st = host._lib, torch.cuda.current_stream().cuda_stream
    od, sd = host.get_obs_dim(), host.get_state_dim()
    obs_h, st_h, rew_h = (torch.zeros(N, od).pin_memory(), torch.zeros(N, sd).pin_memory(), torch.zeros(N).pin_memory())
    staging = torch.zeros(N, 9, device="cuda")
    for t in range(T):
        ref._reset_buf |= masks[t]
        host._reset_buf |= masks[t]
        a = seq.action[t]
        ref.step(a.cuda())
        f = host._sim.begin_step()      # the state the simulator produces for this step
        frame = [pin(x[f]) for x in (seq.dof_state, seq.root_state, seq.rigid_body, seq.dof_force, seq.ft_sensors)]
        act = pin(a)
        H = _native.LgHostStep()
        H.dof_state_host, H.root_state_host, H.rigid_body_host, H.dof_force_host, H.ft_sensors_host = (
            x.data_ptr() for x in frame)
        H.action_host, H.action_staging = act.data_ptr(), staging.data_ptr()
        H.obs_host, H.states_host, H.reward_host = obs_h.data_ptr(), st_h.data_ptr(), rew_h.data_ptr()
        _native.check(lib.lg_step_host(host._P, host._S, host._B, H, float(host.env_steps_count), st), "lg_step_host")
        torch.cuda.synchronize()
        assert torch.equal(host.reset_env_ids, ref.reset_env_ids), t
        for a_, b_, what in ((obs_h, ref._obs_buf, "obs"), (st_h, ref._states_buf, "states"), (rew_h, ref._reward_buf, "reward"),
                             (host._object_goal_poses_buf, ref._object_goal_poses_buf, "goal poses"),
                             (host._applied_torque, ref._applied_torque, "torque"), (host._history, ref._history, "history")):
            assert torch.equal(_bits(a_), _bits(b_)), (t, what)
        assert host.torch_rng_state() == ref.torch_rng_state(), t


def test_torch_stream_refuses_injection_and_mixed_checkpoints(tmp_path):
    cfg = _cfg(256)
    env, _ = _env(cfg)
    with pytest.raises(ValueError, match="injected"):
        env.inject_draws(reset=(np.zeros((256, 24)), np.zeros((256, 8))))
    path = env.save_checkpoint(str(tmp_path / "torch_mode"))
    cfg["rng_stream"] = "philox"
    other, _ = _env(cfg)
    with pytest.raises(ValueError, match="rng_stream"):
        other.load_checkpoint(path)
