"""Per-episode domain-randomisation offsets (extension, "domain_randomization": obs_bias_std / action_bias_std) on the
GPU: off is bit-identical, the offsets are applied exactly where the contract puts them, redrawn by resets only, have
the stated distribution and keying, never touch the reset samples, and every route that steps the env agrees."""
import copy

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SUCCESS = {"success": {"activate": True, "bonus": 5000.0, "position_tolerance": 0.12, "orientation_tolerance": 1.5}}
ALL = {"robot_q": 0.01, "robot_u": 0.05, "object_q": 0.003, "object_q_des": 0.002, "command": 0.02}
WHITE = {"robot_q": 0.005, "robot_u": 0.05, "object_q": 0.002, "object_q_des": 0.0, "command": 0.0}
GROUPS = {"robot_q": (0, 9), "robot_u": (9, 18), "object_q": (18, 25), "object_q_des": (25, 32), "command": (32, 41)}


def _cfg(N, asym=True, obs=None, act=0.0, white=False, keys=True, episode_length=5, **extra):
    from leibnizgym_b200.config import difficulty_config
    cfg = difficulty_config(4, N, asymmetric_obs=asym, seed=3, episode_length=episode_length,
                            termination_conditions=copy.deepcopy(SUCCESS))
    dr = {"activate": True, "obs_noise_std": dict(WHITE if white else {k: 0.0 for k in WHITE}),
          "action_noise_std": 0.02 if white else 0.0}
    if keys:
        dr["obs_bias_std"] = dict(obs or {})
        dr["action_bias_std"] = act
    cfg["domain_randomization"] = dr
    cfg["episode_statistics"] = {"activate": True}
    cfg.update(extra)
    return cfg


def _env(cfg, seq=None, T=8, rank=0, world=1):
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    if seq is None:
        seq = make_sequence(21, T, cfg["num_instances"])
    env = TrifingerEnv(cfg, device=DEV, verbose=False, sim=SyntheticSim(seq.to(DEV), DEV), rank=rank, world_size=world)
    return env, seq


def _masks(N, T, p, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.rand(N, generator=g) < p).to(DEV) for _ in range(T)]


def _bits(t):
    return t.detach().contiguous().view(torch.uint8).cpu()


SUMS = ("_step_stats", "_episode_stats")   # fp64 sums by atomics in any order: equal up to the last bits


def _same(a, b, f):
    if f in SUMS:
        return torch.allclose(a, b, rtol=1e-12, atol=1e-12)
    return torch.equal(_bits(a), _bits(b))


def _ticket_size():
    from leibnizgym_b200 import _native
    lib = _native.load()
    tile = (1 << 20) // int(lib.lg_scan_tiles(1 << 20))
    return (int(lib.lg_pre_resident_tiles()) + 3) * tile + 5


CLEAN = ("_states_buf", "_reward_buf", "_history", "_step_stats", "_successes", "_reset_buf", "_goal_reset_buf",
         "_dones", "_steps_count_buf", "_episode_return", "_last_episode_return", "_last_episode_length",
         "_episode_stats", "_object_goal_poses_buf")
OUTPUTS = ("_obs_buf", "_obs_clipped", "_obs_bf16", "_states_clipped", "_states_bf16", "_action_buf") + CLEAN


def _run(cfg, T, forced, goal_forced, seq, probe=None):
    env, _ = _env(cfg, seq=seq)
    env.enable_clipped_outputs(5.0, 1.0)
    env.enable_bf16_outputs()
    env.reset()
    for t in range(T):
        env.set_forced_resets(forced[t] if t % 3 == 2 else None, goal_forced[t])
        before = None if probe is None else probe.before(env)
        env.step(seq.action[t % seq.num_steps].to(DEV) * 1.3)
        if probe is not None:
            probe.after(env, before, t)
        yield env


def _raw_obs(env):
    """The raw actor observation the post-physics pass reads (trifinger_env.py:959-987)."""
    N, A = env.num_instances, env.get_action_dim()
    dof = env._dof_state.reshape(N, 18)
    obj = env._actors_root_state.view(N, -1, 13)[:, env._sim.slots[1], 0:7]
    return torch.cat([dof[:, 0::2], dof[:, 1::2], obj, env._object_goal_poses_buf, env._action_buf.view(N, A)], dim=1)


def _scale(env, x):
    od = x.shape[1]
    c = torch.tensor(list(env._P.scale_centre)[:od], device=DEV, dtype=torch.float32)
    s = torch.tensor(list(env._P.scale_span)[:od], device=DEV, dtype=torch.float32)
    return (2.0 * (x - c)) / s


@pytest.mark.parametrize("asym", [True, False])
@pytest.mark.parametrize("N", [16384, 4099, "ticket"])
def test_off_is_bit_identical_and_on_is_exact(N, asym):
    """Keys at 0 (white noise on) equal the run without the keys, output for output.  Offsets on every group and the
    action (white noise off): obs == scale_transform(raw + obs_bias) bit for bit, the stored action == clamp(a +
    action_bias) (0 for envs reset by the step), everything clean equals the offsets-off run, and exactly the reset
    envs' offset rows change at each step (goal-only resets change nothing)."""
    N = _ticket_size() if N == "ticket" else N
    T = 9
    from leibnizgym_b200.synthetic import make_sequence
    seq = make_sequence(21, T, N)
    forced, goals = _masks(N, T, 0.3, 8), _masks(N, T, 0.05, 9)
    absent = [{f: getattr(e, f).clone() for f in OUTPUTS if getattr(e, f, None) is not None}
              for e in _run(_cfg(N, asym, white=True, keys=False), T, forced, goals, seq)]
    at_zero = _cfg(N, asym, white=True, obs={k: 0.0 for k in ALL}, act=0.0)
    for t, env in enumerate(_run(at_zero, T, forced, goals, seq)):
        assert env.obs_bias is None and env.action_bias is None
        for f in OUTPUTS:
            a, b = absent[t].get(f), getattr(env, f, None)
            if a is not None:
                assert _same(a, b, f), (t, f)
    del absent
    off_runs = [_clone_clean(e) for e in _run(_cfg(N, asym), T, forced, goals, seq)]

    class Probe:
        def before(self, env):
            return env.obs_bias.clone(), env.action_bias.clone()

        def after(self, env, before, t):
            ob0, ab0 = before
            ids = env.reset_env_ids
            reset = torch.zeros(N, dtype=torch.bool, device=DEV)
            reset[ids] = True
            changed = (env.obs_bias != ob0).any(1) | (env.action_bias != ab0).any(1)
            assert torch.equal(changed, reset), t                       # redrawn by resets, by nothing else
            assert int(env._counts[1]) > 0
            exp_act = torch.clamp(seq.action[t % seq.num_steps].to(DEV) * 1.3 + ab0, -1.0, 1.0)
            exp_act[reset] = 0.0
            assert torch.equal(_bits(env._action_buf), _bits(exp_act)), t
            exp_obs = _scale(env, _raw_obs(env) + env.obs_bias)
            assert torch.equal(_bits(env._obs_buf), _bits(exp_obs)), t
            for f in CLEAN:
                if f == "_states_buf" and not asym:
                    continue
                ref = off_runs[t][f]
                if f == "_states_buf":   # its command columns hold the stored action, which the offset moved
                    got = getattr(env, f)
                    od = env.get_obs_dim()
                    assert torch.equal(_bits(got[:, :32]), _bits(ref[:, :32])), t
                    assert torch.equal(_bits(got[:, od:]), _bits(ref[:, od:])), t
                    continue
                assert _same(getattr(env, f), ref, f), (t, f)

    on = _cfg(N, asym, obs=ALL, act=0.05)
    for _ in _run(on, T, forced, goals, seq, probe=Probe()):
        pass


def _clone_clean(env):
    return {f: getattr(env, f).clone() for f in CLEAN if getattr(env, f, None) is not None}


def test_never_reset_is_zero_and_reset_redraws_everything():
    N = 4099
    env, seq = _env(_cfg(N, obs={"object_q": 0.01}, act=0.05))
    assert int(env.obs_bias.abs().sum()) == 0 and int(env.action_bias.abs().sum()) == 0
    env.reset()
    first = (env.obs_bias.clone(), env.action_bias.clone())
    assert bool((env.obs_bias[:, 18:25] != 0).all()) and bool((env.action_bias != 0).all())
    for t in range(3):
        env.step(seq.action[t].to(DEV))
    env.reset()
    assert bool((env.obs_bias[:, 18:25] != first[0][:, 18:25]).all())
    assert bool((env.action_bias != first[1]).all())


def test_distribution():
    from scipy import stats
    from leibnizgym_b200.params import observation_scale
    from leibnizgym_b200.config import resolve_config
    from leibnizgym_b200.synthetic import make_sequence
    N = 120_000
    sig = {"robot_q": 0.01, "robot_u": 0.0, "object_q": 0.003, "object_q_des": 0.002, "command": 0.02}
    seq = make_sequence(51, 3, N)
    seq.action.mul_(0.5)
    env, _ = _env(_cfg(N, obs=sig, act=0.03, white=True, episode_length=None), seq=seq)
    env.reset()
    b1 = env.obs_bias.double().cpu().numpy()
    a1 = env.action_bias.double().cpu().numpy()
    for name, (lo, hi) in GROUPS.items():
        s = sig[name]
        block = b1[:, lo:hi]
        if s == 0.0:
            assert torch.equal(_bits(env.obs_bias[:, lo:hi]), torch.zeros_like(_bits(env.obs_bias[:, lo:hi]))), name
            continue
        for c in range(hi - lo):
            r = block[:, c]
            assert abs(r.mean()) < 4 * s / np.sqrt(N) and abs(r.std() / s - 1) < 0.02, (name, c, r.mean(), r.std())
        assert stats.kstest(block[:, 0] / np.float32(s), "norm").pvalue > 1e-3, name
    for c in range(9):
        assert abs(a1[:, c].std() / 0.03 - 1) < 0.02
    assert stats.kstest(a1[:, 4] / np.float32(0.03), "norm").pvalue > 1e-3
    assert abs(np.corrcoef(b1[:, 0], b1[:, 1])[0, 1]) < 0.01           # across columns
    assert abs(np.corrcoef(b1[:, 18], b1[:, 22])[0, 1]) < 0.01
    assert abs(np.corrcoef(b1[:, 0], a1[:, 0])[0, 1]) < 0.01
    assert abs(np.corrcoef(b1[:-1, 20], b1[1:, 20])[0, 1]) < 0.01      # across envs
    env.reset()
    b2 = env.obs_bias.double().cpu().numpy()
    assert abs(np.corrcoef(b1[:, 20], b2[:, 20])[0, 1]) < 0.01         # two consecutive episodes of one env
    # white noise on top: residual - offset is the white noise
    clean, _ = _env(_cfg(N, white=False, episode_length=None), seq=seq)
    clean.reset()
    clean.reset()   # each reset() advances the simulator: the same state as `env` for the step below
    env.step(seq.action[1].to(DEV))
    clean.step(seq.action[1].to(DEV))
    lo_, hi_ = observation_scale(resolve_config(_cfg(N)))
    half = torch.tensor((hi_ - lo_) / 2).to(DEV)
    resid = ((env.obs_buf - clean.obs_buf) * half).double().cpu().numpy() - env.obs_bias.double().cpu().numpy()
    for col, s in ((0, 0.005), (9, 0.05), (18, 0.002)):
        r = resid[:, col]
        assert abs(r.mean()) < 4 * s / np.sqrt(N) and abs(r.std() / s - 1) < 0.02, (col, r.mean(), r.std())
        assert stats.kstest(r / s, "norm").pvalue > 1e-3, col


@pytest.mark.parametrize("stream", ["philox", "torch"])
def test_reset_samples_do_not_depend_on_the_offsets(stream):
    """Every reset sample — joint rows, object and goal root rows, goal pose — is bit-identical with the offsets on and
    off, step by step (checked right after the pre-physics pass); two runs with offsets are identical."""
    from leibnizgym_b200 import _native as nat
    N, T = 4099, 8
    masks = _masks(N, T, 0.3, 5)
    envs = []
    for cfg in (_cfg(N, rng_stream=stream), _cfg(N, obs=ALL, act=0.05, rng_stream=stream),
                _cfg(N, obs=ALL, act=0.05, rng_stream=stream)):
        env, seq = _env(cfg, T=T)
        env.reset()
        envs.append(env)
    for t in range(T):
        a = seq.action[t].to(DEV)
        for e in envs:
            e._reset_buf |= masks[t]
            nat.check(e._lib.lg_pre_physics(e._P, e._S, e._B, a.data_ptr(), e._stream()), "lg_pre_physics")
        for e in envs[1:]:
            for name in ("dof_state", "root_state"):
                assert torch.equal(_bits(getattr(envs[0]._sim, name)), _bits(getattr(e._sim, name))), (t, name)
            assert torch.equal(_bits(envs[0]._object_goal_poses_buf), _bits(e._object_goal_poses_buf)), t
            assert torch.equal(_bits(envs[0]._object_goal_movement_buf), _bits(e._object_goal_movement_buf)), t
        for e in envs:
            e._simulate()
            e._call("lg_post_physics", e._P, e._S, e._B, float(e.env_steps_count))
    for f in ("_obs_buf", "_obs_bias", "_action_bias", "_action_buf"):
        assert torch.equal(_bits(getattr(envs[1], f)), _bits(getattr(envs[2], f))), f


def test_two_shards_equal_one_process():
    from leibnizgym_b200.synthetic import StateSequence, make_sequence
    N, T = 8198, 8
    cfg = _cfg(N, obs=ALL, act=0.05, white=True)
    seq = make_sequence(44, T, N)
    masks = _masks(N, T, 0.3, 45)
    whole, _ = _env(cfg, seq=seq)
    shards = []
    for r in range(2):
        lo, hi = r * N // 2, (r + 1) * N // 2
        sq = StateSequence(*(x.contiguous() for x in (seq.dof_state[:, lo:hi], seq.root_state[:, 4 * lo:4 * hi],
                                                      seq.rigid_body[:, lo:hi], seq.dof_force[:, lo:hi],
                                                      seq.ft_sensors[:, lo:hi], seq.action[:, lo:hi])))
        shards.append(_env(cfg, seq=sq, rank=r, world=2)[0])
    for e in [whole] + shards:
        e.reset()
    for t in range(T):
        whole.set_forced_resets(masks[t])
        whole.step(seq.action[t].to(DEV))
        for r, e in enumerate(shards):
            lo, hi = r * N // 2, (r + 1) * N // 2
            e.set_forced_resets(masks[t][lo:hi].contiguous())
            e.step(seq.action[t, lo:hi].to(DEV))
        for f in ("_obs_bias", "_action_bias", "_obs_buf", "_action_buf", "_states_buf"):
            cat = torch.cat([getattr(e, f) for e in shards])
            assert torch.equal(_bits(cat), _bits(getattr(whole, f))), (t, f)


def test_hook_route():
    """IsaacEnvBase.step against the fused step: `reset()` draws the same offsets on both (lg_reset_envs), and steps
    without resets give bit-identical observations; with action offsets the hook route refuses to step."""
    from leibnizgym_b200.env import IsaacEnvBase
    N, T = 4099, 6
    # no success termination: goal resets would draw different goals on the two routes (each keys its draws by an
    # epoch it advances itself), which has nothing to do with the offsets
    cfg = _cfg(N, obs=ALL, episode_length=None, termination_conditions={"success": dict(SUCCESS["success"], activate=False)})
    fused, seq = _env(cfg, T=T)
    hooks, _ = _env(cfg, seq=seq)
    for e in (fused, hooks):
        e.reset()
    assert torch.equal(_bits(fused.obs_bias), _bits(hooks.obs_bias))
    for t in range(T):
        a = seq.action[t].to(DEV)
        fused.step(a)
        IsaacEnvBase.step(hooks, a)
        for f in ("_obs_buf", "_states_buf", "_obs_bias", "_reward_buf"):
            assert torch.equal(_bits(getattr(fused, f)), _bits(getattr(hooks, f))), (t, f)
    withact, _ = _env(_cfg(N, obs=ALL, act=0.05), seq=seq)
    withact.reset()
    with pytest.raises(ValueError, match="action_bias_std"):
        IsaacEnvBase.step(withact, seq.action[0].to(DEV))


def test_graph_replay_equals_eager_steps():
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence
    N, R = 16384, 4
    cfg = _cfg(N, obs=ALL, act=0.05, white=True)
    rm = bernoulli_masks(31, R, N, 0.3, device=DEV)
    gm = bernoulli_masks(32, R, N, 0.05, device=DEV)
    out = []
    for graph in (True, False):
        ring = make_sequence(30, R, N, device=DEV)
        env = TrifingerEnv(cfg, device=DEV, verbose=False, sim=SyntheticSim(ring, DEV))
        env.reset()
        runner = GraphRunner(env, ring, rotate_outputs=True, inject_reset_masks=rm, inject_goal_masks=gm)
        if graph:
            runner.capture(R)
            runner.replay(3)
        else:
            st = torch.cuda.current_stream().cuda_stream
            for t in [0, 1] + list(range(R)) * 3:
                runner._launch_step(t, st)
        torch.cuda.synchronize()
        out.append(env)
    for f in ("_obs_bias", "_action_bias", "_action_buf", "_episode_return"):
        assert torch.equal(_bits(getattr(out[0], f)), _bits(getattr(out[1], f))), f


@pytest.mark.parametrize("route", ["pipeline", "host_outputs"])
def test_host_paths_equal_the_device_path(route):
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    from leibnizgym_b200.wrappers import VecTaskPython
    N, T = 12288, 8
    cfg = _cfg(N, obs=ALL, act=0.05, white=True)
    host = make_sequence(62, T, N).to("cpu", pin=True)

    def build(kind):
        sim = SyntheticSim(host, DEV)
        env = TrifingerEnv(cfg, device=DEV, verbose=False, sim=sim)
        sim.use_sparse_upload(env._P)
        vec = VecTaskPython(env, rl_device="cpu" if kind != "device" else DEV,
                            **({"host_pipeline_chunks": 2} if kind == "pipeline" else {}))
        vec.reset()
        return env, vec

    ref, ref_vec = build("device")
    env, vec = build(route)
    masks = _masks(N, T, 0.3, 63)
    for t in range(1, T):
        for e in (ref, env):
            e._reset_buf |= masks[t]
        o1 = ref_vec.step(host.action[t])[0]
        o2 = vec.step(host.action[t])[0]
        torch.cuda.synchronize()
        for f in ("_obs_bias", "_action_bias", "_action_buf"):
            assert torch.equal(_bits(getattr(ref, f)), _bits(getattr(env, f))), (route, t, f)
        assert torch.equal(_bits(o1["obs"] if isinstance(o1, dict) else o1), _bits(o2["obs"] if isinstance(o2, dict) else o2))


def test_checkpoint_resume_and_refusal(tmp_path):
    N, T = 4099, 10
    cfg = _cfg(N, obs=ALL, act=0.05, white=True)
    env, seq = _env(cfg, T=T)
    masks = _masks(N, T, 0.2, 70)
    env.reset()
    for t in range(T):
        if t == 5:
            path = env.save_checkpoint(str(tmp_path / "mid"))
            resumed, _ = _env(cfg, seq=seq)
            resumed.load_checkpoint(path)
        live = [env] + ([resumed] if t >= 5 else [])
        for e in live:
            e._reset_buf |= masks[t]
            e.step(seq.action[t % seq.num_steps].to(DEV))
        if t >= 5:
            for f in ("_obs_bias", "_action_bias", "_obs_buf", "_action_buf", "_states_buf"):
                assert torch.equal(_bits(getattr(env, f)), _bits(getattr(resumed, f))), (t, f)
    other, _ = _env(_cfg(N, white=True), seq=seq)
    with pytest.raises(ValueError, match="DR offsets"):
        other.load_checkpoint(path)
    obs_only, _ = _env(_cfg(N, obs=ALL, white=True), seq=seq)
    with pytest.raises(ValueError, match="DR offsets"):
        obs_only.load_checkpoint(path)
    other_path = other.save_checkpoint(str(tmp_path / "off"))
    with pytest.raises(ValueError, match="DR offsets"):
        env.load_checkpoint(other_path)
