"""Episode statistics (extension, "episode_statistics": {"activate": True}) on the GPU: the running returns, the
last-episode records and the per-step episode_stats against the torch restatement (tests/episode_reference.py) in
every pre-physics regime, and bit-identity across the routes that step the env: hooks, torch stream, CUDA graph,
shards, the host paths, checkpoints."""
import copy

import pytest
import torch

from episode_reference import EpisodeTracker

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SUCCESS = {"success": {"activate": True, "bonus": 5000.0, "position_tolerance": 0.12, "orientation_tolerance": 1.5}}
FIELDS = ("_episode_return", "_last_episode_return", "_last_episode_length", "_last_episode_success", "_episode_stats")
FIX_RES = 2.0 ** -30   # resolution of the fixed-point return sums, per record


def _cfg(N, asym=True, episode_length=5, seed=3, **extra):
    from leibnizgym_b200.config import difficulty_config
    cfg = difficulty_config(4, N, asymmetric_obs=asym, seed=seed, episode_length=episode_length,
                            termination_conditions=copy.deepcopy(SUCCESS))
    cfg["episode_statistics"] = {"activate": True}
    cfg.update(extra)
    return cfg


def _env(cfg, seq=None, T=8, seq_seed=21, rank=0, world=1):
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    if seq is None:
        seq = make_sequence(seq_seed, T, cfg["num_instances"])
    return TrifingerEnv(cfg, device=DEV, verbose=False, sim=SyntheticSim(seq.to(DEV), DEV), rank=rank, world_size=world), seq


def _masks(N, T, p, seed):
    g = torch.Generator().manual_seed(seed)
    return [(torch.rand(N, generator=g) < p).to(DEV) for _ in range(T)]


def _bits(t):
    return t.detach().contiguous().view(torch.uint8).cpu()


def _same(a, b, where):
    for f in FIELDS:
        assert torch.equal(_bits(getattr(a, f)), _bits(getattr(b, f))), (where, f)


def _check_against_tracker(env, tr, stats, where):
    assert torch.equal(_bits(env.episode_return), _bits(tr.episode_return)), (where, "episode_return")
    assert torch.equal(_bits(env.last_episode_return), _bits(tr.last_episode_return)), (where, "last_episode_return")
    assert torch.equal(env.last_episode_length.cpu(), tr.last_episode_length), (where, "last_episode_length")
    assert torch.equal(env.last_episode_success.cpu(), tr.last_episode_success), (where, "last_episode_success")
    got = env._episode_stats.cpu()
    assert got[0] == stats[0] and got[2] == stats[2] and got[3] == stats[3], (where, got, stats)
    assert abs(float(got[1]) - float(stats[1])) <= FIX_RES * float(stats[0]) + 1e-12 * abs(float(stats[1])), (where, got, stats)


def _ticket_size():
    from leibnizgym_b200 import _native
    lib = _native.load()
    tile = (1 << 20) // int(lib.lg_scan_tiles(1 << 20))   # envs per pre-physics tile
    return (int(lib.lg_pre_resident_tiles()) + 3) * tile + 5


@pytest.mark.parametrize("asym", [True, False])
@pytest.mark.parametrize("N", [16384, 4099, "ticket"])
@pytest.mark.parametrize("episode_length", [5, 7])
def test_fused_steps_match_the_restatement(N, asym, episode_length):
    """Difficulty 4 with success termination (goal resets happen and must not end episodes), timeouts, 30 % forced
    resets on every third step, 20 steps; the restatement is fed the kernel's own rewards, reset ids and flags."""
    N = _ticket_size() if N == "ticket" else N
    env, seq = _env(_cfg(N, asym, episode_length))
    forced = _masks(N, 20, 0.3, 8)
    tr = EpisodeTracker(N)
    env.reset()
    tr.reset(torch.arange(N))
    goal_resets = 0
    for t in range(20):
        env.set_forced_resets(forced[t] if t % 3 == 2 else None)
        env.step(seq.action[t % seq.num_steps].to(DEV))
        tr.reset(env.reset_env_ids.cpu())
        goal_resets += int(env._counts[1])
        stats = tr.post(env._reward_buf.cpu(), env._successes.cpu())
        _check_against_tracker(env, tr, stats, (N, asym, episode_length, t))
        info = env._step_info
        assert float(info["env/episodes/count"]) == float(stats[0])
    assert goal_resets > 0 and int(tr.last_episode_length.gt(0).sum()) == N
    assert bool(tr.last_episode_success.any())


def _hook_pair(cfg, T):
    a, seq = _env(cfg, T=T)
    b, _ = _env(cfg, seq=seq)
    return a, b, seq


@pytest.mark.parametrize("stream", ["philox", "torch"])
def test_hook_route_equals_fused_step(stream):
    """IsaacEnvBase.step (lg_reset_envs, lg_goal_reset_envs, lg_pre_step, lg_post_physics without bookkeeping) against
    the fused TrifingerEnv.step, bit for bit on all five buffers, every step.  The own Philox stream keys its draws by
    an epoch that each route advances differently, so with it both routes read the same injected draws (indexed by
    rank in the reset / goal-reset list); the torch stream draws the same numbers on both routes by construction."""
    from leibnizgym_b200.env import IsaacEnvBase
    N, T = 4099, 12
    fused, hooks, seq = _hook_pair(_cfg(N, rng_stream=stream), T)
    masks = _masks(N, T, 0.3, 4)
    g = torch.Generator().manual_seed(13)
    for e in (fused, hooks):
        e.reset()
    for t in range(T):
        a = seq.action[t % seq.num_steps].to(DEV)
        if stream == "philox":
            draws = [(torch.rand(N, 24, generator=g).numpy(), torch.randn(N, 8, generator=g).numpy()) for _ in range(2)]
        for e in (fused, hooks):
            e._reset_buf |= masks[t]
            if stream == "philox":
                e.inject_draws(reset=draws[0], goal=draws[1])
        fused.step(a)
        IsaacEnvBase.step(hooks, a)
        _same(fused, hooks, (stream, t))
    assert int(fused.last_episode_length.gt(0).sum()) > 0


def test_graph_replay_equals_eager_steps():
    """GraphRunner capture + replay (device clock, chained pre-physics, per-slot forced masks) against the same launches
    made eagerly on a twin env: all five buffers bit-identical."""
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.graph_runner import GraphRunner
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence
    N, R = 16384, 4
    cfg = _cfg(N)
    rm = bernoulli_masks(31, R, N, 0.3, device=DEV)
    gm = bernoulli_masks(32, R, N, 0.05, device=DEV)
    out = []
    for graph in (True, False):
        ring = make_sequence(30, R, N, device=DEV)
        env = TrifingerEnv(cfg, device=DEV, verbose=False, sim=SyntheticSim(ring, DEV))
        env.reset()
        runner = GraphRunner(env, ring, rotate_outputs=True, inject_reset_masks=rm, inject_goal_masks=gm)
        if graph:
            runner.capture(R)      # two eager warm-up steps (t = 0, 1), then steps 0 .. R-1 captured
            runner.replay(3)
        else:
            st = torch.cuda.current_stream().cuda_stream
            for t in [0, 1] + list(range(R)) * 3:
                runner._launch_step(t, st)
        torch.cuda.synchronize()
        out.append(env)
    _same(out[0], out[1], "graph")
    assert float(out[0]._episode_stats[0]) > 0 or int(out[0].last_episode_length.gt(0).sum()) > 0


def test_two_shards_equal_one_process():
    """Two shards of 4 099 envs against one of 8 198: per-env buffers concatenated bit-identical, the shard sums add up
    to the single process's, and the job-wide means agree."""
    from leibnizgym_b200.distributed import stats_to_info
    from leibnizgym_b200.synthetic import StateSequence, make_sequence
    N, T = 8198, 12
    cfg = _cfg(N)
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
    reported = 0.0
    for t in range(T):
        whole.set_forced_resets(masks[t])
        whole.step(seq.action[t].to(DEV))
        for r, e in enumerate(shards):
            lo, hi = r * N // 2, (r + 1) * N // 2
            e.set_forced_resets(masks[t][lo:hi].contiguous())
            e.step(seq.action[t, lo:hi].to(DEV))
        for f in FIELDS[:4]:
            cat = torch.cat([getattr(e, f) for e in shards])
            assert torch.equal(_bits(cat), _bits(getattr(whole, f))), (t, f)
        summed = shards[0]._episode_stats + shards[1]._episode_stats
        ref = whole._episode_stats
        assert torch.equal(summed[[0, 2, 3]], ref[[0, 2, 3]]), t
        assert abs(float(summed[1] - ref[1])) <= FIX_RES * float(ref[0]) * 2 + 1e-12 * abs(float(ref[1])), t
        reported += float(ref[0])
        a = whole.global_step_info()
        b = stats_to_info(torch.zeros(16, dtype=torch.float64), [], episode_stats=summed)
        for k in ("env/episodes/count", "env/episodes/length_sum", "env/episodes/successes"):
            assert a[k] == b[k], (t, k)
        if a["env/episodes/count"] > 0:
            for k in ("env/episodes/mean_return", "env/episodes/mean_length", "env/episodes/success_rate"):
                assert a[k] == pytest.approx(b[k], rel=1e-9, abs=FIX_RES), (t, k)
    assert reported > 0


@pytest.mark.parametrize("route", ["pipeline", "host_outputs"])
def test_host_paths_equal_the_device_path(route):
    """VecTaskPython over the chunked host pipeline (two chunks) and over the host-output path (results stored into
    pinned host memory) against the device path of a twin env."""
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    from leibnizgym_b200.wrappers import VecTaskPython
    N, T = 12288, 10
    cfg = _cfg(N)
    host = make_sequence(62, T, N).to("cpu", pin=True)

    def build(kind):
        sim = SyntheticSim(host, DEV)
        env = TrifingerEnv(cfg, device=DEV, verbose=False, sim=sim)
        sim.use_sparse_upload(env._P)
        if kind == "pipeline":
            vec = VecTaskPython(env, rl_device="cpu", host_pipeline_chunks=2)
        elif kind == "host_outputs":
            vec = VecTaskPython(env, rl_device="cpu")
        else:
            vec = VecTaskPython(env, rl_device=DEV)
        vec.reset()
        return env, vec

    ref, ref_vec = build("device")
    env, vec = build(route)
    masks = _masks(N, T, 0.3, 63)
    for t in range(1, T):
        for e in (ref, env):
            e._reset_buf |= masks[t]
        ref_vec.step(host.action[t])
        vec.step(host.action[t])
        torch.cuda.synchronize()
        _same(ref, env, (route, t))
    assert int(env.last_episode_length.gt(0).sum()) > 0


def test_each_episode_is_counted_once_and_reset_ends_episodes(tmp_path):
    """Counting: the first step after construction reports nothing; over a run the counts reported equal the number of
    resets of envs that had stepped; `reset()` mid-run ends every env that stepped and the next step reports them all;
    a checkpoint taken mid-run continues bit-identically; a checkpoint of the other setting is refused."""
    N, T = 4099, 14
    cfg = _cfg(N, episode_length=6)
    env, seq = _env(cfg, T=T)
    masks = _masks(N, T, 0.2, 70)
    steps = torch.zeros(N, dtype=torch.int64)
    ended = reported = 0
    env.reset()
    for t in range(T):
        if t == 7:
            path = env.save_checkpoint(str(tmp_path / "mid"))
            resumed, _ = _env(cfg, seq=seq)
            resumed.load_checkpoint(path)
        live = [env] + ([resumed] if t >= 7 else [])
        if t == 10:   # every env has stepped since its last reset: reset() ends all N episodes
            ended += int(steps.gt(0).sum())
            steps.zero_()
            for e in live:
                e.reset()
        for e in live:
            e._reset_buf |= masks[t]
            e.step(seq.action[t % seq.num_steps].to(DEV))
        ids = env.reset_env_ids.cpu()
        ended += int(steps[ids].gt(0).sum())
        steps[ids] = 0
        steps += 1
        count = float(env._episode_stats[0])
        if t == 0:
            assert count == 0.0
        if t == 10:
            assert count == N
        reported += count
        if t >= 7:
            _same(env, resumed, ("checkpoint", t))
            assert torch.equal(_bits(env._obs_buf), _bits(resumed._obs_buf)), t
    assert reported == ended > 0
    off = copy.deepcopy(cfg)
    off["episode_statistics"] = {"activate": False}
    other, _ = _env(off, seq=seq)
    with pytest.raises(ValueError, match="episode_statistics"):
        other.load_checkpoint(path)
    other_path = other.save_checkpoint(str(tmp_path / "off"))
    with pytest.raises(ValueError, match="episode_statistics"):
        env.load_checkpoint(other_path)


def test_non_finite_reward_reaches_only_its_env():
    """A NaN in one env's fingertip position (every state of the simulator sequence) makes that env's reward NaN: its
    running return is NaN, a step that reports its episode has a NaN return sum with exact counts, and every other
    env's record equals that of a twin env without the NaN."""
    from leibnizgym_b200.synthetic import StateSequence, make_sequence
    N, T, bad = 4099, 9, 1234
    cfg = _cfg(N, episode_length=4)
    seq = make_sequence(23, T, N)
    ref, _ = _env(cfg, seq=seq)
    nan_seq = StateSequence(*(getattr(seq, f).clone() for f in seq.__dataclass_fields__))
    nan_seq.rigid_body[:, bad, 6, 0] = float("nan")
    env, _ = _env(cfg, seq=nan_seq)
    for e in (ref, env):
        e.reset()
    tr = EpisodeTracker(N)
    tr.reset(torch.arange(N))
    others = (torch.arange(N) != bad).to(DEV)
    saw_nan_sum = False
    for t in range(T):
        for e in (ref, env):
            e.step(seq.action[t].to(DEV))
        tr.reset(env.reset_env_ids.cpu())
        stats = tr.post(env._reward_buf.cpu(), env._successes.cpu())
        got = env._episode_stats.cpu()
        assert got[0] == stats[0] and got[2] == stats[2] and got[3] == stats[3], t
        if torch.isnan(stats[1]):
            assert torch.isnan(got[1]), t
            saw_nan_sum = True
        assert torch.isnan(env.episode_return[bad]), t
        for f in ("_last_episode_return", "_last_episode_length", "_last_episode_success"):
            assert torch.equal(_bits(getattr(env, f)[others]), _bits(getattr(ref, f)[others])), (t, f)
    assert saw_nan_sum and torch.isnan(env.last_episode_return[bad])


def test_off_by_default_changes_nothing():
    from leibnizgym_b200.config import difficulty_config
    N = 1024
    cfg = difficulty_config(4, N, asymmetric_obs=True, seed=3, episode_length=3, termination_conditions=copy.deepcopy(SUCCESS))
    env, seq = _env(cfg)
    assert all(getattr(env, f) is None for f in FIELDS)
    assert env.episode_return is None and env.last_episode_length is None
    assert env._B.episode_return is None and env._B.episode_stats is None
    env.reset()
    for t in range(4):
        _, _, _, info = env.step(seq.action[t].to(DEV))
    assert not any(k.startswith("env/episodes/") for k in info)
    assert not any(k.startswith("env/episodes/") for k in env.global_step_info())
    assert sorted(info) == sorted(["env/rewards/finger_reach_object_rate", "env/rewards/finger_move_penalty",
                                   "env/rewards/object_dist", "env/rewards/object_rot",
                                   "env/current_position_goal/count", "env/current_orientation_goal/count",
                                   "env/average_consecutive_success"])
