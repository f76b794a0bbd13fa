"""Per-term episode returns (extension, "episode_term_returns": {"activate": True}) on the GPU: the running rows, the
records and the per-step episode_term_stats against the torch restatement (tests/episode_term_reference.py) fed the
kernel's own term values, in every pre-physics regime; the slots of a record against its episode return; bit-identity
of the three buffers across the routes that step the env; no effect on any other buffer; the instantiation that runs;
a NaN confined to its env and slot."""
import copy

import pytest
import torch

from episode_term_reference import EpisodeTermTracker, slot_sum_bound

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SUCCESS = {"success": {"activate": True, "bonus": 5000.0, "position_tolerance": 0.12, "orientation_tolerance": 1.5}}
FIELDS = ("_episode_term_return", "_last_episode_term_return", "_episode_term_stats")
EPISODE_FIELDS = ("_episode_return", "_last_episode_return", "_last_episode_length", "_last_episode_success",
                  "_episode_stats")
FIX_RES = 2.0 ** -30   # resolution of the fixed-point sums, per record


def _cfg(N, asym=True, episode_length=5, seed=3, keypoint=False, **extra):
    from leibnizgym_b200.config import difficulty_config
    cfg = difficulty_config(4, N, asymmetric_obs=asym, seed=seed, episode_length=episode_length,
                            termination_conditions=copy.deepcopy(SUCCESS))
    if keypoint:   # the extension term on, one reference term off
        cfg["reward_terms"]["keypoint"] = {"activate": True, "weight": 1500, "scale": 30.0, "eps": 2.0}
        cfg["reward_terms"]["object_rot"]["activate"] = False
    cfg["episode_statistics"] = {"activate": True}
    cfg["episode_term_returns"] = {"activate": True}
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


def _same(a, b, where, fields=FIELDS):
    for f in fields:
        assert torch.equal(_bits(getattr(a, f)), _bits(getattr(b, f))), (where, f)


def _active(cfg):
    from leibnizgym_b200 import _native as nat
    return [bool(cfg["reward_terms"].get(n, {}).get("activate")) for n in nat.TERM_NAMES]


def _ticket_size():
    from leibnizgym_b200 import _native
    lib = _native.load()
    tile = (1 << 20) // int(lib.lg_scan_tiles(1 << 20))   # envs per pre-physics tile
    return (int(lib.lg_pre_resident_tiles()) + 3) * tile + 5


class _Checker:
    """The restatement next to a fused env, fed the kernel's own term values, reset ids and post-step goal-reset flags;
    a second restatement of the absolute values bounds the slot sums."""

    def __init__(self, env, cfg):
        N = env.num_instances
        env.enable_term_rewards()
        self.env, self.cfg = env, cfg
        bonus = cfg["termination_conditions"]["success"]["bonus"]
        self.tr = EpisodeTermTracker(N, _active(cfg), bonus)
        self.abs = EpisodeTermTracker(N, _active(cfg), abs(bonus))
        for t in (self.tr, self.abs):
            t.reset(torch.arange(N))
        self.success = bool(cfg["termination_conditions"]["success"]["activate"])

    def step(self, where):
        env = self.env
        ids = env.reset_env_ids.cpu()
        terms = env._term_rewards.cpu()
        paid = env._goal_reset_buf.cpu() if self.success else torch.zeros(env.num_instances, dtype=torch.bool)
        self.tr.reset(ids)
        self.abs.reset(ids)
        n, stats = self.tr.post(terms, paid)
        self.abs.post(terms.abs(), paid)
        assert torch.equal(_bits(env.episode_term_return), _bits(self.tr.episode_term_return)), (where, "running")
        assert torch.equal(_bits(env.last_episode_term_return), _bits(self.tr.last_episode_term_return)), (where, "record")
        assert torch.equal(env.last_episode_length.cpu(), self.tr.last_episode_length), (where, "length")
        assert float(env._episode_stats[0]) == n, where
        got = env._episode_term_stats.cpu()
        nan = torch.isnan(stats)
        assert torch.equal(torch.isnan(got), nan), (where, got, stats)
        ok = (got - stats).abs()[~nan] <= FIX_RES * n + 1e-12 * stats.abs()[~nan]
        assert bool(ok.all()), (where, got, stats)
        return n, stats

    def check_slot_sums(self, where):
        """Sum of the 8 slots of every record against the record's episode return (fp32, summed by step)."""
        env = self.env
        done = env.last_episode_length.cpu() > 0
        slots = env.last_episode_term_return.cpu()[done].double().sum(1)
        ret = env.last_episode_return.cpu()[done].double()
        bound = slot_sum_bound(self.abs.last_episode_term_return[done].double().sum(1), env.last_episode_length.cpu()[done])
        assert bool(((slots - ret).abs() <= bound).all()), (where, float((slots - ret).abs().max()))
        return int(done.sum())


@pytest.mark.parametrize("asym", [True, False])
@pytest.mark.parametrize("N", [16384, 4099, "ticket"])
@pytest.mark.parametrize("episode_length", [5, 7])
def test_fused_steps_match_the_restatement(N, asym, episode_length):
    """Difficulty 4 with success termination (the bonus slot fills; goal resets must not end episodes), timeouts and 30 %
    forced resets on every third step, 20 steps."""
    N = _ticket_size() if N == "ticket" else N
    cfg = _cfg(N, asym, episode_length)
    env, seq = _env(cfg)
    forced = _masks(N, 20, 0.3, 8)
    env.reset()
    chk = _Checker(env, cfg)
    reported = 0
    for t in range(20):
        env.set_forced_resets(forced[t] if t % 3 == 2 else None)
        env.step(seq.action[t % seq.num_steps].to(DEV))
        reported += chk.step((N, asym, episode_length, t))[0]
    assert reported > 0 and chk.check_slot_sums("end") == N
    assert float(env.last_episode_term_return[:, 7].abs().sum()) > 0      # the bonus was paid and recorded
    assert float(env.episode_term_return[:, [4, 5, 6]].abs().sum()) == 0   # inactive terms stay 0


@pytest.mark.parametrize("asym", [True, False])
def test_keypoint_on_and_a_term_off(asym):
    """The keypoint term fills slot 6; object_rot switched off keeps slot 3 at 0 and is not reported in `info`."""
    N = 4099
    cfg = _cfg(N, asym, 7, keypoint=True)
    env, seq = _env(cfg)
    forced = _masks(N, 16, 0.3, 9)
    env.reset()
    chk = _Checker(env, cfg)
    for t in range(16):
        env.set_forced_resets(forced[t] if t % 3 == 2 else None)
        _, _, _, info = env.step(seq.action[t % seq.num_steps].to(DEV))
        chk.step(("keypoint", asym, t))
    chk.check_slot_sums("keypoint")
    for buf in (env.episode_term_return, env.last_episode_term_return):
        assert float(buf[:, 3].abs().sum()) == 0 and float(buf[:, 6].abs().sum()) > 0
    assert float(env._episode_term_stats[3]) == 0
    keys = sorted(k for k in info if k.startswith("env/episodes/return_sum/"))
    assert keys == sorted(f"env/episodes/return_sum/{n}" for n in
                          ("finger_reach_object_rate", "finger_move_penalty", "object_dist", "keypoint", "success_bonus"))
    g = env.global_step_info()
    assert "env/episodes/return_sum/object_rot" not in g and "env/episodes/return_sum/keypoint" in g


@pytest.mark.parametrize("stream", ["philox", "torch"])
def test_hook_route_equals_fused_step(stream):
    """IsaacEnvBase.step (lg_reset_envs, lg_goal_reset_envs, lg_pre_step, lg_post_physics without bookkeeping) against
    the fused TrifingerEnv.step, bit for bit on the three buffers, every step; with the own Philox stream both routes
    read the same injected draws."""
    from leibnizgym_b200.env import IsaacEnvBase
    N, T = 4099, 12
    cfg = _cfg(N, rng_stream=stream)
    fused, seq = _env(cfg, T=T)
    hooks, _ = _env(cfg, seq=seq)
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
    assert float(fused.last_episode_term_return.abs().sum()) > 0


def test_graph_replay_equals_eager_steps():
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
            runner.capture(R)
            runner.replay(3)
        else:
            st = torch.cuda.current_stream().cuda_stream
            for t in [0, 1] + list(range(R)) * 3:
                runner._launch_step(t, st)
        torch.cuda.synchronize()
        out.append(env)
    _same(out[0], out[1], "graph")
    assert float(out[0].last_episode_term_return.abs().sum()) > 0


def test_two_shards_equal_one_process():
    """Two shards of 4 099 envs against one of 8 198: rows concatenated bit-identical, the shard sums add up to the
    single process's, and the job-wide per-term means agree."""
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
        for f in FIELDS[:2]:
            cat = torch.cat([getattr(e, f) for e in shards])
            assert torch.equal(_bits(cat), _bits(getattr(whole, f))), (t, f)
        count = float(whole._episode_stats[0])
        summed = shards[0]._episode_term_stats + shards[1]._episode_term_stats
        assert bool(((summed - whole._episode_term_stats).abs() <= FIX_RES * count * 2 +
                     1e-12 * whole._episode_term_stats.abs()).all()), t
        reported += count
        a = whole.global_step_info()
        b = stats_to_info(torch.zeros(16, dtype=torch.float64), [], episode_stats=whole._episode_stats,
                          episode_term_stats=summed)
        for k, v in a.items():
            if k.startswith("env/episodes/return_sum/") or k.startswith("env/episodes/mean_return/"):
                assert v == pytest.approx(b[k], rel=1e-9, abs=2 * FIX_RES * max(count, 1.0)), (t, k)
        if count > 0:
            assert "env/episodes/mean_return/object_dist" in a and "env/episodes/mean_return/success_bonus" in a
    assert reported > 0


@pytest.mark.parametrize("route", ["pipeline", "host_outputs"])
def test_host_paths_equal_the_device_path(route):
    """VecTaskPython over the chunked host pipeline (two chunks) and over the host-output path against the device path."""
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
    assert float(env.last_episode_term_return.abs().sum()) > 0


def test_checkpoint_resume_and_setting_mismatch(tmp_path):
    N, T = 4099, 12
    cfg = _cfg(N, episode_length=6)
    env, seq = _env(cfg, T=T)
    masks = _masks(N, T, 0.2, 70)
    env.reset()
    for t in range(T):
        if t == 6:
            path = env.save_checkpoint(str(tmp_path / "mid"))
            resumed, _ = _env(cfg, seq=seq)
            resumed.load_checkpoint(path)
        live = [env] + ([resumed] if t >= 6 else [])
        for e in live:
            e._reset_buf |= masks[t]
            e.step(seq.action[t % seq.num_steps].to(DEV))
        if t >= 6:
            _same(env, resumed, ("checkpoint", t), FIELDS + EPISODE_FIELDS)
    off = copy.deepcopy(cfg)
    off["episode_term_returns"] = {"activate": False}
    other, _ = _env(off, seq=seq)
    with pytest.raises(ValueError, match="episode_term_returns"):
        other.load_checkpoint(path)
    other_path = other.save_checkpoint(str(tmp_path / "off"))
    with pytest.raises(ValueError, match="episode_term_returns"):
        env.load_checkpoint(other_path)


def test_on_versus_off_changes_nothing_else():
    """Episode statistics on in both: with the per-term returns on, every other buffer (the five episode buffers
    included) is bit-identical to the run with them off, every step, and `info` only gains the per-term keys.  The
    step statistics are the exception: with an env count that is not a power of two each CTA's means are rounded before
    the CTAs add them up in fp64 in the order they finish, so a change of timing alone moves their last bits.  They
    must agree to a few ulps."""
    from leibnizgym_b200.checkpoint import _ENV_TENSORS
    N, T = 4099, 12
    on_cfg = _cfg(N)
    off_cfg = copy.deepcopy(on_cfg)
    off_cfg["episode_term_returns"] = {"activate": False}
    on, seq = _env(on_cfg, T=T)
    off, _ = _env(off_cfg, seq=seq)
    assert all(getattr(off, f) is None for f in FIELDS) and off._B.episode_term_return is None
    masks = _masks(N, T, 0.3, 71)
    for e in (on, off):
        e.reset()
    others = [a for n, a in _ENV_TENSORS.items()
              if "_term_" not in a and a != "_step_stats" and getattr(off, a, None) is not None]
    assert set(EPISODE_FIELDS) <= set(others)
    for t in range(T):
        infos = []
        for e in (on, off):
            e.set_forced_resets(masks[t])
            infos.append(e.step(seq.action[t % seq.num_steps].to(DEV))[3])
        _same(on, off, ("on/off", t), others)
        assert torch.allclose(on._step_stats, off._step_stats, rtol=1e-14, atol=0), t
        assert set(infos[0]) - set(infos[1]) == {k for k in infos[0] if k.startswith("env/episodes/return_sum/")}
        assert set(infos[1]) <= set(infos[0])


def test_the_ext_instantiation_runs():
    """torch.profiler names the kernels of a fused step: the post-physics pass is the EXT instantiation (as with the
    episode statistics alone), and the feature adds no kernel."""
    from instantiation_digest import launched
    N = 4099
    on_cfg = _cfg(N)
    off_cfg = copy.deepcopy(on_cfg)
    off_cfg["episode_term_returns"] = {"activate": False}
    got = {}
    for name, cfg in (("on", on_cfg), ("off", off_cfg)):
        env, seq = _env(cfg)
        env.reset()
        env.step(seq.action[0].to(DEV))
        got[name] = launched(lambda: env.step(seq.action[1].to(DEV)))
    assert got["on"] == got["off"]
    assert len(got["on"]["post"]) == 1
    (post,) = got["on"]["post"]
    assert post[2] == 1 and post[5] == 1, post   # REWARD, EXT


def test_nan_in_one_term_reaches_only_its_slot():
    """A NaN in one env's fingertip position makes finger_reach_object_rate NaN for that env (finger_move_penalty, which
    reads the fingertips too, is switched off here): only that env's slot 0 is NaN, the step that reports its episode
    has a NaN in episode_term_stats[0] alone, and every other env's rows equal a twin env's without the NaN."""
    from leibnizgym_b200.synthetic import StateSequence, make_sequence
    N, T, bad = 4099, 9, 1234
    cfg = _cfg(N, episode_length=4)
    cfg["reward_terms"]["finger_move_penalty"]["activate"] = False
    seq = make_sequence(23, T, N)
    ref, _ = _env(cfg, seq=seq)
    nan_seq = StateSequence(*(getattr(seq, f).clone() for f in seq.__dataclass_fields__))
    nan_seq.rigid_body[:, bad, 6, 0] = float("nan")
    env, _ = _env(cfg, seq=nan_seq)
    for e in (ref, env):
        e.reset()
    chk = _Checker(env, cfg)
    others = (torch.arange(N) != bad).to(DEV)
    saw = False
    for t in range(T):
        for e in (ref, env):
            e.step(seq.action[t].to(DEV))
        chk.step(("nan", t))
        row = env.episode_term_return[bad].cpu()
        assert torch.isnan(row[0]) and not bool(torch.isnan(row[1:]).any()), (t, row)
        stats = env._episode_term_stats.cpu()
        if torch.isnan(stats[0]):
            saw = True
        assert not bool(torch.isnan(stats[1:]).any()), (t, stats)
        for f in FIELDS[:2]:
            assert torch.equal(_bits(getattr(env, f)[others]), _bits(getattr(ref, f)[others])), (t, f)
    assert saw and torch.isnan(env.last_episode_term_return[bad, 0])
