"""GPU parity on the inputs where kernels go wrong: NaN, +-inf, +-3.4e38, the fast division's 2^100 edge, denormals and
-0.0, against the CPU oracle (itself pinned to the reference on the same kinds of input, tests/golden/
reference_functions.py).

  A. the batched primitives on the stored adversarial inputs, plus rows with NaN;
  B. whole steps with non-finite / extreme values planted in every source tensor (several in one tile, one cold value
     in a role lane whose other envs stay finite, the last env of a full tile, the ragged tile), through the fused
     clamps of VecTaskPython, the raw env and the hook-by-hook route; then forced resets of poisoned envs;
  C. the episode statistics against the kernel's own per-env outputs, to the resolution of the fixed-point sums;
  D. the stored reward-term cases (random schedules, env-step counts on the window edges) through the fused kernel.
"""
import copy
import itertools
import math
import os
import random
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import reference_functions as rf  # noqa: E402
from tolerances import angle_slack, compare  # noqa: E402

pytestmark = pytest.mark.gpu

NAN, INF = float("nan"), float("inf")
BELOW_2_100 = float(np.nextafter(np.float32(2.0 ** 100), np.float32(0)))   # last numerator of the fast division
TINY = float(np.float32(1e-42))                                             # denormal
VALUES = (NAN, INF, -INF, 3.4e38, -3.4e38, 2.0 ** 100, BELOW_2_100, TINY, -TINY, -0.0)
# source tensor -> number of columns a plant can hit
TENSORS = {"dof_pos": 9, "dof_vel": 9, "obj_pose": 7, "obj_vel": 6, "tip_pos": 9, "tip_rest": 30, "dof_force": 9,
           "ft_sensors": 18, "action": 9}
SUCCESS = {"success": {"activate": True, "bonus": 500.0, "position_tolerance": 0.05, "orientation_tolerance": 1.0}}


@pytest.fixture(scope="module")
def stored():
    with np.load(rf.PATH) as z:
        return {k: z[k] for k in z.files}


def _np(x):
    return x.detach().cpu().float().numpy() if torch.is_tensor(x) else np.asarray(x)


def _check(key, got, exp, where, extra=None):
    ok, detail = compare(key, _np(got), _np(exp), extra_atol=extra)
    assert ok, (where, key, detail)


def _close_nonfinite_exact(got, want, rtol, atol, where):
    """NaN and +-inf at the same positions, finite values within rtol / atol."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)), (where, "NaN positions")
    inf = np.isinf(want)
    assert np.array_equal(np.isinf(got), inf) and np.array_equal(got[inf], want[inf]), (where, "inf positions")
    fin = np.isfinite(want)
    np.testing.assert_allclose(got[fin], want[fin], rtol=rtol, atol=atol, err_msg=str(where))


# ======== A. batched primitives ========================================================================================
def _nan_rows():
    """Rows the stored inputs lack: NaN alone, next to +-inf and next to the other edge values."""
    x = torch.tensor([[NAN] * 9,
                      [NAN, INF, -INF, NAN, 0.0, -0.0, TINY, 3.4e38, -3.4e38],
                      [INF, NAN, -INF, 1.0, NAN, -1.0, 0.5, NAN, 2.0 ** 100]], dtype=torch.float32)
    q_a = torch.tensor([[NAN, 0.0, 0.0, 1.0], [0.0, 0.0, 0.0, NAN], [NAN, INF, 0.0, 1.0], [INF, 0.0, 0.0, 1.0],
                        [-INF, 1.0, 0.0, 0.0], [3.4e38, 0.0, 0.0, 1.0], [0.5, 0.5, 0.5, 0.5]], dtype=torch.float32)
    q_b = torch.tensor([[0.0, 0.0, 0.0, 1.0], [0.5, 0.5, 0.5, 0.5], [0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 0.0, 1.0],
                        [0.0, 0.0, 0.0, 1.0], [0.0, 0.0, 1.0, 0.0], [NAN, 0.0, 0.0, 1.0]], dtype=torch.float32)
    d = torch.tensor([NAN, INF, -INF, -1e-30, -5.0, 3.4e38, TINY], dtype=torch.float32)
    return x, q_a, q_b, d


def test_rowwise_primitives_on_stored_and_nan_inputs(stored):
    """scale / unscale / saturate bit for bit on the stored rows (0, -0, 1e-42, +-3.4e38, inf) and, against the
    oracle live, on rows with NaN: torch.min / torch.max keep NaN, so saturate must too."""
    import oracle.trifinger_oracle as o
    from leibnizgym_b200.utils import torch_utils as tu
    i = rf.primitive_inputs()
    x_nan = _nan_rows()[0]
    lo, hi = i.lo.cuda(), i.hi.cuda()
    for name in ("scale_transform", "unscale_transform", "saturate"):
        fn = getattr(tu, name)
        assert rf.same(_np(fn(i.x.cuda(), lo, hi)), stored[f"primitives/{name}"]), name
        got, want = _np(fn(x_nan.cuda(), lo, hi)), getattr(o, name)(x_nan, i.lo, i.hi).numpy()
        assert rf.same(got, want), (name, got, want)


def test_quaternion_primitives_on_stored_and_nan_inputs(stored):
    """quat_mul bit for bit; the angle within the asin ulp allowance of test_cuda_primitives, NaN / inf in place."""
    import oracle.trifinger_oracle as o
    from leibnizgym_b200.utils import torch_utils as tu
    i = rf.primitive_inputs()
    _, q_a, q_b, _ = _nan_rows()
    assert rf.same(_np(tu.quat_mul(i.a.cuda(), i.b.cuda())), stored["primitives/quat_mul"])
    assert rf.same(_np(tu.quat_mul(q_a.cuda(), q_b.cuda())), o.quat_mul(q_a, q_b).numpy())
    _close_nonfinite_exact(_np(tu.quat_diff_rad(i.a.cuda(), i.b.cuda())), stored["primitives/quat_diff_rad"],
                           1e-6, 1e-7, "quat_diff_rad stored")
    got = _np(tu.quat_diff_rad(q_a.cuda(), q_b.cuda()))
    want = o.quat_diff_rad(q_a, q_b).numpy()
    assert np.isnan(want).sum() >= 3, want
    _close_nonfinite_exact(got, want, 1e-6, 1e-7, "quat_diff_rad nan rows")


@pytest.mark.parametrize("scale", [50.0, 30.0, 3.0])
def test_lgsk_on_stored_and_nan_inputs(stored, scale):
    """The lgsk kernel at the three scales the stored file holds (0, the 1.78 m knee, overflow to 0, 1e-30), and on
    NaN / +-inf / 3.4e38 / denormal distances against the oracle."""
    import oracle.trifinger_oracle as o
    from leibnizgym_b200.utils import torch_utils as tu
    i = rf.primitive_inputs()
    d = _nan_rows()[3]
    _close_nonfinite_exact(_np(tu.lgsk_kernel(i.d.cuda(), scale)), stored[f"primitives/lgsk_{scale:g}"], 2e-6, 1e-44,
                           ("lgsk stored", scale))
    _close_nonfinite_exact(_np(tu.lgsk_kernel(d.cuda(), scale)), o.lgsk(d, scale).numpy(), 2e-6, 1e-44,
                           ("lgsk nan rows", scale))


# ======== B. planted steps ============================================================================================
def _tile_envs(n):
    """Envs per post-physics CTA for an n-env launch: restates pick_tile_envs (csrc/lg_kernels.cu)."""
    capacity = torch.cuda.get_device_properties(0).multi_processor_count * 4
    if (n + 31) // 32 > capacity:
        return 32
    return next((e for e in (16, 24, 28, 32) if (n + e - 1) // e <= capacity), 32)


def _plant(seq, step, env, tensor, col, value):
    from leibnizgym_b200.synthetic import FINGERTIP_BODIES
    if tensor in ("dof_pos", "dof_vel"):
        seq.dof_state[step, env, col, int(tensor == "dof_vel")] = value
    elif tensor == "obj_pose":
        seq.root_state[step, 4 * env + 2, col] = value
    elif tensor == "obj_vel":
        seq.root_state[step, 4 * env + 2, 7 + col] = value
    elif tensor == "tip_pos":
        seq.rigid_body[step, env, FINGERTIP_BODIES[col // 3], col % 3] = value
    elif tensor == "tip_rest":
        seq.rigid_body[step, env, FINGERTIP_BODIES[col // 10], 3 + col % 10] = value
    elif tensor == "dof_force":
        seq.dof_force[step, env, col] = value
    elif tensor == "ft_sensors":
        seq.ft_sensors[step, env, col] = value
    else:
        seq.action[step, env, col] = value


def _out_col(tensor, col):
    """Column of the states row (the observation row is its first 41 columns) that shows a planted source element."""
    base = {"dof_pos": 0, "dof_vel": 9, "obj_pose": 18, "action": 32, "obj_vel": 41, "dof_force": 86, "ft_sensors": 95}
    if tensor == "tip_pos":
        return 47 + 13 * (col // 3) + col % 3
    if tensor == "tip_rest":
        return 47 + 13 * (col // 10) + 3 + col % 10
    return base[tensor] + col


def _plants(N, E, EP, steps, seed):
    """(step, env, tensor, column, value): every (tensor, value) pair once, each in its own env.  The first envs are
    placed on purpose: four plants in one tile; a value of 2^100 (the fast division's cold path) in the last env of a
    role lane whose other EP - 1 envs stay finite; the last env of a full tile; the last two envs (ragged tile)."""
    rng = random.Random(seed)
    tiles = N // E
    placed = [3 * E, 3 * E + 1, 3 * E + 2, 3 * E + 5, 9 * E + E - 1, N - 1, N - 2]
    pool = [e for e in range(N) if e not in placed and not (6 * E <= e < 6 * E + EP)]
    rng.shuffle(pool)
    assert tiles > 9
    out = [(steps[0], 6 * E + EP - 1, "dof_vel", 4, 2.0 ** 100)]
    for k, (tensor, value) in enumerate(itertools.product(TENSORS, VALUES)):
        env = placed[k] if k < len(placed) else pool[k]
        out.append((steps[k % len(steps)], env, tensor, rng.randrange(TENSORS[tensor]), value))
    return out


def _angle_allowance(ora):
    """tests/test_cuda_vs_oracle._angle_allowance_small; a NaN angle (whose terms are NaN on both sides) adds none."""
    cur = np.nan_to_num(angle_slack(ora.obj_hist[0][:, 3:7], ora.goal_poses[:, 3:7]), nan=0.0)
    prev = np.nan_to_num(angle_slack(ora.obj_hist[1][:, 3:7], ora.goal_poses[:, 3:7]), nan=0.0)
    t = ora.terms
    rot = abs(t["object_rot"]["weight"]) * 0.02 / t["object_rot"]["scale"] * cur
    delta = abs(t["object_rot_delta"]["weight"]) * (cur + prev)
    terms = np.zeros((6, len(cur)))
    terms[3], terms[4] = rot, delta
    return terms, rot * t["object_rot"]["activate"] + delta * t["object_rot_delta"]["activate"]


def _check_info(info, ora_info, where, extra=None):
    """`_step_info` against the oracle's: counts exact, means within the parity bound (plus `extra[key]`, a
    data-dependent allowance), NaN / inf of the same kind."""
    assert set(ora_info) <= set(info), (where, sorted(ora_info))
    for k, v in ora_info.items():
        got, exp = float(info[k]), float(v)
        if k.endswith("/count"):
            assert got == exp, (where, k, got, exp)
        elif math.isfinite(exp):
            assert abs(got - exp) <= 1e-5 * abs(exp) + 1.35e-4 + (extra or {}).get(k, 0.0), (where, k, got, exp)
        else:
            assert got == exp or (math.isnan(got) and math.isnan(exp)), (where, k, got, exp)


class _Lockstep:
    """One CUDA env (or several shards of one) and the oracle over the same sequence, with the same injected draws
    (reset / goal-reset rows in ascending-id order, split by shard)."""

    def __init__(self, cfg, seq, world=1, seed=0):
        from leibnizgym_b200.config import resolve_config
        from leibnizgym_b200.env import TrifingerEnv
        from leibnizgym_b200.sim import SyntheticSim
        from leibnizgym_b200.synthetic import StateSequence
        from oracle.trifinger_oracle import OracleEnv, OracleSim
        N = seq.num_envs
        self.N, self.n, self.seq = N, N // world, seq
        self.ora = OracleEnv(resolve_config(cfg), OracleSim(seq, N))
        self.envs, self.shard_seqs = [], []
        for r in range(world):
            lo, hi = r * self.n, (r + 1) * self.n
            sq = StateSequence(seq.dof_state[:, lo:hi], seq.root_state[:, 4 * lo:4 * hi], seq.rigid_body[:, lo:hi],
                               seq.dof_force[:, lo:hi], seq.ft_sensors[:, lo:hi], seq.action[:, lo:hi])
            sq = StateSequence(*(x.contiguous() for x in (sq.dof_state, sq.root_state, sq.rigid_body, sq.dof_force,
                                                          sq.ft_sensors, sq.action))).to("cuda:0")
            env = TrifingerEnv(cfg, device="cuda:0", verbose=False, sim=SyntheticSim(sq, "cuda:0"), rank=r,
                               world_size=world)
            env.enable_term_rewards(True)
            self.envs.append(env)
            self.shard_seqs.append(sq)
        self.g = torch.Generator().manual_seed(seed)

    def _draws(self, k):
        return torch.rand(k, 24, generator=self.g).numpy(), torch.randn(k, 8, generator=self.g).numpy()

    def inject(self, rmask, gmask):
        kr, kg = int(rmask.sum()), int(gmask.sum())
        dr, dg = (self._draws(kr) if kr else None), (self._draws(kg) if kg else None)
        self.ora.inject_draws(reset=dr, goal=dg)
        for r, env in enumerate(self.envs):
            def rows(d, m):
                if d is None:
                    return None
                a, b = int(m[:r * self.n].sum()), int(m[:(r + 1) * self.n].sum())
                return tuple(x[a:b] for x in d)
            env.inject_draws(reset=rows(dr, rmask), goal=rows(dg, gmask))

    def reset(self, reset_fn=None):
        self.inject(torch.ones(self.N, dtype=torch.bool), torch.zeros(self.N, dtype=torch.bool))
        for env in self.envs:
            (reset_fn or env.reset)()
        self.ora.reset()

    def force_and_inject(self, mask):
        self.ora.reset_buf |= mask
        for r, env in enumerate(self.envs):
            env._reset_buf |= mask[r * self.n:(r + 1) * self.n].cuda()
        self.inject(self.ora.reset_buf.clone(), self.ora.goal_reset_buf.clone())


@pytest.mark.parametrize("N, asym, mode, route", [
    (16384, True, "position", "wrapper"),
    (16384, False, "torque", "wrapper_bf16"),
    (4099, True, "torque", "raw"),
    (4099, False, "position", "raw"),
    (4099, True, "position", "wrapper_bf16"),
    (4099, True, "torque", "hooks"),
])
def test_planted_non_finite_and_extreme_values_match_oracle(N, asym, mode, route):
    """Every source tensor gets NaN, +-inf, +-3.4e38, 2^100, the float below 2^100, +-1e-42 and -0.0 somewhere, at
    steps 1-3.  Every step: obs, states, (clipped, bf16) outputs, action_buf, applied torque, the six terms, reward,
    flags, counters, reset ids and `_step_info` against the oracle; the planted columns of obs / states bit for bit
    (except the denormals, which the fast division may round by 1 ulp).  Half of the poisoned envs are reset on the
    next step: a NaN fingertip stays in the reward for exactly one more step (the stale history entry, SURVEY.md §C2)."""
    from leibnizgym_b200.config import difficulty_config
    from leibnizgym_b200.env import IsaacEnvBase
    from leibnizgym_b200.synthetic import make_sequence
    from leibnizgym_b200.wrappers import VecTaskPython
    T = 6
    E = _tile_envs(N)
    EP = E // (2 if asym else 4)
    cfg = difficulty_config(4, N, asymmetric_obs=asym, seed=N % 97, episode_length=4, command_mode=mode,
                            termination_conditions=copy.deepcopy(SUCCESS))
    seq = make_sequence(300 + N, T, N)
    plants = _plants(N, E, EP, (1, 2, 3), seed=N + len(route))
    for p in plants:
        _plant(seq, *p)
    ls = _Lockstep(cfg, seq, seed=N)
    env, ora = ls.envs[0], ls.ora
    wrapped = route.startswith("wrapper")
    vec = None
    if wrapped:
        vec = VecTaskPython(env, rl_device="cuda:0", clip_obs=5.0, clip_actions=1.0,
                            obs_dtype=torch.bfloat16 if route == "wrapper_bf16" else torch.float32)
    ls.reset(vec.reset if wrapped else None)
    clip = lambda x: torch.clamp(x, -5.0, 5.0)  # noqa: E731
    reset_next = [p for k, p in enumerate(plants) if k % 2]      # these envs are reset on the step after their plant
    stale_tip = [p for p in reset_next if p[2] == "tip_pos" and math.isnan(p[4])]
    assert stale_tip
    for t in range(1, T):
        mask = torch.zeros(N, dtype=torch.bool)
        for p in reset_next:
            if p[0] == t - 1:
                mask[p[1]] = True
        ls.force_and_inject(mask)
        act = seq.action[t]
        if wrapped:
            _, _, done, _ = vec.step(act.cuda())
            _, _, ora_done, _ = ora.step(torch.clamp(act, -1.0, 1.0))
        elif route == "raw":
            _, _, done, _ = env.step(act.cuda())
            _, _, ora_done, _ = ora.step(act.clone())
        else:
            _, _, done, _ = IsaacEnvBase.step(env, act.cuda())
            _, _, ora_done, _ = ora.step(act.clone())
        w = (N, asym, mode, route, t)
        _check("obs", env.obs_buf, ora.obs_buf, w)
        if asym:
            _check("states", env.states_buf, ora.states_buf, w)
        assert rf.same(_np(env.action_buf), ora.action_buf.numpy()), (w, "action_buf")
        _check("applied_torque", env._applied_torque, ora.applied_torque, w)
        slack_terms, slack_reward = _angle_allowance(ora)
        _check("terms", env._term_rewards[:6], ora.last_terms, w, slack_terms)
        _check("reward", env.reward_buf, ora.reward_buf, w, slack_reward)
        _check("reset_buf", env._reset_buf, ora.reset_buf, w)
        _check("goal_reset_buf", env._goal_reset_buf, ora.goal_reset_buf, w)
        _check("successes", env._successes, ora.successes, w)
        _check("steps_count", env._steps_count_buf, ora.steps_count_buf, w)
        assert torch.equal(done.cpu(), ora_done), (w, "dones")
        if route != "hooks":
            _check("reset_ids", env.reset_env_ids, ora.last_ids[0], w)
            _check("goal_reset_ids", env.goal_reset_env_ids, ora.last_ids[1], w)
        _check_info(env._step_info, ora.step_info, w)
        outs = [(env.obs_buf, ora.obs_buf, env._obs_clipped, env._obs_bf16)]
        if asym:
            outs.append((env.states_buf, ora.states_buf, env._states_clipped, env._states_bf16))
        for raw, want, clipped, bf16 in outs:
            if wrapped:
                _check("obs", clipped, clip(want), w + ("clipped",))
            if bf16 is not None:
                # NaN where the oracle's clipped output is NaN, elsewhere the bits of the kernel's own fp32 output rounded
                nan_want = torch.isnan(clip(want))
                assert torch.equal(torch.isnan(bf16.float()).cpu(), nan_want), (w, "bf16 NaN positions")
                keep = ~nan_want.cuda()
                assert torch.equal(bf16.view(torch.int16)[keep], clipped.to(torch.bfloat16).view(torch.int16)[keep]), w
        for step, e, tensor, col, value in plants:
            oc = _out_col(tensor, col)
            if step != t or abs(value) == TINY or (oc >= 41 and not asym):
                continue
            src, ref = (env.states_buf, ora.states_buf) if asym else (env.obs_buf, ora.obs_buf)
            assert rf.same(_np(src[e, oc]), ref[e, oc].numpy()), (w, "planted", tensor, col, value,
                                                                   float(src[e, oc]), float(ref[e, oc]))
        # the stale fingertip history: NaN the step after the plant although the env was reset, gone the step after
        for step, e, *_ in stale_tip:
            if t == step + 1:
                assert math.isnan(float(env._term_rewards[1, e])), (w, e)
            elif t == step + 2:
                assert math.isfinite(float(env._term_rewards[1, e])), (w, e)


# ======== C. exact episode statistics ==================================================================================
def _check_stats(stats, terms, reward, resets, dones, succ, active, n, ctas, where):
    """The statistics vector of one shard against its per-env outputs.  A float mean is the fixed-point sum (each value
    rounded to 2^-30, so at most 2^-31 off per env and in the mean) over the CTAs, converted to fp64 (exact, or two
    roundings with a non-power-of-two env count) and added up by fp64 atomics (one rounding per CTA; the cold CTAs'
    butterflies add five): |error| <= 2^-31 + (ctas + 32) 2^-53 sum|x| / n.  Counts are exact; inactive terms are 0."""
    u = 2.0 ** -53

    def mean(slot, x):
        x = np.asarray(x, np.float64)
        s = x.sum()
        got = float(stats[slot])
        if not np.isfinite(s):
            assert got == s or (math.isnan(got) and math.isnan(s)), (where, slot, got, s)
            return
        want = math.fsum(x) / n
        assert abs(got - want) <= 2.0 ** -31 + (ctas + 32) * u * np.abs(x).sum() / n, (where, slot, got, want)

    for k in range(7):
        if active[k]:
            mean(k, terms[k])
        else:
            assert stats[k] == 0.0, (where, k, stats[k])
    mean(10, reward)
    c = float(np.sum(succ))
    assert abs(stats[9] - c / n) <= (ctas + 8) * u * c / n, (where, "successes", stats[9], c / n)
    assert stats[11] == float(np.sum(resets)), (where, "resets", stats[11], np.sum(resets))
    assert stats[12] == float(np.sum(dones)), (where, "dones", stats[12], np.sum(dones))


def _goal_counts(ora, lo, hi):
    """Per-env position / orientation checks of the oracle's termination (trifinger_env.py:1053-1068), for a range."""
    from oracle.trifinger_oracle import quat_diff_rad
    tol = ora.cfg["termination_conditions"]["success"]
    o0, g = ora.obj_hist[0][lo:hi], ora.goal_poses[lo:hi]
    pos = torch.le(torch.norm(g[:, 0:3] - o0[:, 0:3], p=2, dim=-1), tol["position_tolerance"])
    rot = torch.le(quat_diff_rad(o0[:, 3:7], g[:, 3:7]), tol["orientation_tolerance"])
    return float(pos.sum()), float(rot.sum())


def _teleport(seq):
    """One env in every 97 moves a fingertip by 1e4 m at steps 1 and 3: finger_move_penalty ~ -2.5e10 > 2^28, so those
    CTAs sum in fp64 while the other CTAs of the same launch stay in fixed point."""
    seq.rigid_body[1::2, ::97, 6, 0] += 1.0e4


def _non_finite(seq):
    """Step 2: finger_reach_object_rate is +inf in env 11 (its previous fingertip was at 3.4e38) and -inf in env 3000
    (its current one is): the mean is NaN.  Env 20 has a NaN object orientation: object_rot is NaN."""
    seq.rigid_body[1, 11, 11, 1] = 3.4e38
    seq.rigid_body[2, 3000, 16, 2] = 3.4e38
    seq.root_state[2, 4 * 20 + 2, 4] = NAN


@pytest.mark.parametrize("case, N, world, plant", [
    ("pow2", 16384, 1, None),
    ("factor_ragged", 12345, 1, None),
    ("one_env", 1, 1, None),
    ("two_shards", 12346, 2, None),
    ("cold_ctas", 16384, 1, _teleport),
    ("non_finite", 4096, 1, _non_finite),
])
def test_step_statistics_are_exact_sums_of_the_per_env_outputs(case, N, world, plant):
    """`_step_stats` of every shard against the fp64 sums of the same launch's per-env terms, reward and flags, and the
    position / orientation counts against the oracle; the non-finite case also against the oracle's NaN / -inf means."""
    from leibnizgym_b200.config import difficulty_config
    from leibnizgym_b200.synthetic import make_sequence
    T = 5
    cfg = difficulty_config(4, N, asymmetric_obs=True, seed=3, episode_length=3,
                            termination_conditions=copy.deepcopy(SUCCESS))
    seq = make_sequence(500 + N, T, N)
    if plant is not None:
        plant(seq)
    ls = _Lockstep(cfg, seq, world=world, seed=N)
    ls.reset()
    active = [bool(cfg["reward_terms"].get(k, {}).get("activate")) for k in
              ("finger_reach_object_rate", "finger_move_penalty", "object_dist", "object_rot", "object_rot_delta",
               "object_move")] + [False]
    n = ls.n
    seen_cold = seen_nan = False
    for t in range(1, T):
        ls.force_and_inject(torch.zeros(N, dtype=torch.bool))
        for r, env in enumerate(ls.envs):
            env.step(ls.shard_seqs[r].action[t])
        ls.ora.step(seq.action[t].clone())
        for r, env in enumerate(ls.envs):
            w = (case, t, r)
            stats = env._step_stats.cpu().numpy()
            terms = env._term_rewards.cpu().numpy()
            _check_stats(stats, terms, _np(env.reward_buf), _np(env._reset_buf), _np(env._dones), _np(env._successes),
                         active, n, -(-n // _tile_envs(n)), w)
            pos, rot = _goal_counts(ls.ora, r * n, (r + 1) * n)
            assert (stats[7], stats[8]) == (pos, rot), (w, stats[7:9], pos, rot)
            seen_cold |= bool(np.abs(terms[1]).max() >= 2.0 ** 28)
            seen_nan |= bool(np.isnan(stats[0]))
        if world == 1:
            _check_info(ls.envs[0]._step_info, ls.ora.step_info, (case, t))
    if plant is _teleport:
        assert seen_cold
    if plant is _non_finite:
        assert seen_nan


def test_step_statistics_of_the_chunked_host_pipeline():
    """The chunked host pipeline (three chunks of 4096 envs, statistics denominator 12 288: a power-of-two chunk in a
    non-power-of-two shard) against the per-env outputs of the same step taken whole by a twin env."""
    from leibnizgym_b200.config import difficulty_config
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    from leibnizgym_b200.wrappers import VecTaskPython
    N, T = 12288, 5
    cfg = difficulty_config(4, N, asymmetric_obs=True, seed=17, episode_length=2,
                            termination_conditions=copy.deepcopy(SUCCESS))
    host = make_sequence(62, T, N).to("cpu", pin=True)
    g = torch.Generator().manual_seed(5)
    d = (torch.rand(N, 24, generator=g).numpy(), torch.randn(N, 8, generator=g).numpy())

    def build(chunks):
        sim = SyntheticSim(host, "cuda:0")
        env = TrifingerEnv(cfg, device="cuda:0", verbose=False, sim=sim)
        sim.use_sparse_upload(env._P)
        vec = VecTaskPython(env, rl_device="cpu" if chunks else "cuda:0", host_pipeline_chunks=chunks)
        env.inject_draws(reset=d)
        vec.reset()
        return env, vec

    twin, plain = build(0)
    twin.enable_term_rewards(True)
    env, piped = build(3)
    active = [True, True, True, True, False, False, False]
    for t in range(1, T):
        plain.step(host.action[t])
        piped.step(host.action[t])
        torch.cuda.synchronize()
        assert torch.equal(twin._reset_buf, env._reset_buf) and torch.equal(twin.reward_buf, env.reward_buf)
        stats, ref = env._step_stats.cpu().numpy(), twin._step_stats.cpu().numpy()
        _check_stats(stats, twin._term_rewards.cpu().numpy(), _np(twin.reward_buf), _np(twin._reset_buf),
                     _np(twin._dones), _np(twin._successes), active, N, -(-N // 16) + 16, ("host pipeline", t))
        assert (stats[7], stats[8]) == (ref[7], ref[8]), t


# ======== D. stored reward-term cases through the fused kernel ==========================================================
@pytest.mark.parametrize("seed", rf.REWARD_SEEDS)
def test_stored_reward_terms_through_the_fused_kernel(stored, seed):
    """The six terms of tests/golden/reference_functions.py (random weights, scales and schedule windows; objects on
    the goal, fingertips in the cube centre) at every stored env-step count, written into the simulator rows, the goal
    buffer and the history entry and run through lg_post_physics.  The stored arrays were recorded from the oracle,
    whose arithmetic the reference's scripted reward modules reproduced bit for bit (see that file's docstring).
    Where a schedule gate is closed (outside [start, end]) the term is exactly 0."""
    import oracle.trifinger_oracle as o
    from leibnizgym_b200.config import difficulty_config
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    i = rf.reward_inputs(seed)
    N = rf.N_REWARD
    cfg = difficulty_config(4, N, asymmetric_obs=True, seed=seed)
    cfg["reward_terms"] = copy.deepcopy(i.cfg)
    env = TrifingerEnv(cfg, device="cuda:0", verbose=False, sim=SyntheticSim(make_sequence(seed, 2, N).to("cuda:0"),
                                                                             "cuda:0"))
    env.enable_term_rewards(True)
    P = o.reward_term_params(i.cfg)
    hist = torch.cat([i.tips_prev[:, :, 0:3].reshape(N, 9), i.obj_prev[:, 0:7]], dim=1).cuda()
    cur = angle_slack(i.obj[:, 3:7], i.goal[:, 3:7])
    prev = angle_slack(i.obj_prev[:, 3:7], i.goal[:, 3:7])
    for n, T in enumerate(i.steps):
        env._actors_root_state.view(N, 4, 13)[:, 2] = i.obj.cuda()
        env._rigid_body_state[:, [6, 11, 16]] = i.tips.cuda()
        env._object_goal_poses_buf.copy_(i.goal)
        env._history.copy_(hist)    # the kernel shifts the history: rewritten before every call
        env._call("lg_post_physics", env._P, env._S, env._B, float(T))
        got = env._term_rewards[:6].cpu().numpy()
        for k, name in enumerate(o.TERM_ORDER):
            p = P[name]
            want = stored[f"reward{seed}/{name}/T{n}"]
            gate = o._ramp(p["start"], p["end"], T) if name == "object_rot_delta" else o._gate(p["start"], p["end"], T)
            w = (seed, name, T)
            if name in ("finger_reach_object_rate", "object_dist", "object_rot", "object_rot_delta") and gate == 0.0:
                assert np.all(got[k] == 0.0) and np.all(want == 0.0), w
                continue
            extra = None
            if name == "object_rot":
                extra = abs(p["weight"]) * rf.DT * gate / p["scale"] * cur
            elif name == "object_rot_delta":
                extra = abs(p["weight"]) * gate * (cur + prev)
            _check("terms", got[k], want, w, extra)
