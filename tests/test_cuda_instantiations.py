"""Every instantiation of the two fused kernels that the launcher can pick (csrc/lg_kernels.cu: pick_tile_envs,
launch_post, launch_pre), each tested where it is picked, and each case checked to have launched the kernel it names.

  a. which kernel ran: torch.profiler names the instantiation; the coverage test matches the library's own symbol
     table against the instantiations the cases below claim;
  b. oracle parity (tests/lockstep.py: every output, every step) at the launcher's own choice, for every post-physics tile size with ragged tiles of
     nvalid in {1, EP - 1, EP, EP + 1, E - 1} envs (EP = envs per role-lane part), every pre-physics grid regime,
     action_dim 9 and 18; the torch stream's fused step against its hook-by-hook step in every pre-physics regime;
  c. bit-exact invariance with every extension on across forced tile sizes, forced pre-physics paths, PDL off, two
     shards split inside a noise group, graph replay with the device clock, and the hook-by-hook route
     (tests/instantiation_digest.py, one process per forced setting);
  d. DR observation noise and offsets next to a diverged env: the lane's other envs keep their perturbed observations
     bit for bit, and the diverged env's IEEE redo keeps its offset.
"""
import copy
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from instantiation_digest import DEFAULT as DIGEST_SCENARIOS
from instantiation_digest import kernel_args, launched
from lockstep import Lockstep, rf_same
from test_cuda_edges import SUCCESS, _np, _tile_envs

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
KINDS = ("1", "EP-1", "EP", "EP+1", "E-1")
# pre-physics regime -> (TICKET, MINB, SPLIT, DIRECT) of pre_physics_kernel<A, TICKET, MINB, SPLIT, DIRECT, TORCH>
PRE = {"ticket": (1, 6, 0, 0), "direct": (0, 3, 1, 1), "small": (0, 3, 1, 0), "minb4": (0, 4, 1, 0)}
REGIMES_32 = {True: ("small", "small", "small", "minb4", "ticket"), False: ("small", "small", "ticket", "small", "minb4")}


def _regime_of(E, k):
    """Pre-physics regime pinned by the k-th nvalid case of tile size E (env counts in E's range allow these)."""
    return {16: ("small",) * 3 + ("direct",) * 2, 24: ("direct",) * 5, 28: ("direct",) * 3 + ("small",) * 2}.get(E)[k]


def _cases_a9():
    """(asym, E, nvalid kind, clip, ext, regime): all 32 (ASYM, CLIP, E, EXT) combinations, five ragged sizes each."""
    out = []
    for asym in (True, False):
        for E in (16, 24, 28, 32):
            combos = [(False, False), (False, True), (True, False), (True, True), ((E // 8 + asym) % 2 == 0, True)]
            for k, kind in enumerate(KINDS):
                regime = REGIMES_32[asym][k] if E == 32 else _regime_of(E, k)
                out.append((asym, E, kind, *combos[k], regime))
    return out


CASES_A9 = _cases_a9()
CASES_A18 = [(asym, clip, ext, regime) for (asym, clip, ext), regime in zip(
    [(a, c, x) for a in (True, False) for c in (False, True) for x in (False, True)],
    ("small", "direct", "minb4", "ticket", "ticket", "minb4", "direct", "small"))]
TORCH_CASES = [(A, r) for A in (9, 18) for r in ("small", "direct", "minb4", "ticket")]


def _claims():
    """Instantiations the cases of this file assert they launched: ('post', (A, ASYM, REWARD, CLIP, E, EXT)) and
    ('pre', (A, TICKET, MINB, SPLIT, DIRECT, TORCH)).  REWARD = 0 is what reset() launches (lg_fill_observations)."""
    out = set()
    for asym, E, _, clip, ext, regime in CASES_A9:
        out |= {("post", (9, int(asym), r, int(clip), E, int(ext))) for r in (0, 1)} | {("pre", (9, *PRE[regime], 0))}
    for asym, clip, ext, regime in CASES_A18:
        out |= {("post", (18, int(asym), r, int(clip), 32, int(ext))) for r in (0, 1)} | {("pre", (18, *PRE[regime], 0))}
    out |= {("pre", (A, *PRE[r], 1)) for A, r in TORCH_CASES}
    return out


# ======== geometry: the launcher's thresholds, from the device ============================================================
def _device():
    from leibnizgym_b200 import _native as nat
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    return sm, int(nat.load().lg_pre_resident_tiles())


def _nvalid(kind, E, asym):
    EP = E // (2 if asym else 4)
    return {"1": 1, "EP-1": EP - 1, "EP": EP, "EP+1": EP + 1, "E-1": E - 1}[kind]


def _pick_n(A, E, nvalid, regime):
    """Smallest env count of at least ~1000 whose last post-physics tile holds `nvalid` envs, whose tile size is E
    (A = 9) and whose pre-physics grid falls in `regime`; for "minb4" the largest count whose grid is still co-resident
    at the MINB = 4 occupancy (beyond the 3-per-SM grids of the latency-tuned instantiation).  None: not on this device."""
    sm, resident = _device()

    def ok(n):
        tiles = -(-n // 128)
        if A == 9 and E is not None and _tile_envs(n) != E:
            return False
        if regime == "ticket":
            return tiles > resident
        if regime == "direct":
            return 32 <= tiles <= min(128, sm)
        if regime == "minb4":
            return tiles == resident and tiles > 3 * sm
        return tiles <= 3 * sm and not 32 <= tiles <= min(128, sm)

    step = E or 32
    cands = range(1024 - 1024 % step + nvalid, (resident + 2) * 128, step)
    return next((n for n in (reversed(cands) if regime == "minb4" else cands) if ok(n)), None)


def _expect(got, post=None, pre=None, where=None):
    if post is not None:
        assert got["post"] == set(post), (where, "post-physics instantiations", sorted(got["post"]), sorted(post))
    if pre is not None:
        assert got["pre"] == set(pre), (where, "pre-physics instantiations", sorted(got["pre"]), sorted(pre))


# ======== a. the library's instantiations, all claimed ====================================================================
def test_every_built_instantiation_is_claimed_by_a_case():
    """cuobjdump -symbols of the built library, demangled: every post_physics_kernel / pre_physics_kernel instantiation
    it contains is one that a case of this file launches (and asserts it launched)."""
    from leibnizgym_b200 import _native as nat
    cuda = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    tools = [shutil.which(t) or os.path.join(cuda, "bin", t) for t in ("cuobjdump", "cu++filt")]
    missing = [t for t in tools if not os.path.exists(t)]
    if missing:
        pytest.skip(f"CUDA binary tools not found: {missing}")
    if not os.path.exists(nat.LIB_PATH):
        pytest.skip(f"library not built: {nat.LIB_PATH}")
    syms = subprocess.run([tools[0], "-symbols", nat.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = sorted({line.split()[-1] for line in syms.splitlines()
                    if "STO_ENTRY" in line and re.search(r"(post|pre)_physics_kernel", line)})
    demangled = subprocess.run([tools[1]], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    built = {kernel_args(line) for line in demangled.splitlines()} - {None}
    assert len(built) == len(names) and len(built) >= 96, (len(built), len(names))
    claims = _claims()
    assert not built - claims, ("built but not launched by any case", sorted(built - claims))
    assert not claims - built, ("claimed but not in the library", sorted(claims - built))


# ======== b. oracle parity per geometry ===================================================================================
def _lockstep(A, N, asym, clip, ext, post_E, pre, where):
    """Reset + 4 steps against the oracle (tests/lockstep.py) with 30 % forced resets and 5 % forced goal resets;
    ext: keypoint term, moving goal (integrated on both sides), bf16.  reset() and the first step run under the
    profiler."""
    from leibnizgym_b200.config import difficulty_config
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence
    seed, T = N % 1000 + 7 * A, 5
    extra = {"goal_movement": {"rotation": {"activate": True, "rate_magnitude": 0.5}}} if ext else {}
    cfg = difficulty_config(4, N, asymmetric_obs=asym, seed=seed % 97, episode_length=3,
                            command_mode="torque" if A == 9 else "position_impedance",
                            termination_conditions=copy.deepcopy(SUCCESS), **extra)
    run = Lockstep(cfg, make_sequence(seed, T, N, action_dim=A), bernoulli_masks(seed + 1, T, N, 0.3),
                   bernoulli_masks(seed + 2, T, N, 0.05), seed, clip=clip, bf16=ext, keypoint=ext, goal_integration=ext)
    got = launched(run.reset)
    flags = {}
    got1 = launched(lambda: flags.update(r=run.step(1)))
    got["post"] |= got1["post"]
    got["pre"] |= got1["pre"]
    post = {(A, int(asym), r, int(clip), post_E, int(ext)) for r in (0, 1)}
    _expect(got, post=post, pre={(A, *PRE[pre], 0)}, where=where)
    run.check(1, *flags["r"], where)
    for t in range(2, T):
        run.check(t, *run.step(t), where)


@pytest.mark.gpu
@pytest.mark.parametrize("asym, E, kind, clip, ext, regime", CASES_A9,
                         ids=[f"{'a' if c[0] else 's'}-E{c[1]}-nv[{c[2]}]-{'clip' if c[3] else 'raw'}"
                              f"-{'ext' if c[4] else 'plain'}-{c[5]}" for c in CASES_A9])
def test_post_tile_geometry_matches_oracle(asym, E, kind, clip, ext, regime):
    """action_dim 9: the post-physics instantiation of tile size E with a ragged last tile of `kind` envs, and the
    pre-physics instantiation of `regime`, both as the launcher picks them, against the oracle."""
    nvalid = _nvalid(kind, E, asym)
    N = _pick_n(9, E, nvalid, regime)
    if N is None:
        pytest.skip(f"no env count gives tile size {E} with the {regime} pre-physics grid on this device")
    assert N % E == nvalid and _tile_envs(N) == E
    _lockstep(9, N, asym, clip, ext, E, regime, (N, asym, E, kind, clip, ext, regime))


@pytest.mark.gpu
@pytest.mark.parametrize("asym, clip, ext, regime", CASES_A18)
def test_position_impedance_matches_oracle(asym, clip, ext, regime):
    """action_dim 18 (position_impedance): every post-physics instantiation (E = 32) and the four pre-physics
    regimes against the oracle."""
    N = _pick_n(18, 32, 17, regime)
    if N is None:
        pytest.skip(f"no {regime} pre-physics grid on this device")
    _lockstep(18, N, asym, clip, ext, 32, regime, (N, asym, clip, ext, regime))


@pytest.mark.gpu
@pytest.mark.parametrize("A, regime", TORCH_CASES)
def test_torch_stream_fused_step_equals_hooks(A, regime):
    """"rng_stream": "torch": the fused step (TORCH pre-physics instantiation of each regime) against the hook-by-hook
    step, bit for bit, for action_dim 9 and 18."""
    from leibnizgym_b200.env import IsaacEnvBase
    from test_cuda_torch_rng import _cfg, _compare_envs, _env, _masks
    N = _pick_n(A, None, 5, regime)
    if N is None:
        pytest.skip(f"no {regime} pre-physics grid on this device")
    cfg = _cfg(N, difficulty=4, rot=True, asym=True)
    if A == 18:
        cfg["command_mode"] = "position_impedance"
    fused, seq = _env(cfg)
    hooks, _ = _env(cfg)
    if A == 18:   # _env's sequence carries 9 action columns
        from leibnizgym_b200.synthetic import make_sequence
        seq = make_sequence(3, 4, N, action_dim=18)
    rmask, gmask = _masks(N, 3, 0.3, 5), _masks(N, 3, 0.05, 6)
    for t in range(3):
        for e in (fused, hooks):
            e._reset_buf |= rmask[t]
            e._goal_reset_buf |= gmask[t]
        a = seq.action[t].cuda()
        if t == 0:
            got = launched(lambda: fused.step(a))
            E = _tile_envs(N) if A == 9 else 32
            _expect(got, post={(A, 1, 1, 0, E, 1)}, pre={(A, *PRE[regime], 1)}, where=(A, regime, N))
        else:
            fused.step(a)
        IsaacEnvBase.step(hooks, a)
        _compare_envs(fused, hooks, (A, regime, N, t))


# ======== c. bit-exact invariance with every extension on ==================================================================
SETTINGS = [{"LG_TILE_ENVS": "16"}, {"LG_TILE_ENVS": "24"}, {"LG_TILE_ENVS": "28"}, {"LG_TILE_ENVS": "32"},
            {"LG_PRE_TICKET": "1"}, {"LG_PRE_DIRECT": "0"}, {"LG_PDL": "0"}]
FORCED_SCENARIOS = [s for s in DIGEST_SCENARIOS if s.split(":")[-1] in ("eager", "graph", "host") and ":8198:" not in s]


def _digest_run(env_vars, scenarios):
    env = {k: v for k, v in os.environ.items() if k not in ("LG_TILE_ENVS", "LG_PRE_TICKET", "LG_PRE_DIRECT", "LG_PDL",
                                                            "LG_NO_PDL")}
    env.update(env_vars)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.join(HERE, "instantiation_digest.py")]
    res = subprocess.run(cmd + scenarios, capture_output=True, text=True, env=env, cwd=ROOT, timeout=1200)
    assert res.returncode == 0, (env_vars, res.stdout[-2000:], res.stderr[-4000:])
    out = {}
    for line in res.stdout.splitlines():
        if line.startswith("{"):
            d = json.loads(line)
            d["launched"] = {k: {tuple(x) for x in v} for k, v in d["launched"].items()}
            out[d["scenario"]] = d
    assert sorted(out) == sorted(scenarios), (env_vars, sorted(out))
    return out


@pytest.fixture(scope="module")
def default_digests():
    return _digest_run({}, list(DIGEST_SCENARIOS))


def _same_stats(a, b, n, where):
    """`_step_stats`: bit for bit for a power-of-two env count; otherwise each CTA's fp64 scaling and the order of the
    fp64 atomics may differ, to the fixed-point resolution of tests/test_cuda_edges._check_stats."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    if n & (n - 1) == 0:
        assert np.array_equal(a, b), (where, a, b)
    else:
        assert np.all(np.abs(a - b) <= 2.0 ** -30 + 1e-12 * np.abs(b)), (where, a, b)


def _same_episode_stats(a, b, where):
    """`_episode_stats` + `_episode_term_stats`: the count, length sum and success count exact; the return sums, whose
    CTA partition differs between forced tile sizes, to the fixed-point resolution per record."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    exact = [0, 2, 3]
    assert np.array_equal(a[exact], b[exact]), (where, a, b)
    rest = [i for i in range(len(b)) if i not in exact]
    assert np.all(np.abs(a[rest] - b[rest]) <= 2.0 ** -30 * b[0] + 1e-12 * np.abs(b[rest])), (where, a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("setting", SETTINGS, ids=[",".join(f"{k}={v}" for k, v in s.items()) for s in SETTINGS])
def test_forced_launch_paths_are_bit_identical(default_digests, setting):
    """Each forced tile size / pre-physics path / PDL off, own and torch stream, eager and graph replay: every buffer
    group (episode buffers and DR offset rows included) equal to the launcher's own choice; the forced instantiation
    is the one that ran."""
    forced = _digest_run(setting, FORCED_SCENARIOS)
    for name in FORCED_SCENARIOS:
        got, ref = forced[name], default_digests[name]
        assert got["digests"] == ref["digests"], (setting, name, got["digests"], ref["digests"])
        _same_stats(got["stats"], ref["stats"], int(name.split(":")[3]), (setting, name))
        _same_episode_stats(got["episode_stats"], ref["episode_stats"], (setting, name))
        post, pre = got["launched"]["post"], got["launched"]["pre"]
        if name.endswith(":graph"):
            continue
        assert post and pre, (setting, name)
        if "LG_TILE_ENVS" in setting and ":9:" in name:
            assert {p[4] for p in post} == {int(setting["LG_TILE_ENVS"])}, (setting, name, post)
        if "LG_PRE_TICKET" in setting:
            assert all(p[1] == 1 for p in pre), (setting, name, pre)
        if "LG_PRE_DIRECT" in setting:
            assert all(p[4] == 0 for p in pre), (setting, name, pre)
    # the defaults of these env counts take other paths than the forced ones, so each comparison means something
    if "LG_PRE_DIRECT" in setting:
        assert any(p[4] == 1 for d in default_digests.values() for p in d["launched"]["pre"])
    if "LG_TILE_ENVS" in setting:
        assert any(p[4] != int(setting["LG_TILE_ENVS"]) for d in default_digests.values() for p in d["launched"]["post"])


@pytest.mark.gpu
def test_graph_shard_and_route_equivalence(default_digests):
    """Graph replay with the device clock == eager steps with the host clock (the noise epoch comes from reward_coef
    instead of LgCoef); two shards of 4099 envs (a noise group of 4 envs straddles the boundary) == one of 8198 except
    the per-shard ids and statistics; the fused step == the hook-by-hook step with DR observation noise, keypoint,
    moving goal and bf16 on (no action noise: the hook route refuses it)."""
    d = default_digests
    for a in ("ext:a:9:12344:own", "ext:s:9:16376:own", "ext:a:18:12344:own"):
        g, h = d[a + ":graph"], d[a + ":host"]
        assert g["digests"] == h["digests"], (a, g["digests"], h["digests"])
        _same_stats(g["stats"], h["stats"], int(a.split(":")[3]), a)
        _same_episode_stats(g["episode_stats"], h["episode_stats"], a)
    drop = lambda x, keys: {k: v for k, v in x.items() if k not in keys}  # noqa: E731
    one, two = d["ext:a:9:8198:own:eager"]["digests"], d["ext:a:9:8198:own:shards"]["digests"]
    assert drop(one, ("ids",)) == drop(two, ("ids",)), (one, two)
    fused, hooks = d["ext:a:9:12343:torch:fused"]["digests"], d["ext:a:9:12343:torch:hooks"]["digests"]
    assert drop(fused, ("ids", "dones")) == drop(hooks, ("ids", "dones")), (fused, hooks)


@pytest.mark.gpu
def test_hook_route_refuses_action_noise():
    """IsaacEnvBase.step stores the raw action: with action noise it would silently differ from the fused step."""
    from leibnizgym_b200.env import IsaacEnvBase, TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    from instantiation_digest import config
    N = 256
    seq = make_sequence(3, 3, N)
    env = TrifingerEnv(config(N, True, 9, "philox"), device="cuda:0", verbose=False,
                       sim=SyntheticSim(seq.to("cuda:0"), "cuda:0"))
    env.reset()
    with pytest.raises(ValueError, match="TrifingerEnv.step"):
        IsaacEnvBase.step(env, seq.action[1].cuda())
    env.step(seq.action[1].cuda())   # the fused step applies it
    quiet = TrifingerEnv(config(N, True, 9, "philox", action_noise=False), device="cuda:0", verbose=False,
                         sim=SyntheticSim(seq.to("cuda:0"), "cuda:0"))
    quiet.reset()
    IsaacEnvBase.step(quiet, seq.action[1].cuda())


# ======== d. DR observation noise and offsets next to a diverged env =====================================================
NEIGHBOUR_CASES = [(True, 28, 20, "noise"), (False, 16, 7, "noise"), (True, 28, 20, "offset"), (False, 16, 7, "offset"),
                   (True, 28, 20, "both"), (False, 16, 7, "both")]


@pytest.mark.gpu
@pytest.mark.parametrize("value", [2.0 ** 100, float("inf"), float("nan")], ids=["2^100", "inf", "nan"])
@pytest.mark.parametrize("asym, E, last, perturb", NEIGHBOUR_CASES,
                         ids=[f"{'a' if c[0] else 's'}-E{c[1]}" + ("" if c[3] == "noise" else f"-{c[3]}")
                              for c in NEIGHBOUR_CASES])
def test_noisy_neighbours_of_a_diverged_env_are_unchanged(value, asym, E, last, perturb):
    """A joint position of 2^100 / +inf / NaN in one env of a role lane (mid-lane in a full tile, and the last env of
    the ragged tile) sends that lane down the IEEE path.  The planted column carries DR white noise, a per-episode
    offset, or both.  Every other env's obs, clipped obs and bf16 obs stay bit for bit those of the run without the
    plant, noise and offset included; the planted element is torch's 2((v + b) - c) / span of its value v and its own
    offset b (the noise is below its ulp, or it is not finite), clamped like torch.clamp in the clipped copy."""
    from leibnizgym_b200.env import TrifingerEnv
    from leibnizgym_b200.sim import SyntheticSim
    from leibnizgym_b200.synthetic import make_sequence
    from leibnizgym_b200.wrappers import VecTaskPython
    from instantiation_digest import config
    N = _pick_n(9, E, last, "direct")
    assert N is not None and _tile_envs(N) == E
    EP = E // (2 if asym else 4)
    mid = 5 * E + EP + 3 if EP > 4 else 5 * E + EP + 1    # inside the second part of a full tile, neighbours both sides
    col = 4
    cfg = config(N, asym, 9, "philox", action_noise=False)
    cfg["reward_terms"].pop("keypoint")
    cfg["goal_movement"] = {"rotation": {"activate": False}}
    dr = cfg["domain_randomization"]
    dr["obs_noise_std"] = {"robot_q": 0.01 if perturb != "offset" else 0.0, "robot_u": 0.0, "object_q": 0.0,
                           "object_q_des": 0.0, "command": 0.0}
    dr["obs_bias_std"] = {"robot_q": 0.01} if perturb != "noise" else {}
    seq = make_sequence(91, 3, N)
    planted = copy.deepcopy(seq)
    for e in (mid, N - 1):
        planted.dof_state[1:, e, col, 0] = value
    outs, biases = [], []
    for sq in (seq, planted):
        env = TrifingerEnv(cfg, device="cuda:0", verbose=False, sim=SyntheticSim(sq.to("cuda:0"), "cuda:0"))
        vec = VecTaskPython(env, rl_device="cuda:0", clip_obs=5.0, clip_actions=1.0, obs_dtype=torch.bfloat16)
        vec.reset()
        steps = []
        for t in (1, 2):
            vec.step(seq.action[t].cuda())
            steps.append(tuple(x.clone() for x in (env.obs_buf, env._obs_clipped, env._obs_bf16.view(torch.int16))))
            biases.append(torch.zeros(2) if env.obs_bias is None else env.obs_bias[[mid, N - 1], col].cpu())
        outs.append(steps)
    assert (perturb == "noise") == all(float(b.abs().sum()) == 0 for b in biases)
    c0 = torch.tensor(env._P.scale_centre[col], dtype=torch.float32)
    span = torch.tensor(env._P.scale_span[col], dtype=torch.float32)
    for t, (clean, dirty) in enumerate(zip(*outs)):
        want = (2.0 * ((torch.full((2,), value) + biases[2 + t]) - c0)) / span
        for k, (a, b) in enumerate(zip(clean, dirty)):
            a, b = a.clone(), b.clone()
            got = _np(b[[mid, N - 1], col].float() if k < 2 else b[[mid, N - 1], col])
            if k < 2:
                exp = want if k == 0 else torch.clamp(want, -5.0, 5.0)
                assert rf_same(got, exp), (t, k, value, perturb, got, exp)
            a[[mid, N - 1], col] = 0
            b[[mid, N - 1], col] = 0
            bad = torch.nonzero(a != b)[:8].tolist()
            assert not bad, (t, ["obs", "obs_clipped", "obs_bf16"][k], value, perturb, (mid, N), bad,
                             [(float(a[i, j]), float(b[i, j])) for i, j in bad])
