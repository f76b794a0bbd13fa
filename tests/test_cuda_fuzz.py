"""Random whole-env configurations (the generator of tests/golden/fuzz_reference.py) through the CUDA path in lockstep
with the oracle (tests/lockstep.py: every output, every step).

  a. the 12 original configurations at a few hundred envs, no extensions;
  b. a fixed covering design of configuration x launcher geometry x extension (DESIGN below): each row takes its
     configuration from random_scenario, a (tile size, pre-physics regime) pair the launcher picks, an env count with a
     ragged last tile, and a set of extensions; it asserts that the instantiations it names ran.
A failure prints the case as JSON (configuration, N, E, regime, flags, step).
"""
import json
import os
import random
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from fuzz_reference import random_scenario  # noqa: E402

FLAGS = ("clip", "bf16", "kp", "goal", "stats", "terms", "obs", "act")
REGIMES = ("small", "direct", "minb4", "ticket")
# sigma of the per-episode offsets: per observation group (raw units; "command" in action units), and of the action
OBS_BIAS = {"robot_q": 0.02, "robot_u": 0.1, "object_q": 0.005, "object_q_des": 0.003, "command": 0.03}
ACTION_BIAS = 0.05
# (k, command_mode, asymmetric_obs, E, pre-physics regime, last-tile kind, extensions, obs offset groups): the
# configuration is random_scenario(random.Random(2000 + k), 12 + k) with command_mode and asymmetric_obs overridden.
# Extensions: clip = VecTaskPython's fused clamps, bf16 = bf16 copies, kp = keypoint term, goal = the moving goal
# integrated on both sides (rows whose configuration has the moving goal), stats = episode statistics, terms = per-term
# episode returns, obs / act = per-episode DR offsets.  The minb4 and ticket rows run tens of thousands of envs.
DESIGN = [
    (71, "torque", True, 16, "small", "1", "clip bf16 kp goal stats terms", ""),
    (163, "position", True, 16, "small", "EP-1", "clip kp stats terms act", ""),
    (13, "position", True, 16, "small", "EP", "clip bf16 kp stats obs act", "robot_u object_q object_q_des command"),
    (42, "torque", True, 16, "direct", "EP+1", "clip kp goal stats terms", ""),
    (20, "torque", False, 16, "direct", "E-1", "clip bf16 goal stats", ""),
    (189, "torque", False, 16, "direct", "1", "clip kp stats", ""),
    (112, "position", True, 24, "direct", "EP-1", "clip kp goal obs act", "robot_u"),
    (72, "torque", False, 24, "direct", "EP", "clip kp goal stats terms", ""),
    (116, "position", False, 24, "direct", "EP+1", "clip bf16 goal stats terms obs act", "robot_u object_q_des command"),
    (126, "position", True, 28, "direct", "E-1", "clip bf16 kp stats terms obs act", "robot_u object_q object_q_des command"),
    (68, "position", True, 28, "direct", "1", "bf16 kp stats terms obs act", "robot_q robot_u object_q_des"),
    (157, "position", True, 28, "direct", "EP-1", "clip bf16 kp stats obs", "robot_u command"),
    (175, "position", True, 28, "small", "EP", "bf16 kp goal", ""),
    (160, "position", False, 28, "small", "EP+1", "bf16 goal stats terms act", ""),
    (50, "position", False, 32, "small", "E-1", "goal stats obs act", "robot_q object_q"),
    (181, "torque", False, 32, "small", "1", "clip bf16 goal stats obs", "robot_u"),
    (179, "position", True, 32, "small", "EP-1", "kp act", ""),
    (59, "position", False, 32, "minb4", "EP", "clip kp obs", "command"),
    (8, "torque", False, 32, "ticket", "EP+1", "clip bf16 stats terms act", ""),
    (33, "position_impedance", True, 32, "small", "E-1", "stats terms", ""),
    (196, "position_impedance", True, 32, "small", "1", "kp stats terms", ""),
    (176, "position_impedance", False, 32, "small", "EP-1", "kp stats terms obs", "object_q object_q_des"),
    (161, "position_impedance", True, 32, "small", "EP", "clip bf16 stats terms obs", "robot_u object_q object_q_des"),
    (30, "position_impedance", False, 32, "direct", "EP+1", "clip kp stats terms obs act", "command"),
    (12, "position_impedance", True, 32, "direct", "E-1", "clip bf16 kp stats terms obs", "robot_q"),
    (177, "position_impedance", True, 32, "direct", "1", "bf16 kp goal act", ""),
    (106, "position_impedance", False, 32, "direct", "EP-1", "clip bf16 goal obs", "robot_u object_q object_q_des"),
    (180, "position_impedance", False, 32, "minb4", "EP", "bf16 goal stats terms act", ""),
    (17, "position_impedance", False, 32, "ticket", "EP+1", "kp goal obs", "robot_q object_q command"),
]


def design_case(row):
    """The configuration, StateSequence parameters and flags of one DESIGN row (no GPU needed)."""
    k, mode, asym, E, regime, kind, flags, groups = row
    sc = random_scenario(random.Random(2000 + k), 12 + k)
    cfg = json.loads(json.dumps(sc["config"]))
    cfg["command_mode"], cfg["asymmetric_obs"] = mode, asym
    flags = set(flags.split())
    return {"k": k, "scenario": sc, "config": cfg, "A": 18 if mode == "position_impedance" else 9, "asym": asym,
            "E": E, "regime": regime, "kind": kind, "flags": flags,
            "obs_bias": {g: OBS_BIAS[g] for g in groups.split()} if "obs" in flags else {}}


def _scale_schedules(cfg, factor):
    """Schedule windows count env-steps (frame x N): stretched by N / sc["N"] they still open and close within T."""
    for term in cfg["reward_terms"].values():
        for key in ("thresh_sched_start", "thresh_sched_end", "linear_schedule_start", "linear_schedule_end"):
            if key in term:
                term[key] *= factor


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(12))
def test_random_configuration_matches_oracle(idx):
    """The original configurations: a few hundred envs (several tiles, ragged), no extensions."""
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence, plant_goal_rows
    from lockstep import Lockstep
    sc = random_scenario(random.Random(1000 + idx), idx)
    N, T, cfg = sc["N"] * 37, sc["T"], dict(sc["config"])
    cfg["num_instances"] = N
    seq = make_sequence(sc["seed"], T, N, action_dim=sc.get("action_dim", 9))
    if sc.get("plant_goal_rows"):
        plant_goal_rows(seq, sc["seed"])
    run = Lockstep(cfg, seq, bernoulli_masks(sc["seed"], T, N, sc["reset_p"]),
                   bernoulli_masks(sc["seed"] + 1, T, N, sc["goal_reset_p"]), idx)
    run.run(T, json.dumps({"idx": idx, "config": cfg, "N": N}))


@pytest.mark.gpu
@pytest.mark.parametrize("row", DESIGN, ids=[f"k{r[0]}-A{18 if r[1] == 'position_impedance' else 9}-{'a' if r[2] else 's'}"
                                              f"-E{r[3]}-{r[4]}" for r in DESIGN])
def test_design_case_matches_oracle(row):
    """One DESIGN row: its instantiations (asserted from torch.profiler) against the oracle, every output every step."""
    from leibnizgym_b200.synthetic import bernoulli_masks, make_sequence, plant_goal_rows
    from instantiation_digest import launched
    from lockstep import Lockstep
    from test_cuda_edges import _tile_envs
    from test_cuda_instantiations import PRE, _expect, _nvalid, _pick_n
    c = design_case(row)
    sc, cfg, A, E, regime, flags = c["scenario"], c["config"], c["A"], c["E"], c["regime"], c["flags"]
    N = _pick_n(A, E, _nvalid(c["kind"], E, c["asym"]), regime)
    if N is None:
        pytest.skip(f"no env count gives tile size {E} with the {regime} pre-physics grid on this device")
    assert A == 18 or _tile_envs(N) == E
    T = sc["T"]
    cfg["num_instances"] = N
    _scale_schedules(cfg, N // sc["N"])
    where = json.dumps({"row": list(row), "config": cfg, "N": N, "E": E, "regime": regime, "flags": sorted(flags),
                        "obs_bias": c["obs_bias"]})
    seq = make_sequence(sc["seed"], T, N, action_dim=A)
    if sc.get("plant_goal_rows"):
        plant_goal_rows(seq, sc["seed"])
    run = Lockstep(cfg, seq, bernoulli_masks(sc["seed"], T, N, sc["reset_p"]),
                   bernoulli_masks(sc["seed"] + 1, T, N, sc["goal_reset_p"]), c["k"],
                   clip="clip" in flags, bf16="bf16" in flags, keypoint="kp" in flags, goal_integration="goal" in flags,
                   episode_statistics="stats" in flags or "terms" in flags, episode_term_returns="terms" in flags,
                   obs_bias=c["obs_bias"], action_bias=ACTION_BIAS if "act" in flags else 0.0)
    got = launched(run.reset)
    step = {}
    got1 = launched(lambda: step.update(r=run.step(1)))
    ext = bool(flags & {"bf16", "kp", "stats", "terms", "obs", "act"}) or cfg["goal_movement"]["rotation"]["activate"]
    post = {(A, int(c["asym"]), r, int("clip" in flags), E, int(ext)) for r in (0, 1)}
    _expect({k: got[k] | got1[k] for k in got}, post=post, pre={(A, *PRE[regime], 0)}, where=where)
    run.check(1, *step["r"], where)
    for t in range(2, T):
        run.check(t, *run.step(t), where)


def test_design_covers_every_extension_geometry_and_configuration():
    """The covering properties of DESIGN (CPU only)."""
    cases = [design_case(r) for r in DESIGN]
    for c in cases:
        assert c["A"] == 18 and c["E"] == 32 or c["A"] == 9 and (c["E"], c["regime"]) in {
            (16, "small"), (16, "direct"), (24, "direct"), (28, "direct"), (28, "small"), (32, "small"), (32, "minb4"),
            (32, "ticket")}, c["k"]
        assert "terms" not in c["flags"] or "stats" in c["flags"], c["k"]
        assert "goal" not in c["flags"] or c["config"]["goal_movement"]["rotation"]["activate"], c["k"]
        assert ("obs" in c["flags"]) == bool(c["obs_bias"]), c["k"]
    assert len({c["k"] for c in cases}) == len(cases)
    # every extension on and off with each action width, each obs mode and each pre-physics regime
    for f in FLAGS:
        for key, values in (("A", (9, 18)), ("asym", (True, False)), ("regime", REGIMES)):
            for v in values:
                on = [f in c["flags"] for c in cases if c[key] == v]
                assert any(on) and not all(on), (f, key, v)
    # every tile size with obs offsets, action offsets and per-term returns
    for E in (16, 24, 28, 32):
        for f in ("obs", "act", "terms"):
            assert any(c["E"] == E and f in c["flags"] for c in cases), (E, f)
    offsets = [c for c in cases if c["flags"] & {"obs", "act"}]
    assert any(not c["config"]["normalize_obs"] for c in offsets)
    assert any(c["config"]["command_mode"] == "position" for c in offsets)
    assert any({"kp", "goal"} <= c["flags"] for c in offsets)
    # the command-group offsets of the 50-column rows
    assert any(c["A"] == 18 and "command" in c["obs_bias"] for c in cases)
    # tens of thousands of envs through the CPU oracle: few
    assert sum(c["regime"] in ("minb4", "ticket") for c in cases) <= 4
