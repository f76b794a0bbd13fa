"""Per-episode domain-randomisation offsets (extension, "domain_randomization": obs_bias_std / action_bias_std) without
a GPU: the config defaults and errors, the parameter block (unchanged for configs without the keys), the pointer rules
of the C ABI and the ctypes layout."""
import copy
import ctypes as C

import pytest

from leibnizgym_b200 import _native as nat
from leibnizgym_b200.config import default_trifinger_config, difficulty_config, resolve_config
from leibnizgym_b200.params import build_params, dr_bias_sigmas

GROUPS = {"robot_q": (0, 9), "robot_u": (9, 18), "object_q": (18, 25), "object_q_des": (25, 32)}
NEW_FIELDS = ("dr_bias_sigma", "dr_bias_mask", "dr_action_bias_sigma", "_pad_tail3")


def _dr(**keys):
    cfg = difficulty_config(3, 64, seed=5)
    cfg["domain_randomization"] = dict({"activate": True}, **keys)
    return resolve_config(cfg)


def test_config_defaults_are_zero():
    dr = default_trifinger_config()["domain_randomization"]
    assert dr["obs_bias_std"] == {"robot_q": 0.0, "robot_u": 0.0, "object_q": 0.0, "object_q_des": 0.0, "command": 0.0}
    assert dr["action_bias_std"] == 0.0
    groups, act = dr_bias_sigmas(resolve_config({"command_mode": "torque"}))
    assert set(groups.values()) == {0.0} and act == 0.0


def test_keys_are_read_only_when_activated():
    cfg = _dr(obs_bias_std={"object_q": 0.01}, action_bias_std=0.02)
    cfg["domain_randomization"]["activate"] = False
    groups, act = dr_bias_sigmas(cfg)
    assert set(groups.values()) == {0.0} and act == 0.0
    p = build_params(cfg, 64)
    assert p.dr_bias_mask == 0 and p.dr_action_bias_sigma == 0.0 and set(p.dr_bias_sigma) == {0.0}


@pytest.mark.parametrize("bad", [-0.1, float("nan"), float("inf"), "x"])
def test_bad_obs_sigma_names_the_key(bad):
    with pytest.raises(ValueError, match=r"domain_randomization\.obs_bias_std\.robot_u"):
        dr_bias_sigmas(_dr(obs_bias_std={"robot_u": bad}))


@pytest.mark.parametrize("bad", [-1.0, float("nan"), float("-inf"), None])
def test_bad_action_sigma_names_the_key(bad):
    with pytest.raises(ValueError, match=r"domain_randomization\.action_bias_std"):
        dr_bias_sigmas(_dr(action_bias_std=bad))


def test_unknown_group_names_the_key():
    with pytest.raises(ValueError, match=r"domain_randomization\.obs_bias_std.*'object_pose'"):
        dr_bias_sigmas(_dr(obs_bias_std={"object_pose": 0.01}))


def test_errors_are_raised_at_construction_before_any_device_work():
    from leibnizgym_b200.env import TrifingerEnv
    cfg = difficulty_config(3, 64)
    cfg["domain_randomization"] = {"activate": True, "action_bias_std": -1.0}
    with pytest.raises(ValueError, match="action_bias_std"):
        TrifingerEnv(cfg, device="cpu", verbose=False)


def _fields(p):
    out = {}
    for name, _ in nat.LgParams._fields_:
        v = getattr(p, name)
        if name == "terms":
            v = [tuple(getattr(t, f) for f, _ in nat.LgRewardTerm._fields_) for t in v]
        elif hasattr(v, "__len__"):
            v = list(v)
        out[name] = v
    return out


@pytest.mark.parametrize("mode", ["torque", "position", "position_impedance"])
@pytest.mark.parametrize("noise", [False, True])
def test_params_without_the_keys_are_unchanged(mode, noise):
    """A config without the new keys, and one with them at 0, fill every field exactly as before the feature (the
    fields other than the new ones do not read the keys at all); the new fields are zero."""
    base = difficulty_config(3, 256, seed=11, command_mode=mode)
    if noise:
        base["domain_randomization"] = {"activate": True, "action_noise_std": 0.02,
                                        "obs_noise_std": {"robot_q": 0.005, "object_q": 0.002}}
    zeros = copy.deepcopy(base)
    zeros.setdefault("domain_randomization", {"activate": noise})
    zeros["domain_randomization"]["obs_bias_std"] = {g: 0.0 for g in GROUPS}
    zeros["domain_randomization"]["action_bias_std"] = 0.0
    with_keys = copy.deepcopy(base)
    with_keys.setdefault("domain_randomization", {"activate": noise})
    with_keys["domain_randomization"]["obs_bias_std"] = {"object_q": 0.01, "command": 0.1}
    with_keys["domain_randomization"]["action_bias_std"] = 0.05
    a = _fields(build_params(resolve_config(base), 256))
    b = _fields(build_params(resolve_config(zeros), 256))
    c = _fields(build_params(resolve_config(with_keys), 256))
    assert a == b
    for name in NEW_FIELDS:
        assert a[name] in (0, 0.0) or set(a[name]) == {0.0}, name
    for name in a:
        if name not in NEW_FIELDS:
            assert a[name] == c[name], name


def test_params_columns_and_mask():
    A = 9
    cfg = _dr(obs_bias_std={"object_q": 0.01, "command": 0.1, "robot_u": 0.0}, action_bias_std=0.05)
    p = build_params(cfg, 64)
    want = [0.0] * 64
    for c in range(18, 25):
        want[c] = 0.01
    for c in range(32, 32 + A):
        want[c] = 0.1
    got = list(p.dr_bias_sigma)
    assert got == [float(C.c_float(x).value) for x in want]
    assert p.dr_bias_mask == sum(1 << c for c in range(64) if want[c] != 0.0)
    assert p.dr_action_bias_sigma == pytest.approx(0.05)


def test_ctypes_layout():
    names = [f[0] for f in nat.LgBuffers._fields_]
    assert names[-3:] == ["obs_bias", "action_bias", "torch_rng"]
    pnames = [f[0] for f in nat.LgParams._fields_]
    assert pnames[-len(NEW_FIELDS):] == list(NEW_FIELDS)
    assert nat.LgParams.seed.offset + 8 + 8 <= 160   # the hot block is untouched
    lib = nat.load()
    assert lib.lg_struct_size(0) == C.sizeof(nat.LgParams)
    assert lib.lg_struct_size(2) == C.sizeof(nat.LgBuffers)


def _abi_args():
    p, s, b = nat.LgParams(), nat.LgSimState(), nat.LgBuffers()
    p.num_envs, p.action_dim, p.dr_activate = 64, 9, 1
    s.dof_state, s.root_state, s.rigid_body = 0x10000, 0x20000, 0x30000
    for i, name in enumerate(("obs", "action", "reward", "reset", "goal_reset", "successes", "steps_count", "goal_pose",
                              "goal_movement", "history", "control")):
        setattr(b, name, 0x100000 * (i + 1))
    return p, s, b


def _refused(lib, p, s, b, text):
    """Every entry point validates before any CUDA call: lg_reset_envs with an empty list returns right after it."""
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == -1
    assert text in lib.lg_last_error()
    assert lib.lg_post_physics(p, s, b, 0.0, None) == -1
    assert lib.lg_pre_physics(p, s, b, 0x5000000, None) == -1
    assert lib.lg_fill_observations(p, s, b, None) == -1
    assert lib.lg_pre_step(p, s, b, None) == -1


def test_obs_sigma_needs_obs_bias_through_the_abi():
    lib = nat.load()
    p, s, b = _abi_args()
    p.dr_bias_sigma[20] = 0.01
    p.dr_bias_mask = 1 << 20
    _refused(lib, p, s, b, b"needs LgBuffers.obs_bias")
    b.obs_bias = 0x9000000
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0


def test_action_sigma_needs_action_bias_through_the_abi():
    lib = nat.load()
    p, s, b = _abi_args()
    p.dr_action_bias_sigma = 0.05
    _refused(lib, p, s, b, b"needs LgBuffers.action_bias")
    b.action_bias = 0x9000000
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0


def test_mask_and_sigmas_must_agree_through_the_abi():
    lib = nat.load()
    p, s, b = _abi_args()
    b.obs_bias, b.action_bias = 0x9000000, 0xa000000
    p.dr_bias_sigma[3] = 0.01                     # sigma without its mask bit
    _refused(lib, p, s, b, b"dr_bias_mask must mark exactly")
    p.dr_bias_mask = 1 << 3
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0
    p.dr_bias_mask |= 1 << 4                      # a mask bit without its sigma
    _refused(lib, p, s, b, b"dr_bias_mask must mark exactly")
    p.dr_bias_mask = 1 << 3
    p.dr_bias_sigma[3] = -0.01
    _refused(lib, p, s, b, b"dr_bias_sigma: finite")
    p.dr_bias_sigma[3] = 0.0
    p.dr_bias_mask = 0
    p.dr_bias_sigma[41] = 0.01                    # beyond obs_dim = 41
    p.dr_bias_mask = 1 << 41
    _refused(lib, p, s, b, b"dr_bias_sigma: finite")
    p.dr_bias_sigma[41] = 0.0
    p.dr_bias_mask = 0
    p.dr_action_bias_sigma = float("nan")
    _refused(lib, p, s, b, b"dr_action_bias_sigma must be finite")


def test_offsets_need_dr_activate_through_the_abi():
    lib = nat.load()
    p, s, b = _abi_args()
    b.obs_bias, b.action_bias = 0x9000000, 0xa000000
    p.dr_activate = 0
    p.dr_action_bias_sigma = 0.05
    _refused(lib, p, s, b, b"need dr_activate")
    p.dr_action_bias_sigma = 0.0
    p.dr_bias_sigma[20] = 0.01
    p.dr_bias_mask = 1 << 20
    _refused(lib, p, s, b, b"need dr_activate")
    p.dr_activate = 1
    assert lib.lg_reset_envs(p, s, b, None, 0, None) == 0
