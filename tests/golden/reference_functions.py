"""Stored outputs of the reference's building blocks for tests/test_oracle_vs_reference_live.py: its primitives, its six
reward terms and its samplers, on random and adversarial inputs — a wider net than the whole-step scenarios (inf,
3.4e38, denormals, identical / antipodal / non-unit / zero quaternions, distances at the lgsk knee, env-step counts on,
inside and outside random schedule windows, and the samplers' use of torch's generator).

The inputs are pure functions of fixed seeds and are rebuilt by the test; only the outputs are stored, in
functions/reference_functions.npz.

    LEIBNIZ_REFERENCE_ROOT=<checkout of pairlab/leibnizgym> python tests/golden/reference_functions.py
        calls the reference's own functions (the reward terms through TorchScript, as the reference runs them), checks
        that the oracle reproduces every output bit for bit, and records the reference's outputs;
    python tests/golden/reference_functions.py --oracle
        records the oracle's outputs instead.

The committed file was recorded with --oracle: the reference's source was not at hand when the suite was made
self-contained.  The oracle's arithmetic is unchanged since commit ebe2532, whose live comparison of these functions
against the reference (the same checks at larger N) found them bit-identical.  Recording from the reference replaces it
with the reference's own outputs.
"""
from __future__ import annotations

import importlib.util
import math
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
PATH = os.path.join(HERE, "functions", "reference_functions.npz")   # not a whole-step scenario: kept out of *.npz

N_PRIMITIVES = 512      # rows 0..300 are hand-placed edge cases
N_REWARD = 256          # rows 0..96 are hand-placed edge cases
K_SAMPLES = 1000
REWARD_SEEDS = (0, 1, 2)
DT = 0.02


def load_reference(root: str) -> types.SimpleNamespace:
    """The reference's pure modules, imported from where they lie (nothing is copied)."""
    tc = types.ModuleType("termcolor")
    tc.colored = lambda s, *a, **k: s
    sys.modules.setdefault("termcolor", tc)

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(root, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    pkg = types.ModuleType("leibnizgym"); pkg.__path__ = []          # noqa: E702
    utils = types.ModuleType("leibnizgym.utils"); utils.__path__ = []  # noqa: E702
    sys.modules["leibnizgym"], sys.modules["leibnizgym.utils"] = pkg, utils
    tu = load("leibnizgym.utils.torch_utils", "leibnizgym/utils/torch_utils.py")
    load("leibnizgym.utils.mdp", "leibnizgym/utils/mdp.py")
    rw = load("_ref_rewards", "leibnizgym/envs/trifinger/rewards.py")
    sm = load("_ref_sample", "leibnizgym/envs/trifinger/sample.py")
    return types.SimpleNamespace(tu=tu, rw=rw, sm=sm)


# ---- inputs ------------------------------------------------------------------------------------------------------
def _quats(g, n, unit=True):
    q = torch.randn(n, 4, generator=g)
    return q / q.norm(dim=1, keepdim=True) if unit else q


def _poses(g, n):
    p = torch.zeros(n, 13)
    p[:, 0:3] = torch.rand(n, 3, generator=g) * 0.6 - 0.3
    p[:, 3:7] = _quats(g, n)
    p[:, 7:13] = torch.randn(n, 6, generator=g) * 0.1
    return p


def primitive_inputs():
    g = torch.Generator().manual_seed(1)
    N = N_PRIMITIVES
    x = torch.randn(N, 9, generator=g) * 3
    x[:5] = torch.tensor([0.0, -0.0, 1e-42, 3.4e38, -3.4e38, float("inf"), 1.0, -1.0, 0.5])[None]
    lo, hi = -torch.rand(9, generator=g) - 0.1, torch.rand(9, generator=g) + 0.1
    a, b = _quats(g, N), _quats(g, N)
    b[:100] = a[:100]                     # identical
    b[100:200] = -a[100:200]              # antipodal
    a[200:300] = _quats(g, 100, unit=False) * 3   # non-unit: |v| > 1 -> clamp
    a[300] = 0.0                           # zero quaternion
    r, p, y = (torch.rand(N, generator=g) * 2 * math.pi for _ in range(3))
    d = torch.cat([torch.rand(N, generator=g) * 2.5, torch.tensor([0.0, 1.78, 1.8, 5.0, 1e-30])])
    return types.SimpleNamespace(x=x, lo=lo, hi=hi, a=a, b=b, r=r, p=p, y=y, d=d)


def reward_inputs(seed):
    """Poses, a random reward-term config and the env-step counts on, inside and outside its schedule windows."""
    g = torch.Generator().manual_seed(100 + seed)
    rs = np.random.RandomState(seed)
    N = N_REWARD
    obj, obj_prev, goal = _poses(g, N), _poses(g, N), _poses(g, N)[:, :7].contiguous()
    tips = torch.stack([_poses(g, N) for _ in range(3)], dim=1)
    tips_prev = torch.stack([_poses(g, N) for _ in range(3)], dim=1)
    obj[:64, 0:7] = goal[:64]                                  # on the goal: d = 0, theta = 0
    tips[64:96, :, 0:3] = obj[64:96, None, 0:3]                # fingertips in the cube centre
    start, end = float(rs.randint(0, 1000)), float(rs.randint(1000, 5000))
    cfg = {
        "finger_reach_object_rate": {"activate": True, "weight": float(-rs.randint(1, 900)), "norm_p": 2,
                                     "thresh_sched_start": start, "thresh_sched_end": end},
        "finger_move_penalty": {"activate": True, "weight": -float(rs.rand())},
        "object_dist": {"activate": True, "weight": float(rs.randint(1, 3000)),
                        "thresh_sched_start": start, "thresh_sched_end": end},
        "object_rot": {"activate": True, "weight": float(rs.randint(1, 3000)), "scale": float(1 + 4 * rs.rand()),
                       "epsilon": 0.01, "thresh_sched_start": start, "thresh_sched_end": end},
        "object_rot_delta": {"activate": True, "weight": float(-rs.randint(1, 500)),
                             "linear_schedule_start": start, "linear_schedule_end": end},
        "object_move": {"activate": True, "weight": float(-rs.randint(1, 900))},
    }
    steps = (0.0, start, start + 1.0, 0.5 * (start + end), end, end + 1.0, 1e9)
    return types.SimpleNamespace(obj=obj, obj_prev=obj_prev, goal=goal, tips=tips, tips_prev=tips_prev, cfg=cfg,
                                 steps=steps)


# ---- outputs: name -> tensor, the same names from the oracle and from the reference -------------------------------
def primitives(ref=None):
    import oracle.trifinger_oracle as o
    i = primitive_inputs()
    tu = ref.tu if ref is not None else o
    out = {"scale_transform": tu.scale_transform(i.x, i.lo, i.hi),
           "unscale_transform": tu.unscale_transform(i.x, i.lo, i.hi),
           "saturate": tu.saturate(i.x, i.lo, i.hi),
           "quat_mul": tu.quat_mul(i.a, i.b), "quat_conjugate": tu.quat_conjugate(i.a),
           "quat_diff_rad": tu.quat_diff_rad(i.a, i.b)}
    euler = ref.tu.quaternion_from_euler_xyz if ref is not None else o.quat_from_euler_xyz
    out["quat_from_euler_xyz"] = euler(i.r, i.p, i.y)
    lgsk = ref.rw.lgsk_kernel if ref is not None else o.lgsk
    for scale in (50.0, 30.0, 3.0):
        out[f"lgsk_{scale:g}"] = lgsk(i.d, scale)
    return out


def reward_terms(seed, ref=None):
    """The six reward terms at every env-step count of reward_inputs(seed): `term/T<index>`."""
    i = reward_inputs(seed)
    out = {}
    if ref is not None:
        rw = ref.rw
        classes = {"finger_reach_object_rate": rw.FingerReachObjectRatePenalty,
                   "finger_move_penalty": rw.FingertipMovementPenalty, "object_dist": rw.ObjectDistanceReward,
                   "object_rot": rw.ObjectRotationReward, "object_rot_delta": rw.ObjectRotationDeltaReward,
                   "object_move": rw.ObjectMoveReward}
        m = {k: torch.jit.script(classes[k](name=k, **dict(v))) for k, v in i.cfg.items()}
        for n, T in enumerate(i.steps):
            out[f"finger_reach_object_rate/T{n}"] = m["finger_reach_object_rate"].compute(T, i.tips, i.tips_prev, i.obj,
                                                                                           i.obj_prev)
            out[f"finger_move_penalty/T{n}"] = m["finger_move_penalty"].compute(DT, i.tips, i.tips_prev)
            out[f"object_dist/T{n}"] = m["object_dist"].compute(DT, T, i.obj, i.goal)
            out[f"object_rot/T{n}"] = m["object_rot"].compute(DT, T, i.obj, i.goal)
            out[f"object_rot_delta/T{n}"] = m["object_rot_delta"].compute(DT, T, i.obj, i.obj_prev, i.goal)
            out[f"object_move/T{n}"] = m["object_move"].compute(i.obj, i.obj_prev, i.goal)
        return out
    import oracle.trifinger_oracle as o
    P = o.reward_term_params(i.cfg)
    for n, T in enumerate(i.steps):
        out[f"finger_reach_object_rate/T{n}"] = o.finger_reach_object_rate(P["finger_reach_object_rate"], T, i.tips,
                                                                           i.tips_prev, i.obj, i.obj_prev)
        out[f"finger_move_penalty/T{n}"] = o.finger_move_penalty(P["finger_move_penalty"], DT, i.tips, i.tips_prev)
        out[f"object_dist/T{n}"] = o.object_dist(P["object_dist"], DT, T, i.obj, i.goal)
        out[f"object_rot/T{n}"] = o.object_rot(P["object_rot"], DT, T, i.obj, i.goal)
        out[f"object_rot_delta/T{n}"] = o.object_rot_delta(P["object_rot_delta"], DT, T, i.obj, i.obj_prev, i.goal)
        out[f"object_move/T{n}"] = o.object_move(P["object_move"], i.obj, i.obj_prev, i.goal)
    return out


def samplers(ref=None):
    """Same seed, same call order: what the samplers draw from torch's global generator (CPU)."""
    k = K_SAMPLES
    torch.manual_seed(123)
    if ref is not None:
        sm = ref.sm
        x, y = sm.random_xy(k, 0.15, "cpu")
        return {"random_xy_x": x, "random_xy_y": y, "random_z": sm.random_z(k, 0.03, 0.2, "cpu"),
                "random_orientation": sm.random_orientation(k, "cpu"),
                "random_angular_vel": sm.random_angular_vel(k, "cpu", 0.5),
                "random_yaw_orientation": sm.random_yaw_orientation(k, "cpu")}
    import oracle.trifinger_oracle as o
    d = o.Draws()                        # draws from torch's global generator, in the reference's order
    x, y = o.random_xy(d, k, 0.15, (0, 1))
    return {"random_xy_x": x, "random_xy_y": y, "random_z": o.random_z(d, k, 0.03, 0.2, 2),
            "random_orientation": o.random_orientation(d, k), "random_angular_vel": o.random_angular_vel(d, k, 0.5),
            "random_yaw_orientation": o.random_yaw_orientation(d, k, 3)}


def groups(ref=None):
    """Every stored array, keyed `<group>/<name>`; the groups are the units the tests check."""
    out = {f"primitives/{k}": v for k, v in primitives(ref).items()}
    for seed in REWARD_SEEDS:
        out.update({f"reward{seed}/{k}": v for k, v in reward_terms(seed, ref).items()})
    out.update({f"samplers/{k}": v for k, v in samplers(ref).items()})
    return out


def same(a, b) -> bool:
    """Bit-level agreement as the comparison has always counted it: equal values (0.0 == -0.0), NaN where NaN."""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def main(argv):
    if "--oracle" in argv:
        arrays = groups()
    else:
        root = os.environ.get("LEIBNIZ_REFERENCE_ROOT")
        if not root or not os.path.isdir(os.path.join(root, "leibnizgym")):
            raise SystemExit("set LEIBNIZ_REFERENCE_ROOT to a checkout of pairlab/leibnizgym (or pass --oracle)")
        arrays = groups(load_reference(root))
        mine = groups()
        bad = [k for k in arrays if not same(mine[k].detach().numpy(), arrays[k].detach().numpy())]
        if bad:
            raise SystemExit(f"the oracle differs from the reference in {len(bad)} arrays, e.g. {bad[:5]}; nothing written")
    np.savez_compressed(PATH, **{k: v.detach().numpy() for k, v in arrays.items()})
    print(f"{PATH}: {len(arrays)} arrays, {os.path.getsize(PATH)} bytes")


if __name__ == "__main__":
    main(sys.argv[1:])
