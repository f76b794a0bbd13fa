"""Parity tolerances (BASELINE.json north_star): masks / ids / counters bit-exact;
rewards, observations and states within 1e-5 relative for fp32.

A small absolute floor is needed next to the relative bound because several quantities are
differences of nearly equal numbers (norm - previous norm, |theta| - |previous theta|) whose
value can be arbitrarily close to zero while each operand carries a 1-ulp sampling error
(sin/cos/exp/asin differ by <= 2 ulp between CUDA libdevice and torch's SLEEF).  The floor
is stated per key, relative to the natural magnitude of the quantity."""
import numpy as np

RTOL = 1e-5

EXACT = {"reset_in", "goal_reset_in", "reset_ids", "goal_reset_ids", "dof_index_list", "root_index_list0",
         "root_index_list1", "root_index_list_move", "reset_buf", "goal_reset_buf", "steps_count", "successes", "sched_step"}

# Absolute floors.  Each is at most 4x the largest error OBSERVED beyond the relative bound on the B200 over the three
# BASELINE-size scenarios (tests/test_cuda_round2.py::test_observed_parity_errors_are_recorded re-measures them on every
# GPU run, asserts exactly that, and leaves the numbers in gpurun_out/observed_parity_errors.json; round 2:
# obs / states 8.9e-8 absolute and 3.3e-7 relative, i.e. nothing beyond the relative bound; torques and reset joint
# rows bit-identical; goal poses 2.2e-8; terms 4.3e-5 and reward 3.6e-5 beyond the relative bound).
# Where the term floor comes from: finger_reach_object_rate is weight x sum of six DIFFERENCES of 2-norms of ~0.1-0.6 m
# (rewards.py:219-235), near zero while each norm carries up to one ulp (2^-24 x 0.5 m = 3e-8) of legitimate
# evaluation-order difference: |weight| 750 x 2 ulps = 4.5e-5 is what is seen, 3 ulps (1.35e-4) what is allowed.
ATOL = {
    "obs": 1e-6, "states": 1e-6, "action_buf": 0.0, "applied_torque": 1e-7,
    "goal_pose": 1e-7, "goal_movement": 1e-7,
    "pre_sim_dof": 1e-7, "pre_sim_obj_root": 1e-7, "pre_sim_goal_root": 1e-7,
    "terms": 1.35e-4, "reward": 1.35e-4,
}


def angle_slack(q_a, q_b):
    """Per-env allowance (radians) for theta = 2 asin(min(|v|, 1)) (utils/torch_utils.py:145-150).
    d(theta)/d|v| = 2 / sqrt(1 - |v|^2) is unbounded as theta -> pi: one ulp of |v| (which a different
    but equally valid fp32 evaluation order of the 2-norm, or of the sampled goal quaternion's
    normalisation, legitimately produces) moves theta by up to ~7e-4 rad there.  The allowance is
    2 ulp of |v| through that slope; it is ~5e-7 rad for well-conditioned pairs."""
    import torch
    from oracle.trifinger_oracle import quat_conjugate, quat_mul
    v = quat_mul(torch.as_tensor(q_a), quat_conjugate(torch.as_tensor(q_b)))[:, :3].double().norm(dim=-1).clamp(max=1.0)
    eps = 2.0 ** -23
    return (2.0 * 2.0 * eps / torch.sqrt(torch.clamp(1.0 - v * v, min=2.0 * eps))).numpy()


def compare(key, got, expected, extra_atol=None):
    """Returns (ok, detail).  `extra_atol` (broadcastable) adds a data-dependent absolute allowance."""
    got, expected = np.asarray(got), np.asarray(expected)
    if got.shape != expected.shape:
        return False, f"shape {got.shape} != {expected.shape}"
    if key in EXACT:
        ok = np.array_equal(got.astype(np.int64), expected.astype(np.int64))
        return ok, "" if ok else f"{int((got.astype(np.int64) != expected.astype(np.int64)).sum())} entries differ"
    g, x = got.astype(np.float64), expected.astype(np.float64)
    with np.errstate(invalid="ignore"):
        err = np.abs(g - x)   # inf - inf is NaN
    bound = ATOL[key] + RTOL * np.abs(x)
    if extra_atol is not None:
        bound = bound + np.asarray(extra_atol, dtype=np.float64)
    # The relative bound applies to finite expectations only (RTOL * inf would accept anything).  Equal values agree
    # (an infinity equals itself; -0.0 == +0.0, which the fast division's -0 -> +0 needs) and NaN agrees with NaN.
    close = np.isfinite(x) & (err <= bound)
    bad = ~(close | (g == x) | (np.isnan(g) & np.isnan(x)))
    if bad.any():
        i = np.unravel_index(np.argmax(np.where(bad, np.nan_to_num(err, nan=np.inf), -1.0)), err.shape)
        return False, f"{int(bad.sum())} entries off; worst at {i}: got {g[i]!r} expected {x[i]!r} err {err[i]:.3e}"
    return True, f"max abs err {np.where(close, err, 0).max() if err.size else 0:.3e}"
