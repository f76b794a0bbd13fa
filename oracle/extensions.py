"""CPU restatements of the EXTENSION features — TEST INFRASTRUCTURE, PARITY UNPINNED.

Neither exists in the reference (SURVEY.md §0: `grep -i keypoint|quat_rotate` finds nothing and
`leibnizgym/dr/__init__.py` is empty), so there is no reference output to pin against; these
functions state the definitions the CUDA kernels implement (SURVEY.md §8c) in plain torch.
"""
from __future__ import annotations

import numpy as np
import torch

from .trifinger_oracle import OracleEnv, scale_transform

CUBE_SIZE = 0.065


def quat_rotate(q: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """Rotate v [...,3] by unit quaternion q [...,4] (xyzw): v + 2 w (q_v x v) + 2 q_v x (q_v x v)."""
    qv, w = q[..., :3], q[..., 3:4]
    t = 2.0 * torch.cross(qv, v, dim=-1)
    return v + w * t + torch.cross(qv, t, dim=-1)


def cube_keypoints(pose: torch.Tensor, size: float = CUBE_SIZE) -> torch.Tensor:
    """[n,7] poses -> [n,8,3] world-frame corners; corner k has signs (bit0, bit1, bit2) of k."""
    h = size / 2
    corners = torch.tensor([[(h if k & 1 else -h), (h if k & 2 else -h), (h if k & 4 else -h)] for k in range(8)],
                           dtype=pose.dtype)
    p, q = pose[:, None, 0:3], pose[:, None, 3:7].expand(-1, 8, -1)
    return p + quat_rotate(q, corners[None].expand(pose.shape[0], -1, -1))


def keypoint_reward(weight: float, dt: float, obj_pose: torch.Tensor, goal_pose: torch.Tensor,
                    scale: float = 30.0, eps: float = 2.0) -> torch.Tensor:
    """w dt mean_k 1 / (e^{s d_k} + eps + e^{-s d_k}),  d_k = |kp_k(object) - kp_k(goal)|."""
    d = torch.norm(cube_keypoints(obj_pose) - cube_keypoints(goal_pose), p=2, dim=-1)
    s = d * scale
    return (weight * dt) * (1.0 / (s.exp() + eps + (-s).exp())).mean(dim=-1)


def integrate_goal_rows(rows: np.ndarray, dt: float) -> np.ndarray:
    """Oracle of lg_integrate_goal (extension; stands in for PhysX on the moving-goal task's goal body):
    rows [n, 13] = pos | quat xyzw | lin vel | world-frame ang vel.  p += v dt; q <- normalize(exp(w dt/2) (x) q).
    float64 throughout."""
    r = np.asarray(rows, dtype=np.float64).copy()
    w = r[:, 10:13]
    mag = np.linalg.norm(w, axis=1)
    half = 0.5 * mag * dt
    k = np.where(mag > 1e-12, np.sin(half) / np.maximum(mag, 1e-300), 0.5 * dt)
    dq = np.concatenate([w * k[:, None], np.cos(half)[:, None]], axis=1)          # xyzw
    q = r[:, 3:7]
    x1, y1, z1, w1 = dq.T
    x2, y2, z2, w2 = q.T
    out = np.stack([w1 * x2 + x1 * w2 + y1 * z2 - z1 * y2,
                    w1 * y2 - x1 * z2 + y1 * w2 + z1 * x2,
                    w1 * z2 + x1 * y2 - y1 * x2 + z1 * w2,
                    w1 * w2 - x1 * x2 - y1 * y2 - z1 * z2], axis=1)
    r[:, 3:7] = out / np.linalg.norm(out, axis=1, keepdims=True)
    r[:, 0:3] += r[:, 7:10] * dt
    return r


class OffsetOracleEnv(OracleEnv):
    """OracleEnv whose actor observation carries per-episode DR offsets (extension "domain_randomization":
    obs_bias_std): obs = scale_transform(raw + obs_bias) on the columns `bias_cols` (those with sigma != 0; the others
    keep their raw value, -0 included); states stay clean.  The caller sets `obs_bias` [N, obs_dim] to the rows the
    env's resets drew and steps with the perturbed action (action + action offset, clamped like the env)."""

    obs_bias = None
    bias_cols = ()

    def fill_observations_and_states(self):
        norm = self.cfg["normalize_obs"]
        self.cfg["normalize_obs"] = False
        try:
            super().fill_observations_and_states()
        finally:
            self.cfg["normalize_obs"] = norm
        if self.obs_bias is not None and len(self.bias_cols):
            c = list(self.bias_cols)
            self.obs_buf[:, c] = self.obs_buf[:, c] + self.obs_bias[:, c]
        if norm:
            self.obs_buf = scale_transform(self.obs_buf, self.obs_lo, self.obs_hi)
            if self.asym:
                self.states_buf = scale_transform(self.states_buf, self.st_lo, self.st_hi)
