"""The motion sffg_sweep_edges certifies, in the kernel's operation order: pose(tau) = start + tau (end - start) per
coordinate in double, each operation rounded to nearest; angles start + tau * wrap(end - start) (ROT_INTERPOLATE) or 0
(ROT_REFERENCE); and the motion bound mu of include/sffg.h: |end_xyz - start_xyz|, plus rho times the sum of the wrapped
angle differences in interpolate mode (here with the exact rho, not the kernel's rounded-up one)."""
import numpy as np

from edge_samples import wrap


def poses(starts, ends, tau, rot_mode=0):
    """edges [n][6] (or one edge [6], broadcast) at parameters tau [n] -> float64 [n][6]"""
    s = np.atleast_2d(np.asarray(starts, dtype=np.float64))
    f = np.atleast_2d(np.asarray(ends, dtype=np.float64))
    t = np.asarray(tau, dtype=np.float64).reshape(-1, 1)
    out = np.zeros((max(len(s), len(t)), 6))
    out[:, :3] = s[:, :3] + t * (f[:, :3] - s[:, :3])
    if rot_mode == 1:
        out[:, 3:] = s[:, 3:] + t * wrap(f[:, 3:] - s[:, 3:])
    return out


def motion_bound(starts, ends, rho, rot_mode=0):
    """-> float64 [n]: no robot point moves faster than this per unit tau"""
    s = np.atleast_2d(np.asarray(starts, dtype=np.float64))
    f = np.atleast_2d(np.asarray(ends, dtype=np.float64))
    mu = np.linalg.norm(f[:, :3] - s[:, :3], axis=1)
    if rot_mode == 1:
        mu = mu + rho * np.abs(wrap(f[:, 3:] - s[:, 3:])).sum(axis=1)
    return mu


def radius(robot):
    """rho: the largest distance of a robot vertex from the robot origin"""
    return float(np.linalg.norm(np.asarray(robot, dtype=np.float64).reshape(-1, 3), axis=1).max())
