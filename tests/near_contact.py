"""Near-contact poses with double angles that float32 cannot hold (shared by the CPU and GPU tests of the f64 pose paths).

A bracket is a pair of poses that differ only along one translation axis, `lo` colliding and `hi` free, found by bisection
with the CPU oracle until they are less than 1e-9 of the scene scale apart.  Poses moved a small `off` into or out of the
contact and given angles far outside [-pi, pi) are where a kernel that narrows the angle to float before building its
FP32 rotation would give the wrong verdict."""
import numpy as np


def seed_poses(orc, obst_tris, seed, n, rng):
    """n seeded poses: orc.gen_poses in `rng` (3-D), or for a 2-D map (rng None) z = 0, pitch = roll = 0 and x, y, yaw
    uniform over the map's bounds"""
    if rng is not None:
        return orc.gen_poses(seed, 0, n, rng).astype(np.float64)
    r = np.random.RandomState(seed)
    lo, hi = obst_tris.reshape(-1, 3).min(0), obst_tris.reshape(-1, 3).max(0)
    p = np.zeros((n, 6))
    p[:, 0] = r.uniform(lo[0], hi[0], n)
    p[:, 1] = r.uniform(lo[1], hi[1], n)
    p[:, 3] = r.uniform(-np.pi, np.pi, n)
    return p


def boundary_brackets(orc, obst, robot, seed, n, rng, lift, iters=80, axis=2):
    """-> (lo, hi) float64 [k][6]: lo collides, hi = lo moved along `axis` by less than 1e-9 of the scene scale is free.

    `obst`, `robot` are orc.ObbModel; the seeds are the colliding poses of seed_poses(...) that are free once moved by
    +lift along `axis`."""
    p = seed_poses(orc, obst.tris, seed, n, rng)
    hit, _ = orc.collide_obbtree(obst, robot, p)
    up = p.copy()
    up[:, axis] += lift
    up_hit, _ = orc.collide_obbtree(obst, robot, up)
    keep = (hit == 1) & (up_hit == 0)
    lo, hi = p[keep], up[keep]
    tol = 1e-9 * float(np.abs(obst.tris).max())
    for _ in range(iters):
        if len(lo) == 0 or float((hi[:, axis] - lo[:, axis]).max()) < tol:
            break
        mid = lo.copy()
        mid[:, axis] = 0.5 * (lo[:, axis] + hi[:, axis])
        v, _ = orc.collide_obbtree(obst, robot, mid)
        c = v == 1
        lo[c, axis] = mid[c, axis]
        hi[~c, axis] = mid[~c, axis]
    assert len(lo) == 0 or float((hi[:, axis] - lo[:, axis]).max()) < tol, "bisection did not converge"
    return lo, hi


def wide_angles(a, K, seed, cols=(3, 4, 5)):
    """a copy of poses `a` whose angles in `cols` get 2*pi*K*(+-1, random per angle) and a perturbation of about 1e-9 rad
    in double, so that no angle is a float (not even at K = 0)"""
    r = np.random.RandomState(seed)
    out = np.array(a, dtype=np.float64, copy=True)
    cols = list(cols)
    sign = r.choice([-1.0, 1.0], size=(len(out), len(cols)))
    tiny = r.uniform(0.5e-9, 1.5e-9, size=(len(out), len(cols))) * r.choice([-1.0, 1.0], size=(len(out), len(cols)))
    out[:, cols] = out[:, cols] + 2.0 * np.pi * K * sign + tiny
    return out


def near_contact_poses(lo, hi, off, K, seed, axis=2, cols=(3, 4, 5)):
    """-> (inside, outside): lo moved by -off and hi moved by +off along `axis`, both with wide_angles(K).  The verdicts of
    the returned poses are whatever the oracle says of them; moving the angles changes the pose by ~1e-9 rad."""
    inside = np.array(lo, dtype=np.float64, copy=True)
    outside = np.array(hi, dtype=np.float64, copy=True)
    inside[:, axis] -= off
    outside[:, axis] += off
    return wide_angles(inside, K, seed, cols), wide_angles(outside, K, seed + 1, cols)


# per scene (conftest.CASES key): seed poses, lift, bisection axis, perturbed angle columns.  The lifts are about the
# robot's size, which gives ~600-1100 brackets out of 20 000 seeds; in 2-D the bracket runs along x and only yaw moves.
SETUP = {
    "B": (20000, 10.0, 2, (3, 4, 5)),
    "T": (20000, 30.0, 2, (3, 4, 5)),
    "2D": (20000, 10.0, 0, (3,)),
}


def case_brackets(orc, meshes, cases, case, seed):
    """-> (obst model, robot model, lo, hi, axis, cols) of one scene"""
    on, rn, rng = cases[case]
    n, lift, axis, cols = SETUP[case]
    mo, mr = orc.ObbModel(meshes[on]), orc.ObbModel(meshes[rn])
    lo, hi = boundary_brackets(orc, mo, mr, seed, n, rng, lift, axis=axis)
    return mo, mr, lo, hi, axis, cols


def narrowed(poses):
    """the poses with their angles rounded to float32 (what an FP32 stage that narrows the angle sees)"""
    out = np.array(poses, dtype=np.float64, copy=True)
    out[:, 3:] = out[:, 3:].astype(np.float32).astype(np.float64)
    return out
