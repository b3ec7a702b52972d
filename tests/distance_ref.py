"""CPU reference of the separation distance (sffg_distance_poses), written apart from the CUDA kernel: numpy, float64.

Triangle pairs are measured by enumeration -- every segment pair minimised over the unit square of its parameters by
its interior critical point and the clamped optimum on each of the square's four sides (the distance is convex there), and
every vertex measured against the other triangle by its foot on the plane when that lies inside, else against the three
edges.  A pose's distance is the minimum over all (obstacle triangle, robot triangle) pairs; triangles are visited in
order of their box distance to the placed robot's box, and the visit stops once that bound exceeds the best distance."""
import numpy as np


def rotation(yaw, pitch, roll):
    """FillRotationMatrix (ZYX Euler) for arrays of angles -> [n][3][3]"""
    sy, cy, sp, cp, sr, cr = np.sin(yaw), np.cos(yaw), np.sin(pitch), np.cos(pitch), np.sin(roll), np.cos(roll)
    R = np.empty(np.shape(yaw) + (3, 3))
    R[..., 0, 0] = cy * cp
    R[..., 0, 1] = cy * sp * sr - sy * cr
    R[..., 0, 2] = cy * sp * cr + sy * sr
    R[..., 1, 0] = sy * cp
    R[..., 1, 1] = sy * sp * sr + cy * cr
    R[..., 1, 2] = sy * sp * cr - cy * sr
    R[..., 2, 0] = -sp
    R[..., 2, 1] = cp * sr
    R[..., 2, 2] = cp * cr
    return R


def place(robot, pose):
    """robot triangles [m][3][3] at pose (x y z yaw pitch roll) in the world frame"""
    pose = np.asarray(pose, dtype=np.float64)
    R = rotation(pose[3], pose[4], pose[5])
    return np.asarray(robot, dtype=np.float64).reshape(-1, 3, 3) @ R.T + pose[:3]


def _dot(a, b):
    return (a * b).sum(-1)


def point_segment(x, a, b):
    """nearest point of segment [a, b] to x (arrays [..., 3])"""
    d = b - a
    dd = _dot(d, d)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(dd > 0, np.clip(_dot(x - a, d) / np.where(dd > 0, dd, 1.0), 0.0, 1.0), 0.0)
    return a + t[..., None] * d


def seg_seg(p0, p1, q0, q1):
    """-> (squared distance, point on [p0, p1], point on [q0, q1])"""
    d1, d2, r = p1 - p0, q1 - q0, p0 - q0
    a, e, b, c, f = _dot(d1, d1), _dot(d2, d2), _dot(d1, d2), _dot(d1, r), _dot(d2, r)
    cand = []
    one = np.ones_like(a)
    with np.errstate(divide="ignore", invalid="ignore"):
        for s in (0.0, 1.0):
            t = np.where(e > 0, np.clip((b * s + f) / np.where(e > 0, e, 1.0), 0.0, 1.0), 0.0)
            cand.append((s * one, t))
        for t in (0.0, 1.0):
            s = np.where(a > 0, np.clip((b * t - c) / np.where(a > 0, a, 1.0), 0.0, 1.0), 0.0)
            cand.append((s, t * one))
        den = a * e - b * b
        ok = den > 1e-300
        si = np.where(ok, (b * f - c * e) / np.where(ok, den, 1.0), 0.0)
        ti = np.where(ok, (a * f - b * c) / np.where(ok, den, 1.0), 0.0)
        inside = ok & (si >= 0) & (si <= 1) & (ti >= 0) & (ti <= 1)
        cand.append((np.where(inside, si, 0.0), np.where(inside, ti, 0.0)))
    best = None
    for s, t in cand:
        P, Q = p0 + s[..., None] * d1, q0 + t[..., None] * d2
        d = _dot(P - Q, P - Q)
        if best is None:
            best = [d, P, Q]
        else:
            m = d < best[0]
            best = [np.where(m, d, best[0]), np.where(m[..., None], P, best[1]), np.where(m[..., None], Q, best[2])]
    return best[0], best[1], best[2]


def point_triangle(x, T):
    """nearest point of triangle T [..., 3, 3] to x [..., 3]"""
    a, b, c = T[..., 0, :], T[..., 1, :], T[..., 2, :]
    n = np.cross(b - a, c - a)
    nn = _dot(n, n)
    with np.errstate(divide="ignore", invalid="ignore"):
        foot = x - (_dot(x - a, n) / np.where(nn > 0, nn, 1.0))[..., None] * n
    # barycentric signs of the foot: the sub-triangle normals point along n when it lies inside
    inside = nn > 0
    for u, v in ((a, b), (b, c), (c, a)):
        inside &= _dot(np.cross(v - u, foot - u), n) >= 0
    best = foot
    bd = np.where(inside, _dot(x - foot, x - foot), np.inf)
    for u, v in ((a, b), (b, c), (c, a)):
        p = point_segment(x, u, v)
        d = _dot(x - p, x - p)
        m = d < bd
        bd = np.where(m, d, bd)
        best = np.where(m[..., None], p, best)
    return best


def tri_dist(P, Q):
    """distance of disjoint triangles P, Q ([..., 3, 3]) -> (d, nearest point on P, nearest point on Q)"""
    P = np.asarray(P, dtype=np.float64)
    Q = np.asarray(Q, dtype=np.float64)
    best = None

    def take(d2, p, q):
        nonlocal best
        if best is None:
            best = [d2, p, q]
        else:
            m = d2 < best[0]
            best = [np.where(m, d2, best[0]), np.where(m[..., None], p, best[1]), np.where(m[..., None], q, best[2])]

    for i in range(3):
        for j in range(3):
            take(*seg_seg(P[..., i, :], P[..., (i + 1) % 3, :], Q[..., j, :], Q[..., (j + 1) % 3, :]))
    for i in range(3):
        q = point_triangle(P[..., i, :], Q)
        take(_dot(P[..., i, :] - q, P[..., i, :] - q), P[..., i, :], q)
        p = point_triangle(Q[..., i, :], P)
        take(_dot(Q[..., i, :] - p, Q[..., i, :] - p), p, Q[..., i, :])
    return np.sqrt(best[0]), best[1], best[2]


def distance_batch(obst, robot, poses, max_dist=np.inf, contact=None, chunk=256):
    """-> (dist float64[n], points float64[n][6]) with the rules of sffg_distance_poses: min(d, max_dist), 0 where
    `contact` (the contact verdicts of the poses) is 1; points = robot point, obstacle point, NaN unless 0 < dist < max_dist"""
    O = np.asarray(obst, dtype=np.float64).reshape(-1, 3, 3)
    r = np.asarray(robot, dtype=np.float64).reshape(-1, 3, 3)
    poses = np.asarray(poses, dtype=np.float64).reshape(-1, 6)
    n, nr = len(poses), len(r)
    dist = np.full(n, float(max_dist))
    pts = np.full((n, 6), np.nan)
    if len(O) == 0:
        return dist, pts
    olo, ohi = O.min(1), O.max(1)
    for i in range(n):
        if contact is not None and contact[i]:
            dist[i] = 0.0
            continue
        W = place(r, poses[i])
        lo, hi = W.reshape(-1, 3).min(0), W.reshape(-1, 3).max(0)
        gap = np.maximum(np.maximum(olo - hi, lo - ohi), 0.0)
        lb = np.sqrt((gap * gap).sum(1))
        order = np.argsort(lb, kind="stable")
        best, bp = float(max_dist), None
        for s in range(0, len(order), chunk):
            ids = order[s:s + chunk]
            ids = ids[lb[ids] < best]
            if len(ids) == 0:
                break
            Rt = np.broadcast_to(W[None], (len(ids), nr, 3, 3)).reshape(-1, 3, 3)
            Ot = np.broadcast_to(O[ids][:, None], (len(ids), nr, 3, 3)).reshape(-1, 3, 3)
            d, pr, po = tri_dist(Rt, Ot)
            k = int(np.argmin(d))
            if d[k] < best:
                best, bp = float(d[k]), np.concatenate([pr[k], po[k]])
        if bp is not None:
            dist[i], pts[i] = best, bp
    return dist, pts


def point_soup_distance(x, tris):
    """distance of point x [3] to a triangle soup [m][3][3]"""
    T = np.asarray(tris, dtype=np.float64).reshape(-1, 3, 3)
    p = point_triangle(np.broadcast_to(np.asarray(x, dtype=np.float64), (len(T), 3)), T)
    return float(np.sqrt(_dot(p - x, p - x).min()))
