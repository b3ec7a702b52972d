"""The sample poses of an edge as Solver<T,R>::isPathFree visits them (src/problemStruct.h:154-168), in the operation
order of the edge kernels: parts = distance6 / sample_dist, indices 1 .. S with index < parts, position
start + (index * dir) / parts in double, angles wrapped into [-pi, pi) and interpolated the same way (ROT_INTERPOLATE) or
0 (ROT_REFERENCE)."""
import numpy as np

PI = 3.14159265358979323846


def wrap(a):
    return np.where(a < -PI, a + 2.0 * PI, np.where(a >= PI, a - 2.0 * PI, a))


def edge_samples(start, end, sample_dist=0.1, rot_mode=0):
    """-> float64 [S][6]: the sample poses of one edge, sample k (1-based) in row k - 1"""
    s = np.asarray(start, dtype=np.float64)
    f = np.asarray(end, dtype=np.float64)
    total = 0.0
    for k in range(3):
        d = s[k] - f[k]
        total = total + d * d
    adir = [float(wrap(f[3 + k] - s[3 + k])) for k in range(3)]
    for k in range(3):
        total = total + adir[k] * adir[k]
    parts = np.sqrt(total) / sample_dist
    S = int(np.ceil(parts)) - 1 if parts > 1.0 else 0
    idx = np.arange(1, S + 1, dtype=np.float64)
    out = np.zeros((S, 6))
    for k in range(3):
        out[:, k] = s[k] + (idx * (f[k] - s[k])) / parts
        if rot_mode == 1:
            out[:, 3 + k] = s[3 + k] + (idx * adir[k]) / parts
    return out


def all_samples(starts, ends, sample_dist=0.1, rot_mode=0):
    """-> (poses float64 [N][6], edge of each pose int64 [N], sample index of each pose int64 [N])"""
    rows, edge, index = [], [], []
    for e, (s, f) in enumerate(zip(np.asarray(starts), np.asarray(ends))):
        p = edge_samples(s, f, sample_dist, rot_mode)
        rows.append(p)
        edge.append(np.full(len(p), e, dtype=np.int64))
        index.append(np.arange(1, len(p) + 1, dtype=np.int64))
    if not rows:
        return np.zeros((0, 6)), np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    return np.concatenate(rows), np.concatenate(edge), np.concatenate(index)
