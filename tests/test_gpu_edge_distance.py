"""GPU tests of the per-edge separation distance (sffg_distance_edges, Environment.EdgeDistance): the minimum of the pose
query over the samples isPathFree checks, bit for bit, the lowest sample reporting it, contact exactly where isPathFree
says not free, and the point, form and argument rules of include/sffg.h."""
import numpy as np
import pytest

import distance_ref as DR
import edge_samples as ES
from conftest import CASES, SEED

pytestmark = pytest.mark.gpu

TOL = 1e-9


def radius(robot):
    return float(np.linalg.norm(np.asarray(robot).reshape(-1, 3), axis=1).max())


def seeded_edges(orc, m, seed, length=4.0):
    s = orc.gen_poses(SEED + seed, 0, m, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
    d = np.random.RandomState(seed).normal(size=(m, 3))
    e = s.copy()
    e[:, :3] += length * d / np.linalg.norm(d, axis=1, keepdims=True)
    return s, e


def expected(env, starts, ends, md, rot_mode):
    """(dist, index, samples, edge of each sample, index of each sample, pose distances) from env.Distance"""
    poses, edge, index = ES.all_samples(starts, ends, 0.1, rot_mode)
    dp = env.Distance(poses, md) if len(poses) else np.zeros(0)
    m = len(starts)
    dist = np.full(m, float(md))
    np.minimum.at(dist, edge, dp)
    best = np.zeros(m, dtype=np.int64)
    first = np.full(m, np.iinfo(np.int64).max)
    at = dp == dist[edge]
    np.minimum.at(first, edge[at], index[at])
    reached = dist < md
    best[reached] = first[reached]
    return dist, best, poses, edge, index


def check_edges(env, obst, robot, starts, ends, md, rot_mode):
    d, idx, pts = env.EdgeDistance(starts, ends, md, 0.1, rot_mode, points=True)
    free, first = env.isPathFree(starts, ends, 0.1, rot_mode, want_first_hit=True)
    dist, best, poses, edge, index = expected(env, starts, ends, md, rot_mode)
    np.testing.assert_array_equal(d, dist)
    np.testing.assert_array_equal(d == 0, free == 0)
    np.testing.assert_array_equal(idx[free == 0], first[free == 0])
    np.testing.assert_array_equal(idx[free == 1], best[free == 1])
    written = (d > 0) & (d < md)
    np.testing.assert_array_equal(~np.isnan(pts).any(1), written)
    # points: on the robot at sample index, on the soup, as far apart as the distance
    S = max(1.0, float(np.abs(obst).max()), float(np.abs(poses[:, :3]).max()) + radius(robot)) if len(poses) else 1.0
    w = np.nonzero(written)[0]
    gap = np.linalg.norm(pts[w, :3] - pts[w, 3:], axis=1)
    assert np.all(np.abs(gap - d[w]) <= TOL * S)
    for i in w[:: max(1, len(w) // 25)]:
        k = np.nonzero((edge == i) & (index == idx[i]))[0][0]
        assert DR.point_soup_distance(pts[i, 3:], obst) <= TOL * S
        assert DR.point_soup_distance(pts[i, :3], DR.place(robot, poses[k])) <= TOL * S
    return d, idx


@pytest.mark.parametrize("rot_mode", [0, 1])
def test_against_pose_query(sff, orc, meshes, gold_edges, rot_mode):
    rho = radius(meshes["robot_small_s10"])
    caps = (0.1 * rho, rho, 4 * rho, np.inf)
    env = sff.Environment(meshes["building_s10"], meshes["robot_small_s10"])
    s, e = seeded_edges(orc, 20000, 31)
    if rot_mode == 1:
        e[:, 3:] = orc.gen_poses(SEED + 32, 0, len(e), [-45, 45, -45, 45, 0, 125]).astype(np.float64)[:, 3:]
    s = np.concatenate([gold_edges["B_starts"], s])
    e = np.concatenate([gold_edges["B_ends"], e])
    for md in caps:
        d, idx = check_edges(env, meshes["building_s10"], meshes["robot_small_s10"], s, e, md, rot_mode)
        assert 0 < (d == 0).mean() < 1 and (0 < d).any()
    # triang_s10 and the long 2-D golden edges (hundreds of samples each)
    for on, rn, ss, ee in (("triang_s10", "robot_cyl_small_s10", *seeded_edges(orc, 2000, 33, 6.0)),
                           ("triangles_tri", "robot_small_s1", gold_edges["2D_starts"], gold_edges["2D_ends"])):
        env2 = sff.Environment(meshes[on], meshes[rn])
        r2 = radius(meshes[rn])
        for md in (0.1 * r2, r2, 4 * r2, np.inf):
            check_edges(env2, meshes[on], meshes[rn], ss, ee, md, rot_mode)


def test_against_independent_reference(sff, orc, meshes):
    ob, rb = meshes["building_s10"], meshes["robot_small_s10"]
    env = sff.Environment(ob, rb)
    s, e = seeded_edges(orc, 400, 41, 1.0)
    d, idx = env.EdgeDistance(s, e)
    free = np.nonzero((d > 0) & np.isfinite(d))[0][:40]
    assert len(free) == 40
    for i in free:
        p = ES.edge_samples(s[i], e[i])
        dref, _ = DR.distance_batch(ob, rb, p)
        S = max(1.0, float(np.abs(ob).max()), float(np.abs(p[:, :3]).max()) + radius(rb))
        assert abs(d[i] - dref.min()) <= TOL * S


def test_grazing_edges(sff, orc, meshes):
    """edges parallel to a floor bisected on their height: the colliding one reports 0, the free one 0 < dist <= 1e-8 S"""
    rob = meshes["robot_small_s1"]
    floor = np.array([[[-50, -50, 0.0], [50, -50, 0.0], [0, 50, 0.0]]])
    env = sff.Environment(floor, rob)
    m = 40
    r = np.random.RandomState(4)
    s = np.zeros((m, 6))
    s[:, :2] = r.uniform(-5, 5, (m, 2))
    e = s.copy()
    e[:, :2] += r.uniform(-3, 3, (m, 2))
    lo, hi = np.full(m, -1.0), np.full(m, 1.0)   # lo: colliding height, hi: free height
    for _ in range(80):
        mid = 0.5 * (lo + hi)
        s[:, 2] = e[:, 2] = mid
        free, _ = orc.edges_free(floor, rob, s, e, 0.1, 0)[:2]
        lo = np.where(free == 0, mid, lo)
        hi = np.where(free == 1, mid, hi)
    sc, ec, sf, ef = s.copy(), e.copy(), s.copy(), e.copy()
    sc[:, 2] = ec[:, 2] = lo
    sf[:, 2] = ef[:, 2] = hi
    assert np.all(env.EdgeDistance(sc, ec)[0] == 0)
    d = env.EdgeDistance(sf, ef)[0]
    S = max(1.0, 50.0)
    assert np.all(d > 0) and np.all(d <= 1e-8 * S), np.max(d / S)


def test_forms_and_splits(sff, orc, meshes):
    import torch
    env = sff.Environment(meshes["building_s10"], meshes["robot_small_s10"])
    md = 4 * radius(meshes["robot_small_s10"])
    s, e = seeded_edges(orc, 20000, 51)
    d, idx = env.EdgeDistance(s, e, md)
    for m in (1, 7, 600, 20000):
        dm, im, pm = env.EdgeDistance(s[:m], e[:m], md, points=True)
        np.testing.assert_array_equal(dm, d[:m])
        np.testing.assert_array_equal(im, idx[:m])
        ts, te = torch.from_numpy(s[:m]).cuda(), torch.from_numpy(e[:m]).cuda()
        out = torch.empty(m, dtype=torch.float64, device="cuda")
        io = torch.empty(m, dtype=torch.int32, device="cuda")
        po = torch.empty((m, 6), dtype=torch.float64, device="cuda")
        env.edge_distance_device(ts, te, md, out=out, index_out=io, points=po)
        env.sync_check()
        np.testing.assert_array_equal(out.cpu().numpy(), dm)
        np.testing.assert_array_equal(io.cpu().numpy(), im)
        np.testing.assert_array_equal(po.cpu().numpy(), pm)
    # one host call above the staging size (chunked), and its pieces
    big_s, big_e = np.concatenate([s] * 15), np.concatenate([e] * 15)
    db, ib = env.EdgeDistance(big_s, big_e, md)
    np.testing.assert_array_equal(db, np.tile(d, 15))
    np.testing.assert_array_equal(ib, np.tile(idx, 15))


def test_builders_and_refit(sff, orc, meshes):
    ob, rb = meshes["building_s10"], meshes["robot_small_s10"]
    host = sff.Environment(ob, rb, build=sff.BUILD_HOST)
    dev = sff.Environment(ob, rb, build=sff.BUILD_DEVICE)
    s, e = seeded_edges(orc, 3000, 61)
    for md in (radius(rb), np.inf):
        a, b = host.EdgeDistance(s, e, md), dev.EdgeDistance(s, e, md)
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1], b[1])
    c, sn = np.cos(0.05), np.sin(0.05)
    moved = ob @ np.array([[c, -sn, 0.0], [sn, c, 0.0], [0.0, 0.0, 1.0]]).T + [0.7, -0.4, 0.3]
    dev.refit_obstacles(moved)
    check_edges(dev, moved, rb, s[:500], e[:500], np.inf, 0)


def test_edge_cases_and_errors(sff, meshes):
    import ctypes as C
    obst, robot = meshes["triang_s10"], meshes["robot_cyl_small_s10"]
    env = sff.Environment(obst, robot)
    s = np.random.RandomState(0).uniform(-50, 50, (100, 6))
    e = s.copy()
    e[50:, 0] += 0.05   # shorter than sample_dist: no samples
    for md in (2.5, np.inf):
        d, idx, pts = env.EdgeDistance(s, e, md, points=True)
        assert np.all(d == md) and np.all(idx == 0) and np.all(np.isnan(pts))
    d, idx, pts = env.EdgeDistance(np.zeros((0, 6)), np.zeros((0, 6)), 1.0, points=True)
    assert d.shape == (0,) and idx.shape == (0,) and pts.shape == (0, 6)
    empty = sff.Environment(np.zeros((0, 3, 3)), robot)
    e2 = s + 3.0
    for md in (2.5, np.inf):
        d, idx, pts = empty.EdgeDistance(s, e2, md, points=True)
        assert np.all(d == md) and np.all(idx == 0) and np.all(np.isnan(pts))
    L = sff._lib.load()
    out = np.empty(100)
    ok = env.EdgeDistance(s, e2, 5.0)
    d_only = np.empty(100)
    assert L.sffg_distance_edges(env._h, s.ctypes.data, e2.ctypes.data, 100, 0.1, 0, 5.0, d_only.ctypes.data, None, None) == 0
    np.testing.assert_array_equal(d_only, ok[0])
    for bad in (0.0, -1.0, np.nan):
        with pytest.raises(sff.SffgError) as ei:
            env.EdgeDistance(s, e2, bad)
        assert ei.value.code == 3
    args = (s.ctypes.data, e2.ctypes.data, 100, 0.1, 0, 1.0, out.ctypes.data, None, None)
    assert L.sffg_distance_edges(None, *args) == 3
    assert L.sffg_distance_edges(env._h, None, *args[1:]) == 3
    assert L.sffg_distance_edges(env._h, args[0], None, *args[2:]) == 3
    assert L.sffg_distance_edges(env._h, *args[:6], None, None, None) == 3
    assert L.sffg_distance_edges(env._h, *args[:3], 0.0, *args[4:]) == 3
    assert L.sffg_distance_edges(env._h, *args[:4], 2, *args[5:]) == 3
    assert L.sffg_distance_edges(env._h, args[0], args[1], -1, *args[3:]) == 3
    assert L.sffg_distance_edges_device(env._h, None, C.c_void_p(16), 100, 0.1, 0, 1.0, C.c_void_p(16), None, None, None) == 3
    assert L.sffg_distance_edges_device(env._h, C.c_void_p(16), C.c_void_p(16), -1, 0.1, 0, 1.0, C.c_void_p(16), None, None, None) == 3
