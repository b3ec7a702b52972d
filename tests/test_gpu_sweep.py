"""GPU tests of the continuous edge check (sffg_sweep_edges, Environment.SweepEdges): the certificate of include/sffg.h on
a dense grid of the motion, the stop pose against the pose query bit for bit, completeness through the motion bound,
consistency with isPathFree, walls and poles that the samples step over, forms, splits, builders, edge cases and the
argument errors."""
import numpy as np
import pytest

import edge_samples as ES
import sweep_motion as SM
from conftest import SEED

pytestmark = pytest.mark.gpu

TOL = 1e-9
GRID = 64


def seeded_edges(orc, m, seed, length=4.0, rot_mode=0):
    s = orc.gen_poses(SEED + seed, 0, m, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
    d = np.random.RandomState(seed).normal(size=(m, 3))
    e = s.copy()
    e[:, :3] += length * d / np.linalg.norm(d, axis=1, keepdims=True)
    if rot_mode == 1:
        e[:, 3:] = orc.gen_poses(SEED + seed + 1, 0, m, [-45, 45, -45, 45, 0, 125]).astype(np.float64)[:, 3:]
    return s, e


def scale(obst, s, e, robot):
    """S of the pose query's accuracy bound over every pose of the motions"""
    reach = max(float(np.abs(s[:, :3]).max()), float(np.abs(e[:, :3]).max())) if len(s) else 0.0
    return max(1.0, float(np.abs(obst).max()) if len(obst) else 0.0, reach + SM.radius(robot))


def grid_taus(s, e, rot_mode):
    """per edge: GRID evenly spaced tau on [0, 1] plus the tau of every isPathFree sample -> (edge of each tau, tau,
    largest gap between neighbouring taus of each edge)"""
    edge, tau, gap = [], [], np.zeros(len(s))
    for i in range(len(s)):
        n = len(ES.edge_samples(s[i], e[i], 0.1, rot_mode))
        f = e[i]
        total = sum((s[i][k] - f[k]) ** 2 for k in range(3)) + sum(float(ES.wrap(f[3 + k] - s[i][3 + k])) ** 2 for k in range(3))
        ts = np.unique(np.concatenate([np.linspace(0.0, 1.0, GRID), np.arange(1, n + 1) / (np.sqrt(total) / 0.1)]))
        gap[i] = np.diff(ts).max()
        edge.append(np.full(len(ts), i))
        tau.append(ts)
    return np.concatenate(edge), np.concatenate(tau), gap


def check_sweep(env, obst, robot, s, e, margin, rot_mode, label=""):
    clear, t, dist = env.SweepEdges(s, e, margin, rot_mode)
    S = scale(obst, s, e, robot)
    c, st = clear == 1, clear == 0
    assert np.all(c | st)
    assert np.all(t[c] == 1.0) and np.all(dist[c] == margin)
    assert np.all((t[st] >= 0) & (t[st] < 1)) and np.all(dist[st] < margin)
    # the stop pose: the pose query at max_dist = margin, bit for bit; 0 exactly on contact
    ps = SM.poses(s[st], e[st], t[st], rot_mode)
    if len(ps):
        np.testing.assert_array_equal(env.Distance(ps, margin), dist[st])
        np.testing.assert_array_equal(dist[st] == 0, env.Collide(ps) == 1)
    # the certified part: [0, t) of stopped edges, [0, 1] of clear ones
    edge, tau, gap = grid_taus(s, e, rot_mode)
    d = env.Distance(SM.poses(s[edge], e[edge], tau, rot_mode), np.inf)
    certified = c[edge] | (tau < t[edge])
    assert np.all(d[certified] >= 0.5 * margin - TOL * S), (label, np.min(d[certified] - 0.5 * margin))
    # completeness: a grid minimum that keeps every pose >= margin away (through mu) forces a clear edge
    gmin = np.full(len(s), np.inf)
    np.minimum.at(gmin, edge, d)
    must = gmin >= margin + 0.5 * SM.motion_bound(s, e, SM.radius(robot), rot_mode) * gap + TOL * S
    assert np.all(clear[must] == 1), (label, np.nonzero(must & st)[0][:8])
    assert np.all(clear[gmin < 0.5 * margin - TOL * S] == 0)
    # consistency with sampling: a clear motion passes isPathFree
    free = env.isPathFree(s, e, 0.1, rot_mode)
    assert np.all(free[c] == 1)
    print(f"{label} margin {margin:.4g} mode {rot_mode}: {int(c.sum())}/{len(s)} clear, {int((st & (dist == 0)).sum())} stop "
          f"in contact; isPathFree passes {int((free == 1).sum())}, of which the sweep stops {int(((free == 1) & st).sum())}; "
          f"{int(must.sum())} clear through mu")
    return clear, t, dist


def margin_floor(obst):
    """1e-6 max(1, max |obstacle coordinate| rounded up to float): the smallest margin sffg_sweep_edges accepts"""
    a = float(np.abs(obst).max()) if len(obst) else 0.0
    f = np.float32(a)
    if float(f) < a:
        f = np.nextafter(f, np.float32(np.inf))
    return 1e-6 * max(1.0, float(f))


@pytest.mark.parametrize("rot_mode", [0, 1])
def test_certificate_on_the_golden_scenes(sff, orc, meshes, gold_edges, rot_mode):
    ob, rb = meshes["building_s10"], meshes["robot_small_s10"]
    env = sff.Environment(ob, rb)
    rho = SM.radius(rb)
    s, e = seeded_edges(orc, 1500, 71, rot_mode=rot_mode)
    s = np.concatenate([gold_edges["B_starts"], s])
    e = np.concatenate([gold_edges["B_ends"], e])
    for margin in (0.01 * rho, 0.1 * rho, rho):
        clear, t, dist = check_sweep(env, ob, rb, s, e, margin, rot_mode, "building")
        assert 0 < clear.mean() < 1 and (dist == 0).any() and ((dist > 0) & (dist < margin)).any()
    for on, rn, ss, ee in (("triang_s10", "robot_cyl_small_s10", *seeded_edges(orc, 600, 73, 6.0, rot_mode)),
                           ("triangles_tri", "robot_small_s1", gold_edges["2D_starts"], gold_edges["2D_ends"])):
        env2 = sff.Environment(meshes[on], meshes[rn])
        r2 = SM.radius(meshes[rn])
        for margin in (0.01 * r2, 0.1 * r2, r2):
            check_sweep(env2, meshes[on], meshes[rn], ss, ee, margin, rot_mode, on)


def test_thin_wall_between_samples(sff):
    """a flat robot crossing a wall of no thickness between two samples: isPathFree says free, the sweep stops just before
    the wall, at the place the closed form gives"""
    robot = np.array([[[0.0, -0.2, -0.2], [0.0, 0.2, -0.2], [0.0, 0.0, 0.3]]])
    wall = np.array([[[0.05, -5, -5], [0.05, 5, -5], [0.05, -5, 5]], [[0.05, 5, -5], [0.05, 5, 5], [0.05, -5, 5]]])
    env = sff.Environment(wall, robot)
    s = np.array([[-1.0, 0, 0, 0, 0, 0], [-1.0, 1, 1, 0, 0, 0]])
    e = np.array([[1.0, 0, 0, 0, 0, 0], [1.0, 1, 1, 0, 0, 0]])
    assert np.all(env.isPathFree(s, e, 0.1, 0) == 1)
    L, tc = 2.0, 0.525   # travel, and the tau at which the robot lies in the wall's plane
    for margin in (0.001, 0.01, 0.02, 0.04):
        clear, t, dist = env.SweepEdges(s, e, margin)
        assert np.all(clear == 0)
        assert np.all(t >= tc - margin / L - 1e-12) and np.all(t <= tc - margin / (2 * L) + 1e-12), t
        assert np.all(dist >= 0.5 * margin - 1e-9) and np.all(dist < margin), dist
        np.testing.assert_array_equal(env.Distance(SM.poses(s, e, t), margin), dist)
        check_sweep(env, wall, robot, s, e, margin, 0, "wall")


def test_pole_swept_by_yaw(sff):
    """interpolate mode, a pure-yaw edge that swings a blade through a pole of no thickness between two samples"""
    blade = np.array([[[0.8, 0.0, -0.8], [1.8, 0.0, -0.8], [1.3, 0.0, 0.8]]])
    phi = 0.55
    c, sn = np.cos(phi), np.sin(phi)
    pole = np.array([[[1.0 * c, 1.0 * sn, -1.0], [1.5 * c, 1.5 * sn, -1.0], [1.25 * c, 1.25 * sn, 1.0]]])
    env = sff.Environment(pole, blade)
    s = np.array([[0.0, 0, 0, 0.0, 0, 0]])
    e = np.array([[0.0, 0, 0, 1.0, 0, 0]])   # yaw 0 -> 1: samples at yaw 0.1 k, the pole at 0.55
    assert env.isPathFree(s, e, 0.1, 1)[0] == 1
    assert env.isPathFree(s, e, 0.1, 0)[0] == 1
    touching = SM.poses(s, e, [phi], 1)
    assert env.Distance(touching, 1.0)[0] < 1e-9
    for margin in (0.005, 0.02, 0.1):
        clear, t, dist = env.SweepEdges(s, e, margin, 1)
        assert clear[0] == 0 and t[0] < phi and 0.5 * margin - 1e-9 <= dist[0] < margin, (t, dist)
        check_sweep(env, pole, blade, s, e, margin, 1, "pole")
        # reference mode keeps the identity rotation: the blade never turns into the pole
        assert env.SweepEdges(s, e, margin, 0)[0][0] == 1


def test_forms_and_splits(sff, orc, meshes):
    import torch
    env = sff.Environment(meshes["building_s10"], meshes["robot_small_s10"])
    margin = 0.1 * SM.radius(meshes["robot_small_s10"])
    for rot_mode in (0, 1):
        s, e = seeded_edges(orc, 20000, 81, rot_mode=rot_mode)
        ref = env.SweepEdges(s, e, margin, rot_mode)
        for m in (1, 7, 600, 20000):
            got = env.SweepEdges(s[:m], e[:m], margin, rot_mode)
            for a, b in zip(got, ref):
                np.testing.assert_array_equal(a, b[:m])
            ts, te = torch.from_numpy(s[:m]).cuda(), torch.from_numpy(e[:m]).cuda()
            co = torch.empty(m, dtype=torch.uint8, device="cuda")
            to = torch.empty(m, dtype=torch.float64, device="cuda")
            do = torch.empty(m, dtype=torch.float64, device="cuda")
            env.sweep_edges_device(ts, te, margin, rot_mode, clear_out=co, t_out=to, dist_out=do)
            env.sync_check()
            for a, b in zip((co, to, do), ref):
                np.testing.assert_array_equal(a.cpu().numpy(), b[:m])
            only = env.sweep_edges_device(ts, te, margin, rot_mode)
            env.sync_check()
            np.testing.assert_array_equal(only.cpu().numpy(), ref[0][:m])
        # one host call above the staging size, in several chunks
        big = env.SweepEdges(np.concatenate([s] * 15), np.concatenate([e] * 15), margin, rot_mode)
        for a, b in zip(big, ref):
            np.testing.assert_array_equal(a, np.tile(b, 15))


def test_builders_and_refit(sff, orc, meshes):
    ob, rb = meshes["building_s10"], meshes["robot_small_s10"]
    host = sff.Environment(ob, rb, build=sff.BUILD_HOST)
    dev = sff.Environment(ob, rb, build=sff.BUILD_DEVICE)
    rho = SM.radius(rb)
    for rot_mode in (0, 1):
        s, e = seeded_edges(orc, 3000, 91, rot_mode=rot_mode)
        for margin in (0.01 * rho, rho):
            for a, b in zip(host.SweepEdges(s, e, margin, rot_mode), dev.SweepEdges(s, e, margin, rot_mode)):
                np.testing.assert_array_equal(a, b)
    c, sn = np.cos(0.05), np.sin(0.05)
    moved = ob @ np.array([[c, -sn, 0.0], [sn, c, 0.0], [0.0, 0.0, 1.0]]).T + [0.7, -0.4, 0.3]
    dev.refit_obstacles(moved)
    s, e = seeded_edges(orc, 500, 93)
    check_sweep(dev, moved, rb, s, e, 0.1 * rho, 0, "refit")


def test_edge_cases(sff, meshes):
    obst, robot = meshes["triang_s10"], meshes["robot_cyl_small_s10"]
    env = sff.Environment(obst, robot)
    r = np.random.RandomState(0)
    s = np.concatenate([r.uniform(-60, 60, (400, 2)), r.uniform(0, 100, (400, 1)), r.uniform(-3, 3, (400, 3))], axis=1)
    for margin in (0.5, 2.0):
        for rot_mode in (0, 1):
            # zero-length edges: one pose decides
            clear, t, dist = env.SweepEdges(s, s, margin, rot_mode)
            d0 = env.Distance(SM.poses(s, s, np.zeros(len(s)), rot_mode), margin)
            np.testing.assert_array_equal(clear == 1, d0 >= margin)
            assert np.all(t[clear == 0] == 0) and np.all(t[clear == 1] == 1)
            np.testing.assert_array_equal(dist, d0)
        # rotations without translation in reference mode: motionless (mu = 0), the identity pose decides
        e = s.copy()
        e[:, 3:] = r.uniform(-3, 3, (len(s), 3))
        clear, t, dist = env.SweepEdges(s, e, margin, 0)
        d0 = env.Distance(SM.poses(s, s, np.zeros(len(s)), 0), margin)
        np.testing.assert_array_equal(clear == 1, d0 >= margin)
        np.testing.assert_array_equal(dist, d0)
        assert 0 < clear.mean() < 1
    # no obstacles: everything clear
    empty = sff.Environment(np.zeros((0, 3, 3)), robot)
    e = s + 3.0
    for rot_mode in (0, 1):
        clear, t, dist = empty.SweepEdges(s, e, 0.25, rot_mode)
        assert np.all(clear == 1) and np.all(t == 1.0) and np.all(dist == 0.25)
    # no edges
    clear, t, dist = env.SweepEdges(np.zeros((0, 6)), np.zeros((0, 6)), 1.0)
    assert clear.shape == t.shape == dist.shape == (0,)
    # a non-finite coordinate the motion uses: never clear, t = 0, dist = NaN
    bad_s, bad_e = s[:3].copy(), s[:3] + 1.0
    bad_e[0, 0] = np.nan
    bad_e[1, 1] = np.inf
    bad_e[2, 3] = np.nan
    clear, t, dist = env.SweepEdges(bad_s, bad_e, 1.0, 1)
    assert np.all(clear == 0) and np.all(t == 0) and np.all(np.isnan(dist))
    assert env.SweepEdges(bad_s[2:], bad_e[2:], 1.0, 0)[0][0] in (0, 1)   # reference mode ignores the angles


def test_argument_errors(sff, meshes):
    import ctypes as C
    obst, robot = meshes["triang_s10"], meshes["robot_cyl_small_s10"]
    env = sff.Environment(obst, robot)
    L = sff._lib.load()
    s = np.random.RandomState(1).uniform(-50, 50, (10, 6))
    e = s + 1.0
    cl, t, d = np.empty(10, dtype=np.uint8), np.empty(10), np.empty(10)
    args = (s.ctypes.data, e.ctypes.data, 10, 0, 1.0, cl.ctypes.data, t.ctypes.data, d.ctypes.data)
    assert L.sffg_sweep_edges(env._h, *args) == 0
    assert L.sffg_sweep_edges(env._h, *args[:6], None, None) == 0   # t and dist are optional
    np.testing.assert_array_equal(cl, env.SweepEdges(s, e, 1.0)[0])
    assert L.sffg_sweep_edges(None, *args) == 3
    assert L.sffg_sweep_edges(env._h, None, *args[1:]) == 3
    assert L.sffg_sweep_edges(env._h, args[0], None, *args[2:]) == 3
    assert L.sffg_sweep_edges(env._h, *args[:5], None, *args[6:]) == 3
    assert L.sffg_sweep_edges(env._h, args[0], args[1], -1, *args[3:]) == 3
    assert L.sffg_sweep_edges(env._h, *args[:3], 2, *args[4:]) == 3
    lim = margin_floor(obst)
    for bad in (0.0, -1.0, np.nan, np.inf, 0.5 * lim):
        assert L.sffg_sweep_edges(env._h, *args[:4], bad, *args[5:]) == 3, bad
        assert L.sffg_sweep_edges(env._h, None, None, 0, 0, bad, None, None, None) == 3, bad
        assert L.sffg_sweep_edges_device(env._h, None, None, 0, 0, bad, None, None, None, None) == 3, bad
        with pytest.raises(sff.SffgError) as ei:
            env.SweepEdges(s, e, bad)
        assert ei.value.code == 3
    assert L.sffg_sweep_edges(env._h, None, None, 0, 0, lim, None, None, None) == 0
    assert L.sffg_sweep_edges_device(env._h, None, None, 0, 0, lim, None, None, None, None) == 0
    # the floor of the limit is 1e-6 (obstacles within the unit box, or none)
    empty = sff.Environment(np.zeros((0, 3, 3)), robot)
    assert L.sffg_sweep_edges(empty._h, None, None, 0, 0, 0.9e-6, None, None, None) == 3
    assert L.sffg_sweep_edges(empty._h, None, None, 0, 0, 1e-6, None, None, None) == 0
    dev = (C.c_void_p(16), C.c_void_p(16))
    assert L.sffg_sweep_edges_device(None, *dev, 10, 0, 1.0, C.c_void_p(16), None, None, None) == 3
    assert L.sffg_sweep_edges_device(env._h, None, dev[1], 10, 0, 1.0, C.c_void_p(16), None, None, None) == 3
    assert L.sffg_sweep_edges_device(env._h, *dev, 10, 0, 1.0, None, None, None, None) == 3
    assert L.sffg_sweep_edges_device(env._h, *dev, -1, 0, 1.0, C.c_void_p(16), None, None, None) == 3
    assert L.sffg_sweep_edges_device(env._h, *dev, 10, 2, 1.0, C.c_void_p(16), None, None, None) == 3
    for bad in (0.0, -1.0, np.nan, np.inf, 0.5 * lim):
        assert L.sffg_sweep_edges_device(env._h, *dev, 10, 0, bad, C.c_void_p(16), None, None, None) == 3
