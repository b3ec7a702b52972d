"""GPU tests of the separation distance query (sffg_distance_poses, Environment.Distance) against the CPU reference of
tests/distance_ref.py: contact gives exactly 0, free poses their distance within 1e-9 S, the cap and the point rules."""
import numpy as np
import pytest

import distance_ref as DR
import near_contact as NC
from conftest import CASES, SEED

pytestmark = pytest.mark.gpu

TOL = 1e-9


def radius(robot):
    return float(np.linalg.norm(np.asarray(robot).reshape(-1, 3), axis=1).max())


def scale(obst, robot, poses):
    """S of the accuracy rule, per pose"""
    p = np.asarray(poses, dtype=np.float64)
    return np.maximum(max(1.0, float(np.abs(obst).max())), np.linalg.norm(p[:, :3], axis=1) + radius(robot))


def check_rules(d, pts, dref, md, S):
    """the cap, accuracy and point rules of include/sffg.h for free poses with reference distances dref"""
    tol = TOL * S
    assert np.all(d > 0)
    far, near = dref >= md + tol, dref < md - tol
    assert np.all(d[far] == md), np.nonzero(d[far] != md)[0][:8]
    err = np.abs(d - dref)
    assert np.all(err[near] <= tol[near]), (np.max(err[near] / S[near]) if near.any() else 0)
    mid = ~far & ~near
    assert np.all((d[mid] == md) | (err[mid] <= tol[mid]))
    written = (d > 0) & (d < md)
    assert np.array_equal(~np.isnan(pts).any(1), written)
    assert np.all(np.isnan(pts[~written]))
    gap = np.linalg.norm(pts[written, :3] - pts[written, 3:], axis=1)
    assert np.all(np.abs(gap - d[written]) <= tol[written])


@pytest.mark.parametrize("fmt", ["f32", "f64"])
@pytest.mark.parametrize("case", ["B", "D", "T", "2D", "2Dd"])
def test_golden_scenes(sff, meshes, gold_collision, case, fmt):
    on, rn, _ = CASES[case]
    obst, robot = meshes[on], meshes[rn]
    env = sff.Environment(obst, robot)
    poses = gold_collision[f"{case}_poses"][:1200].astype(np.float32 if fmt == "f32" else np.float64)
    hit = env.Collide(poses)
    assert 0 < hit.sum() < len(hit)
    sub = np.nonzero(hit == 0)[0][:300]
    p64 = poses[sub].astype(np.float64)
    dref, _ = DR.distance_batch(obst, robot, p64)
    S = scale(obst, robot, p64)
    rho = radius(robot)
    for md in (0.1 * rho, rho, 4 * rho, np.inf):
        d, pts = env.Distance(poses, md, points=True)
        assert d.dtype == np.float64 and pts.shape == (len(poses), 6)
        np.testing.assert_array_equal(d == 0, hit == 1)
        assert np.all(np.isnan(pts[hit == 1]))
        check_rules(d[sub], pts[sub], dref, md, S)
        np.testing.assert_array_equal(env.Distance(poses, md), d)   # the points do not change the distances


@pytest.mark.parametrize("case", ["B", "T"])
def test_points_lie_on_robot_and_soup(sff, orc, meshes, case):
    on, rn, rng = CASES[case]
    obst, robot = meshes[on], meshes[rn]
    env = sff.Environment(obst, robot)
    poses = orc.gen_poses(SEED, 777, 4000, rng).astype(np.float64)
    d, pts = env.Distance(poses, np.inf, points=True)
    free = np.nonzero(d > 0)[0][:60]
    assert len(free) == 60 and np.all(np.isfinite(d[free]))
    S = scale(obst, robot, poses[free])
    for k, i in enumerate(free):
        assert DR.point_soup_distance(pts[i, 3:], obst) <= TOL * S[k]
        assert DR.point_soup_distance(pts[i, :3], DR.place(robot, poses[i])) <= TOL * S[k]


@pytest.mark.parametrize("case", ["B", "2D"])
def test_near_contact_brackets(sff, orc, meshes, case):
    """poses a bisection left within 1e-9 of the scene scale of contact: the colliding side reports 0, the free side a
    positive distance of at most 1e-8 S"""
    mo, mr, lo, hi, axis, cols = NC.case_brackets(orc, meshes, CASES, case, SEED)
    lo, hi = lo[:300], hi[:300]
    assert len(lo) > 50
    on, rn, _ = CASES[case]
    env = sff.Environment(meshes[on], meshes[rn])
    assert np.all(env.Distance(lo) == 0)
    d = env.Distance(hi)
    S = scale(meshes[on], meshes[rn], hi)
    assert np.all(d > 0) and np.all(d <= 1e-8 * S), np.max(d / S)


def test_hierarchy_independence_and_refit(sff, meshes, gold_collision):
    on, rn, rng = CASES["B"]
    obst, robot = meshes[on], meshes[rn]
    poses = gold_collision["B_poses"]
    host = sff.Environment(obst, robot, build=sff.BUILD_HOST)
    dev = sff.Environment(obst, robot, build=sff.BUILD_DEVICE)
    for md in (radius(robot), np.inf):
        np.testing.assert_array_equal(host.Distance(poses, md), dev.Distance(poses, md))
    # the soup moved (rotated about z and shifted): refitted hierarchy against the reference on the moved soup
    c, s = np.cos(0.05), np.sin(0.05)
    Rz = np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    moved = obst @ Rz.T + [0.7, -0.4, 0.3]
    dev.refit_obstacles(moved)
    p = poses[:600].astype(np.float64)
    hit = dev.Collide(p)
    d, pts = dev.Distance(p, np.inf, points=True)
    np.testing.assert_array_equal(d == 0, hit == 1)
    sub = np.nonzero(hit == 0)[0][:200]
    dref, _ = DR.distance_batch(moved, robot, p[sub])
    check_rules(d[sub], pts[sub], dref, np.inf, scale(moved, robot, p[sub]))


def test_device_form_and_chunking(sff, meshes):
    import torch
    on, rn, rng = CASES["B"]
    obst, robot = meshes[on], meshes[rn]
    env = sff.Environment(obst, robot)
    md = 4 * radius(robot)
    n = 1 << 20
    poses = sff.gen_poses_device(SEED, 0, n, rng)
    host_poses = poses.cpu().numpy()
    d, pts = env.Distance(host_poses, md, points=True)
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    dpts = torch.empty((n, 6), dtype=torch.float64, device="cuda")
    env.distance_device(poses, md, out=out, points=dpts)
    env.sync_check()
    np.testing.assert_array_equal(out.cpu().numpy(), d)
    np.testing.assert_array_equal(dpts.cpu().numpy(), pts)
    d64 = env.distance_device(poses.double(), md)
    env.sync_check()
    assert d64.dtype == torch.float64 and d64.shape == (n,)
    parts = [env.Distance(host_poses[a:a + 300007], md) for a in range(0, n, 300007)]
    np.testing.assert_array_equal(np.concatenate(parts), d)
    small = [env.Distance(host_poses[a:a + b], md) for a, b in ((0, 1), (1, 31), (32, 33), (65, 4096))]
    np.testing.assert_array_equal(np.concatenate(small), d[:4161])
    assert 0 < (d == 0).mean() < 0.5 and 0 < (d == md).mean() < 1


def test_edge_cases_and_errors(sff, meshes):
    import ctypes as C
    obst, robot = meshes["triang_s10"], meshes["robot_cyl_small_s10"]
    env = sff.Environment(obst, robot)
    d, pts = env.Distance(np.zeros((0, 6), dtype=np.float32), 1.0, points=True)
    assert d.shape == (0,) and pts.shape == (0, 6)
    empty = sff.Environment(np.zeros((0, 3, 3)), robot)
    p = np.random.RandomState(0).uniform(-50, 50, (100, 6))
    for md in (2.5, np.inf):
        d, pts = empty.Distance(p, md, points=True)
        assert np.all(d == md) and np.all(np.isnan(pts))
    for bad in (0.0, -1.0, np.nan):
        with pytest.raises(sff.SffgError) as ei:
            env.Distance(p, bad)
        assert ei.value.code == 3
    L = sff._lib.load()
    out = np.empty(100)
    assert L.sffg_distance_poses(env._h, None, 1, 100, 1.0, out.ctypes.data, None) == 3
    assert L.sffg_distance_poses(env._h, p.ctypes.data, 1, 100, 1.0, None, None) == 3
    assert L.sffg_distance_poses(None, p.ctypes.data, 1, 100, 1.0, out.ctypes.data, None) == 3
    assert L.sffg_distance_poses_device(env._h, None, 1, 100, 1.0, C.c_void_p(16), None, None) == 3
    assert L.sffg_distance_poses_device(env._h, p.ctypes.data, 1, -1, 1.0, out.ctypes.data, None, None) == 3
