"""GPU tests of the clearance grid's per-cell separating plane (phase A of the pose and edge kernels): every verdict
equals the CPU oracle and the verdict of an environment without the grid (SFFG_CLEARANCE_GRID=0), at poses that graze the
plane, in cells where no plane may clear the pose, after a refit, and in the edge kernel."""
import numpy as np
import pytest

from conftest import CASES, SEED
from near_contact import boundary_brackets

pytestmark = pytest.mark.gpu

OFFSETS = (1e-2, 3e-3, 1e-3, 1e-4, 1e-5, 1e-6)   # the plane test's margin is about 1.3e-3 on building_s10


def grid_and_plain(sff, obst, robot, monkeypatch):
    env = sff.Environment(obst, robot)
    assert env.info["grid_cells"] > 0
    with monkeypatch.context() as mp:
        mp.setenv("SFFG_CLEARANCE_GRID", "0")
        plain = sff.Environment(obst, robot)
    assert plain.info["grid_cells"] == 0
    return env, plain


def check_all_inputs(orc, env, plain, obst, robot, poses):
    """float32, float64 and matrix input: grid == no grid == oracle, exactly"""
    mo, mr = orc.ObbModel(obst), orc.ObbModel(robot)
    p32 = poses.astype(np.float32)
    want32, _ = orc.collide_obbtree(mo, mr, p32.astype(np.float64))
    want64, _ = orc.collide_obbtree(mo, mr, poses)
    for p, want in ((p32, want32), (poses, want64)):
        got = env.Collide(p)
        np.testing.assert_array_equal(got, plain.Collide(p))
        bad = np.nonzero(got != want)[0]
        assert len(bad) == 0, (p.dtype, len(bad), p[bad[:4]])
    R = np.stack([orc.rotation(q) for q in poses])
    got = env.CollideTransforms(R, poses[:, :3])
    np.testing.assert_array_equal(got, plain.CollideTransforms(R, poses[:, :3]))
    np.testing.assert_array_equal(got, want64)
    return want64


def near_contact(orc, obst, robot, seed, axis):
    """poses 1e-2 .. 1e-6 inside and outside a contact found by bisection along `axis`"""
    lo, hi = boundary_brackets(orc, orc.ObbModel(obst), orc.ObbModel(robot), seed, 40000, CASES["B"][2], 0.5, axis=axis)
    assert len(lo) > 100
    out = []
    for off in OFFSETS:
        a, b = lo.copy(), hi.copy()
        a[:, axis] -= off
        b[:, axis] += off
        out += [a, b]
    return np.concatenate(out)


@pytest.mark.parametrize("robot", ["robot_small_s10", "robot_cyl_small_s10"])   # 8 distinct vertices / 64: the box
@pytest.mark.parametrize("axis", [0, 2])                                       # against walls / floors
def test_near_contact_poses_at_the_walls(sff, orc, meshes, monkeypatch, robot, axis):
    obst, rob = meshes["building_s10"], meshes[robot]
    env, plain = grid_and_plain(sff, obst, rob, monkeypatch)
    poses = near_contact(orc, obst, rob, SEED + 7 + axis, axis)
    want = check_all_inputs(orc, env, plain, obst, rob, poses)
    assert 0.2 < want.mean() < 0.8


def quad(p0, p1, p2, p3):
    return np.array([[*p0, *p1, *p2], [*p0, *p2, *p3]], dtype=np.float64)


def box_faces(lo, hi):
    x0, y0, z0 = lo
    x1, y1, z1 = hi
    return np.concatenate([
        quad((x0, y0, z0), (x1, y0, z0), (x1, y1, z0), (x0, y1, z0)), quad((x0, y0, z1), (x1, y0, z1), (x1, y1, z1), (x0, y1, z1)),
        quad((x0, y0, z0), (x1, y0, z0), (x1, y0, z1), (x0, y0, z1)), quad((x0, y1, z0), (x1, y1, z0), (x1, y1, z1), (x0, y1, z1)),
        quad((x0, y0, z0), (x0, y1, z0), (x0, y1, z1), (x0, y0, z1)), quad((x1, y0, z0), (x1, y1, z0), (x1, y1, z1), (x1, y0, z1))])


def uniform_poses(seed, n, lo, hi):
    r = np.random.RandomState(seed)
    return np.concatenate([r.uniform(lo, hi, (n, 3)), r.uniform(-np.pi, np.pi, (n, 3))], 1)


# synthetic soups for robot_small_s10 (bounding radius 2.77, 0.13 thick):
#  corner  floor and two walls meeting in a corner: cells near the corner have geometry within reach on two or three sides
#  slot    two parallel plates 0.6 apart: a robot between them has obstacles within reach on both sides
#  cell    the six faces of a cube of half-size 3 about the origin: every direction's bound lies below the cells inside,
#          so their best plane leaves no room (the no-plane record); the robot turns freely at the centre only
SOUPS = {
    "corner": (lambda: np.concatenate([quad((0, 0, 0), (20, 0, 0), (20, 20, 0), (0, 20, 0)), quad((0, 0, 0), (0, 20, 0), (0, 20, 20), (0, 0, 20)),
                                       quad((0, 0, 0), (20, 0, 0), (20, 0, 20), (0, 0, 20))]), (-1.0, -1.0, -1.0), (4.0, 4.0, 4.0)),
    "slot": (lambda: np.concatenate([quad((-10, -10, 0), (10, -10, 0), (10, 10, 0), (-10, 10, 0)),
                                     quad((-10, -10, 0.6), (10, -10, 0.6), (10, 10, 0.6), (-10, 10, 0.6))]), (-4.0, -4.0, -0.5), (4.0, 4.0, 1.1)),
    "cell": (lambda: box_faces((-3, -3, -3), (3, 3, 3)), (-1.0, -1.0, -1.0), (1.0, 1.0, 1.0)),
}


@pytest.mark.parametrize("soup", sorted(SOUPS))
def test_cells_where_a_plane_must_not_clear_the_pose(sff, orc, meshes, monkeypatch, soup):
    make, lo, hi = SOUPS[soup]
    obst, rob = make(), meshes["robot_small_s10"]
    env, plain = grid_and_plain(sff, obst, rob, monkeypatch)
    poses = uniform_poses(SEED + len(soup), 60000, lo, hi)
    want = check_all_inputs(orc, env, plain, obst, rob, poses)
    assert 0.05 < want.mean() < 0.999


def test_refit_rebuilds_the_planes(sff, orc, meshes, monkeypatch):
    obst, rob = meshes["building_s10"], meshes["robot_small_s10"]
    poses = near_contact(orc, obst, rob, SEED + 21, 0)
    shift = np.array([0.37, -0.21, 0.5])
    moved = (obst.reshape(-1, 3) + shift).reshape(obst.shape)
    env, plain = grid_and_plain(sff, obst, rob, monkeypatch)
    env.refit_obstacles(moved)
    plain.refit_obstacles(moved)
    moved_poses = poses.copy()
    moved_poses[:, :3] += shift
    # both the poses that follow the walls and the old poses, which the moved walls now leave free or cut
    check_all_inputs(orc, env, plain, moved, rob, np.concatenate([moved_poses, poses]))


@pytest.mark.parametrize("rot_mode", [0, 1])
def test_edges_near_the_walls(sff, orc, meshes, monkeypatch, rot_mode):
    """edge samples see the plane too: free flags and first hits equal the oracle and the grid-less environment"""
    obst, rob = meshes["building_s10"], meshes["robot_small_s10"]
    env, plain = grid_and_plain(sff, obst, rob, monkeypatch)
    s = near_contact(orc, obst, rob, SEED + 31, 2)[::4]
    e = s.copy()
    e[:, 0] += 1.5
    e[:, 3:] += 0.4
    free, first = env.isPathFree(s, e, 0.1, rot_mode, want_first_hit=True)
    pf, pfirst = plain.isPathFree(s, e, 0.1, rot_mode, want_first_hit=True)
    wf, wh, _ = orc.edges_free(obst, rob, s, e, 0.1, rot_mode)
    np.testing.assert_array_equal(free, pf)
    np.testing.assert_array_equal(first, pfirst)
    np.testing.assert_array_equal(free, wf)
    np.testing.assert_array_equal(first, wh)


# poses_past_grid - colliding poses on the sweep below with the library before the planes existed
PARENT_NEAR_MISSES_PAST_GRID = 19608   # (1 948 with the planes)


def test_planes_cut_the_near_misses_that_reach_the_traversal(sff, orc, meshes):
    """seeded bench-shape sweep of case B: fewer free poses reach phase B than with the clear bit alone"""
    on, rn, rng = CASES["B"]
    n = 400000
    poses = orc.gen_poses(SEED, 12345, n, rng)
    env = sff.Environment(meshes[on], meshes[rn])
    env.enable_counters(True)
    got = env.Collide(poses)
    cnt = env.read_counters()
    want, _ = orc.collide_obbtree(orc.ObbModel(meshes[on]), orc.ObbModel(meshes[rn]), poses.astype(np.float64))
    np.testing.assert_array_equal(got, want)
    near_misses = cnt["poses_past_grid"] - int(want.sum())
    assert cnt["poses_past_grid"] == cnt["poses_past_root"]
    assert 0 <= near_misses < PARENT_NEAR_MISSES_PAST_GRID, near_misses
