"""GPU tests of the contact-witness probe of phase B (each clearance-grid cell keeps the two triangles that mark it nearest
its centre, and a pose past the grid tries them before the hierarchy walk): every verdict with the probe equals the
verdict without it (SFFG_WITNESS=0), without the grid (SFFG_CLEARANCE_GRID=0) and the CPU oracle, for the bench stream,
near-contact poses in every input format, other scenes, edges and a refit; and the probe saves most of the walk."""
import numpy as np
import pytest

from conftest import CASES, SEED
from near_contact import boundary_brackets, seed_poses

pytestmark = pytest.mark.gpu

OFFSETS = (1e-2, 1e-3, 1e-4, 1e-6)


@pytest.fixture
def three_envs(sff, monkeypatch):
    """-> make(obst, robot) = (probe, no probe, no grid)"""
    def make(obst, robot):
        env = sff.Environment(obst, robot)
        with monkeypatch.context() as mp:
            mp.setenv("SFFG_WITNESS", "0")
            off = sff.Environment(obst, robot)
        with monkeypatch.context() as mp:
            mp.setenv("SFFG_CLEARANCE_GRID", "0")
            plain = sff.Environment(obst, robot)
        assert env.info["grid_cells"] > 0 and plain.info["grid_cells"] == 0
        # the witnesses are there (8 bytes per cell) only in the first
        assert env.info["device_bytes"] - off.info["device_bytes"] == 8 * env.info["grid_cells"]
        return env, off, plain
    return make


def check_formats(orc, envs, obst, robot, poses, formats=("f32", "f64", "matrix")):
    """every environment gives the oracle's verdicts in every requested input format"""
    mo, mr = orc.ObbModel(obst), orc.ObbModel(robot)
    want64 = None
    for fmt in formats:
        if fmt == "f32":
            p = poses.astype(np.float32)
            want, _ = orc.collide_obbtree(mo, mr, p.astype(np.float64))
            got = [e.Collide(p) for e in envs]
        else:
            if want64 is None:
                want64, _ = orc.collide_obbtree(mo, mr, poses)
            want = want64
            if fmt == "f64":
                got = [e.Collide(poses) for e in envs]
            else:
                R = np.stack([orc.rotation(q) for q in poses])
                got = [e.CollideTransforms(R, poses[:, :3]) for e in envs]
        for g in got:
            bad = np.nonzero(g != want)[0]
            assert len(bad) == 0, (fmt, len(bad), poses[bad[:4]])
    return want64


def test_bench_stream_slice(sff, orc, meshes, three_envs):
    on, rn, rng = CASES["B"]
    poses = orc.gen_poses(SEED, 0, 1 << 20, rng)
    envs = three_envs(meshes[on], meshes[rn])
    want, _ = orc.collide_obbtree(orc.ObbModel(meshes[on]), orc.ObbModel(meshes[rn]), poses.astype(np.float64))
    for e in envs:
        np.testing.assert_array_equal(e.Collide(poses), want)
    assert 0.05 < want.mean() < 0.2


@pytest.mark.parametrize("axis", [0, 2])   # walls / floors
def test_near_contact_poses(sff, orc, meshes, three_envs, axis):
    obst, rob = meshes["building_s10"], meshes["robot_small_s10"]
    envs = three_envs(obst, rob)
    lo, hi = boundary_brackets(orc, orc.ObbModel(obst), orc.ObbModel(rob), SEED + 41 + axis, 40000, CASES["B"][2], 0.5, axis=axis)
    assert len(lo) > 100
    parts = []
    for off in OFFSETS:
        a, b = lo.copy(), hi.copy()
        a[:, axis] -= off
        b[:, axis] += off
        parts += [a, b]
    want = check_formats(orc, envs, obst, rob, np.concatenate(parts))
    assert 0.2 < want.mean() < 0.8


@pytest.mark.parametrize("case", ["D", "2D"])   # dense3d_s1, the 2-D map
def test_other_scenes(sff, orc, meshes, three_envs, case):
    on, rn, rng = CASES[case]
    obst, rob = meshes[on], meshes[rn]
    envs = three_envs(obst, rob)
    poses = seed_poses(orc, obst, SEED + 3, 200000, rng)
    want = check_formats(orc, envs, obst, rob, poses, ("f32", "f64") if rng is not None else ("f64",))
    assert want.sum() > 0


@pytest.mark.parametrize("rot_mode", [0, 1])
def test_edges_first_hit(sff, orc, meshes, three_envs, rot_mode):
    on, rn, rng = CASES["B"]
    obst, rob = meshes[on], meshes[rn]
    env, off, _ = three_envs(obst, rob)
    s = orc.gen_poses(SEED + 5, 0, 4096, rng).astype(np.float64)
    r = np.random.RandomState(SEED + rot_mode)
    e = s + np.concatenate([r.uniform(-4, 4, (len(s), 3)), r.uniform(-0.5, 0.5, (len(s), 3))], 1)
    free, first = env.isPathFree(s, e, 0.1, rot_mode, want_first_hit=True)
    pf, pfirst = off.isPathFree(s, e, 0.1, rot_mode, want_first_hit=True)
    wf, wh, _ = orc.edges_free(obst, rob, s, e, 0.1, rot_mode)
    np.testing.assert_array_equal(free, pf)
    np.testing.assert_array_equal(first, pfirst)
    np.testing.assert_array_equal(free, wf)
    np.testing.assert_array_equal(first, wh)
    assert 0 < free.mean() < 1


def test_refit_rebuilds_the_witnesses(sff, orc, meshes, three_envs):
    on, rn, rng = CASES["B"]
    obst, rob = meshes[on], meshes[rn]
    shift = np.array([0.37, -0.21, 0.5])
    moved = (obst.reshape(-1, 3) + shift).reshape(obst.shape)
    envs = three_envs(obst, rob)
    for e in envs:
        e.refit_obstacles(moved)
    poses = orc.gen_poses(SEED + 9, 0, 200000, rng).astype(np.float64)
    check_formats(orc, envs, moved, rob, poses, ("f64",))


# Walk steps per pose past the grid with the probe over the same without it, on the bench stream: 0.114 measured on a
# B200 over 2^24 poses (3.36 -> 0.38 steps), close to the CPU estimate (89 % of the colliding poses touch their cell's
# nearest triangle).  0.2 leaves room for the sampling of a smaller slice and fails if the probe stops settling contacts.
MAX_STEPS_RATIO = 0.2


def test_probe_skips_most_of_the_walk(sff, orc, meshes, three_envs):
    on, rn, rng = CASES["B"]
    poses = orc.gen_poses(SEED, 1 << 20, 1 << 19, rng)
    env, off, _ = three_envs(meshes[on], meshes[rn])
    per_pose = []
    verdicts = []
    for e in (env, off):
        e.enable_counters(True)
        verdicts.append(e.Collide(poses))
        c = e.read_counters()
        assert c["poses_past_grid"] == c["poses_past_root"] > 0
        per_pose.append(c["traversal_steps"] / c["poses_past_grid"])
    np.testing.assert_array_equal(verdicts[0], verdicts[1])
    assert per_pose[0] <= MAX_STEPS_RATIO * per_pose[1], per_pose


# (grid_cells, grid_cell_size, device_bytes) of the bench environment and of the 2-D map under each switch setting, as
# reported by the build before the grid's sizing moved into clearance_grid.cu: no test fixed the sizing before that.
GRID_SIZING = {
    ("B", None): (2798432, 0.6927118897438049, 39352620),
    ("B", "SFFG_WITNESS"): (2798432, 0.6927118897438049, 16965164),
    ("B", "SFFG_CLEARANCE_GRID"): (0, 0.0, 5421632),
    ("2D", None): (8632224, 0.4128884789622589, 104695876),
    ("2D", "SFFG_WITNESS"): (8632224, 0.4128884789622589, 35638084),
    ("2D", "SFFG_CLEARANCE_GRID"): (0, 0.0, 30160),
}


@pytest.mark.parametrize("case,switch", list(GRID_SIZING))
def test_grid_sizing(sff, meshes, monkeypatch, case, switch):
    on, rn, _ = CASES[case]
    if switch:
        monkeypatch.setenv(switch, "0")
    info = sff.Environment(meshes[on], meshes[rn]).info
    assert (info["grid_cells"], info["grid_cell_size"], info["device_bytes"]) == GRID_SIZING[case, switch]
