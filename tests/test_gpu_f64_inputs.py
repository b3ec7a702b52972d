"""GPU tests of the double-precision pose and edge entry points with angles float32 cannot hold.

Poses sit 1e-3 .. 1e-5 inside or outside a contact (tests/near_contact.py) with 2*pi*K added to their angles, K up to
1600 (|a| ~ 1e4 rad), plus a few at +-1e6 and +-1e12.  Every comparison is exact equality with the CPU oracle at the
double pose itself: no tolerance, no allowed exceptions.  Failures list the pose indices and the oracle's margins."""
import numpy as np
import pytest

import near_contact as NC
from conftest import CASES, SEED

pytestmark = pytest.mark.gpu

KS = (0, 1, 2, 16, 160, 1600)
OFFSETS = (1e-3, 1e-4, 1e-5)


@pytest.fixture(scope="module")
def brackets():
    """near_contact.case_brackets per scene, computed on first use"""
    return {}


def scene(orc, meshes, brackets, case):
    if case not in brackets:
        brackets[case] = NC.case_brackets(orc, meshes, CASES, case, SEED + 50)
    return brackets[case]


def pose_batch(lo, hi, axis, cols, seed=0):
    """every (K, off) band of near-contact poses, then poses at +-1e6 and +-1e12 rad -> (poses, band label per pose)"""
    parts, labels = [], []
    for K in KS:
        for off in OFFSETS:
            inside, outside = NC.near_contact_poses(lo, hi, off, K, seed + 100 * K + int(-np.log10(off)), axis, cols)
            parts += [inside, outside]
            labels += [f"K={K} off={off:g} inside"] * len(inside) + [f"K={K} off={off:g} outside"] * len(outside)
    r = np.random.RandomState(seed + 1)
    for mag in (1e6, 1e12):
        p = np.concatenate([lo[:64], hi[:64]]).copy()
        p[:, list(cols)] = r.uniform(0.5, 1.0, (len(p), len(cols))) * mag * r.choice([-1.0, 1.0], (len(p), len(cols)))
        parts.append(p)
        labels += [f"|a|~{mag:g}"] * len(p)
    return np.ascontiguousarray(np.concatenate(parts)), np.array(labels)


def report(orc, meshes, case, poses, labels, got, want):
    bad = np.nonzero(got != want)[0]
    if len(bad) == 0:
        return ""
    on, rn, _ = CASES[case]
    bands = {b: int((labels[bad] == b).sum()) for b in dict.fromkeys(labels[bad])}
    return (f"{case}: {len(bad)} of {len(poses)} verdicts differ; per band {bands}; poses {bad[:8]}, got {got[bad[:8]]}, "
            f"oracle {want[bad[:8]]}, oracle margins {orc.pose_margin(meshes[on], meshes[rn], poses[bad[:8]])}")


@pytest.mark.parametrize("build", ["host", "device"])
@pytest.mark.parametrize("case", list(NC.SETUP))
def test_pose_verdicts_with_double_angles(sff, orc, meshes, brackets, case, build):
    """sffg_collide_poses_f64 (Environment.Collide on float64) and sffg_collide_poses_device on a float64 tensor"""
    import torch
    mo, mr, lo, hi, axis, cols = scene(orc, meshes, brackets, case)
    on, rn, _ = CASES[case]
    env = sff.Environment(meshes[on], meshes[rn], build=sff.BUILD_HOST if build == "host" else sff.BUILD_DEVICE)
    poses, labels = pose_batch(lo, hi, axis, cols)
    want, _ = orc.collide_obbtree(mo, mr, poses)
    assert 0.3 < want.mean() < 0.7
    got = env.Collide(poses)
    assert not report(orc, meshes, case, poses, labels, got, want), report(orc, meshes, case, poses, labels, got, want)
    d = env.collide_device(torch.from_numpy(poses).cuda())
    torch.cuda.synchronize()
    env.sync_check()
    got_d = d.cpu().numpy()
    assert not report(orc, meshes, case, poses, labels, got_d, want), report(orc, meshes, case, poses, labels, got_d, want)
    env.close()


@pytest.mark.parametrize("case", list(NC.SETUP))
def test_check_moves_zero_length_is_the_end_pose_verdict(sff, orc, meshes, brackets, case):
    """sffg_check_moves with start == end (what the planner hosts call per expansion step): no samples, so ok = 1 - the
    oracle's verdict at the end pose; one large call and planner-sized calls (the fused pose + edge launch)"""
    mo, mr, lo, hi, axis, cols = scene(orc, meshes, brackets, case)
    on, rn, _ = CASES[case]
    env = sff.Environment(meshes[on], meshes[rn])
    poses, labels = pose_batch(lo, hi, axis, cols, seed=3)
    want, _ = orc.collide_obbtree(mo, mr, poses)
    for rot_mode in (sff.ROT_REFERENCE, sff.ROT_INTERPOLATE):
        ok = env.checkMoves(poses, poses, 0.1, rot_mode)
        assert not report(orc, meshes, case, poses, labels, 1 - ok, want), report(orc, meshes, case, poses, labels, 1 - ok, want)
    sel = np.random.RandomState(5).choice(len(poses), 4 * 500, replace=False)
    ok = np.concatenate([env.checkMoves(poses[sel[i:i + 500]], poses[sel[i:i + 500]]) for i in range(0, len(sel), 500)])
    got, w = 1 - ok, want[sel]
    assert not report(orc, meshes, case, poses[sel], labels[sel], got, w), report(orc, meshes, case, poses[sel], labels[sel], got, w)
    env.close()


def check_edges(orc, meshes, case, env, s, e, sample, mode, models):
    on, rn, _ = CASES[case]
    free, first = env.isPathFree(s, e, sample, mode, want_first_hit=True)
    wf, wh, _ = orc.edges_free(meshes[on], meshes[rn], s, e, sample, mode, models=models)
    bad = np.nonzero((free != wf) | (first != wh))[0]
    assert len(bad) == 0, (f"{len(bad)} of {len(s)} edges differ: {bad[:8]}, free {free[bad[:8]]} vs {wf[bad[:8]]}, "
                           f"first hit {first[bad[:8]]} vs {wh[bad[:8]]}")
    return wf, wh


@pytest.mark.parametrize("case", ["B", "T"])
def test_interpolated_edge_through_a_near_contact_pose(sff, orc, meshes, brackets, case):
    """s = q - dir/P, e = s + dir with |dir| = L and P = L / sample: sample 1 of the edge is the near-contact pose q (up to
    double rounding of the translation), carried through the FP32 stage with q's wide, non-float angles"""
    mo, mr, lo, hi, axis, cols = scene(orc, meshes, brackets, case)
    on, rn, _ = CASES[case]
    env = sff.Environment(meshes[on], meshes[rn])
    r = np.random.RandomState(11)
    qs = []
    for K in (16, 160, 1600):
        for off in (1e-4, 1e-5):
            qs += list(NC.near_contact_poses(lo, hi, off, K, 200 + K, axis, cols))
    q = np.concatenate(qs)
    L, sample = 1.0, 0.1
    d = r.normal(size=(len(q), 3))
    d *= L / np.linalg.norm(d, axis=1, keepdims=True)
    s = q.copy()
    s[:, :3] = q[:, :3] - d * (sample / L)
    e = s.copy()
    e[:, :3] = s[:, :3] + d
    wf, wh = check_edges(orc, meshes, case, env, s, e, sample, sff.ROT_INTERPOLATE, (mo, mr))
    assert (wh == 1).sum() > len(q) // 4      # the near-contact sample decides a good share of the edges
    env.close()


def wide_edges(orc, m, seed, spread, wrap_share=0.5):
    """edges of translation length 4 in the building's free space region; start angles uniform in +-spread, end angles
    start + a difference that crosses +-pi for about `wrap_share` of the angles"""
    r = np.random.RandomState(seed)
    s = orc.gen_poses(SEED + seed, 0, m, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
    s[:, 3:] = r.uniform(-spread, spread, (m, 3))
    d = r.normal(size=(m, 3))
    e = s.copy()
    e[:, :3] += 4.0 * d / np.linalg.norm(d, axis=1, keepdims=True)
    diff = r.uniform(-0.5, 0.5, (m, 3))
    wrap = r.uniform(size=(m, 3)) < wrap_share
    diff[wrap] = r.choice([-1.0, 1.0], wrap.sum()) * r.uniform(np.pi, 2 * np.pi - 0.1, wrap.sum())
    e[:, 3:] = s[:, 3:] + diff
    return s, e


def test_edges_with_wide_and_wrapping_angles_both_modes(sff, orc, meshes):
    """sffg_check_edges: angles in +-10 and +-1000 whose differences cross +-pi (the single wrap of Point::distance), and a
    few edges between unrelated angles of +-1000 (differences of ~2000 rad, ~20 000 samples)"""
    on, rn, _ = CASES["B"]
    mo, mr = orc.ObbModel(meshes[on]), orc.ObbModel(meshes[rn])
    env = sff.Environment(meshes[on], meshes[rn])
    for spread in (10.0, 1000.0):
        s, e = wide_edges(orc, 3000, int(spread), spread)
        for mode in (sff.ROT_REFERENCE, sff.ROT_INTERPOLATE):
            wf, _ = check_edges(orc, meshes, "B", env, s, e, 0.1, mode, (mo, mr))
            assert 0.05 < wf.mean() < 0.95
    r = np.random.RandomState(2)
    s, e = wide_edges(orc, 24, 9, 1000.0)
    e[:, 3:] = r.uniform(-1000, 1000, (24, 3))
    assert min(orc.edge_num_samples(s[i], e[i]) for i in range(24)) > 1000
    for mode in (sff.ROT_REFERENCE, sff.ROT_INTERPOLATE):
        check_edges(orc, meshes, "B", env, s, e, 0.1, mode, (mo, mr))
    env.close()


@pytest.mark.parametrize("m", [1, 7, 600, 9000])
def test_check_edges_device_matches_host_and_oracle(sff, orc, meshes, m):
    """sffg_check_edges_device: m < 8192 shares an edge among several warps (scratch word + finalize_edges_kernel),
    m >= 8192 runs one warp per edge"""
    import torch
    on, rn, _ = CASES["B"]
    mo, mr = orc.ObbModel(meshes[on]), orc.ObbModel(meshes[rn])
    env = sff.Environment(meshes[on], meshes[rn])
    s, e = wide_edges(orc, m, 30 + m, 1000.0)
    for mode in (sff.ROT_REFERENCE, sff.ROT_INTERPOLATE):
        wf, wh = check_edges(orc, meshes, "B", env, s, e, 0.1, mode, (mo, mr))
        ds, de = torch.from_numpy(s).cuda(), torch.from_numpy(e).cuda()
        first = torch.full((m,), -7, dtype=torch.int32, device="cuda")
        free = env.edges_device(ds, de, 0.1, mode, first_hit_out=first)
        torch.cuda.synchronize()
        env.sync_check()
        np.testing.assert_array_equal(free.cpu().numpy(), wf)
        np.testing.assert_array_equal(first.cpu().numpy(), wh)
    env.close()


def test_first_hit_is_the_minimum_over_warps(sff, orc, meshes):
    """parallel walls every 10 units along x and edges of 400 .. 4000 samples along x: with 1, 3 or 16 edges each edge is
    split over many warps and several warps' ranges hold colliding samples; first_hit must be the first wall's sample"""
    rob = meshes["robot_small_s1"]
    xs = 3.93 + 10.0 * np.arange(40)
    walls = np.array([[[x, -50, -50], [x, 50, -50], [x, 0, 50]] for x in xs], dtype=np.float64)
    env = sff.Environment(walls, rob)
    mo, mr = orc.ObbModel(walls), orc.ObbModel(rob)
    r = np.random.RandomState(8)
    for m in (1, 3, 16):
        s = np.zeros((m, 6))
        s[:, 1:3] = r.uniform(-5, 5, (m, 2))
        s[:, 0] = r.uniform(-2, 2, m)
        e = s.copy()
        e[:, 0] += r.uniform(40, 399, m)
        free, first = env.isPathFree(s, e, 0.1, sff.ROT_REFERENCE, want_first_hit=True)
        wf, wh, _ = orc.edges_free(walls, rob, s, e, 0.1, 0, models=(mo, mr))
        np.testing.assert_array_equal(free, wf)
        np.testing.assert_array_equal(first, wh)
        # every edge is blocked, first by the wall at xs[0]: its sample lies within a robot width before that wall
        assert not wf.any()
        x_hit = s[:, 0] + 0.1 * first
        assert np.all((x_hit > xs[0] - 1.0) & (x_hit < xs[0])), x_hit
    env.close()


@pytest.mark.parametrize("sample", [0.05, 0.25, 1.0])
def test_edges_at_other_sample_distances(sff, orc, meshes, sample):
    on, rn, _ = CASES["B"]
    mo, mr = orc.ObbModel(meshes[on]), orc.ObbModel(meshes[rn])
    env = sff.Environment(meshes[on], meshes[rn])
    s, e = wide_edges(orc, 2000, 60, 10.0)
    for mode in (sff.ROT_REFERENCE, sff.ROT_INTERPOLATE):
        wf, _ = check_edges(orc, meshes, "B", env, s, e, sample, mode, (mo, mr))
        assert 0.05 < wf.mean() < 0.95
    env.close()
