"""GPU parity tests of the local planner (isPathFree) through sffg_check_edges."""
import numpy as np
import pytest

from conftest import CASES, SEED

pytestmark = pytest.mark.gpu


def test_edges_golden_building(sff, meshes, gold_edges):
    env = sff.Environment(meshes["building_s10"], meshes["robot_small_s10"])
    s, e = gold_edges["B_starts"], gold_edges["B_ends"]
    for mode in (0, 1):
        free, first = env.isPathFree(s, e, 0.1, mode, want_first_hit=True)
        np.testing.assert_array_equal(free, gold_edges[f"B_free_m{mode}"])
        np.testing.assert_array_equal(first, gold_edges[f"B_first_m{mode}"])


def test_edges_golden_2d_long(sff, meshes, gold_edges):
    env = sff.Environment(meshes["triangles_tri"], meshes["robot_small_s1"])
    free, first = env.isPathFree(gold_edges["2D_starts"], gold_edges["2D_ends"], 0.1, 0, want_first_hit=True)
    np.testing.assert_array_equal(free, gold_edges["2D_free_m0"])
    np.testing.assert_array_equal(first, gold_edges["2D_first_m0"])


def test_edges_seeded_vs_oracle_and_properties(sff, orc, meshes):
    ob, rb = meshes["building_s10"], meshes["robot_small_s10"]
    env = sff.Environment(ob, rb)
    m = 20000
    r = np.random.RandomState(1)
    s = orc.gen_poses(SEED + 5, 0, m, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
    d = r.normal(size=(m, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    e = s.copy()
    e[:, :3] += 4.0 * d
    free, first = env.isPathFree(s, e, 0.1, 0, want_first_hit=True)
    wf, wh, _ = orc.edges_free(ob, rb, s, e, 0.1, 0, models=(orc.ObbModel(ob), orc.ObbModel(rb)))
    np.testing.assert_array_equal(free, wf)
    np.testing.assert_array_equal(first, wh)
    assert np.all((first == 0) == (free == 1))
    # the sample at first_hit really collides and (reference mode) carries identity rotation
    hit = np.nonzero(first > 0)[0][:2000]
    parts = np.array([orc.distance6(s[i], e[i]) for i in hit]) / 0.1
    pos = np.zeros((len(hit), 6))
    pos[:, :3] = s[hit, :3] + (first[hit, None] * (e[hit, :3] - s[hit, :3])) / parts[:, None]
    assert env.Collide(pos).all()
    # opt-in interpolate mode: the rotation varies along the edge (the group's swept box is the cube around the robot's
    # bounding sphere), start and end orientations unrelated
    k = 4000
    e1 = e[:k].copy()
    e1[:, 3:] = orc.gen_poses(SEED + 6, 0, k, [-45, 45, -45, 45, 0, 125]).astype(np.float64)[:, 3:]
    free1, first1 = env.isPathFree(s[:k], e1, 0.1, 1, want_first_hit=True)
    wf1, wh1, _ = orc.edges_free(ob, rb, s[:k], e1, 0.1, 1, models=(orc.ObbModel(ob), orc.ObbModel(rb)))
    np.testing.assert_array_equal(free1, wf1)
    np.testing.assert_array_equal(first1, wh1)
    assert 0.05 < free1.mean() < 0.95
    # a free edge stays free when shortened from the far end at the same sampling phase (prefix property)
    assert env.isPathFree(s[:0], e[:0]).shape == (0,)


def test_edge_sample_counts_match_reference_loop(sff, orc, meshes):
    """an obstacle placed only at the LAST sample index tells whether the kernel visits exactly index < parts"""
    rob = meshes["robot_small_s1"]
    wall = np.array([[[3.9, -5, -5], [3.9, 5, -5], [3.9, 0, 5]]], dtype=np.float64)   # plane x = 3.9
    env = sff.Environment(wall, rob)
    s = np.zeros((4, 6))
    e = np.zeros((4, 6))
    e[:, 0] = [4.0, 3.7, 3.6, 0.05]     # 39 samples reach x=3.9 (hit: robot half width .247); 3.7 -> last sample 3.6 (hit at 3.653+.247)
    free, first = env.isPathFree(s, e, 0.1, 0, want_first_hit=True)
    wf, wh, _ = orc.edges_free(wall, rob, s, e, 0.1, 0)
    np.testing.assert_array_equal(free, wf)
    np.testing.assert_array_equal(first, wh)


def test_check_moves_is_collide_or_not_path_free(sff, orc, meshes):
    """sffg_check_moves: `env.Collide(newPoint) || !isPathFree(node, newPoint)` rejects (src/forest.h:246, src/rrt.h:149):
    planner-sized and large batches against the oracle, and against the two separate engine calls"""
    on, rn, rng = CASES["B"]
    env = sff.Environment(meshes[on], meshes[rn])
    mo, mr = orc.ObbModel(meshes[on]), orc.ObbModel(meshes[rn])
    for m in (1, 640, 70000):
        s = orc.gen_poses(SEED + 21, 0, m, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
        d = np.random.RandomState(m).randn(m, 3)
        e = orc.gen_poses(SEED + 22, 0, m, rng).astype(np.float64)
        e[:, :3] = s[:, :3] + 4.0 * d / np.linalg.norm(d, axis=1, keepdims=True)
        ok = env.checkMoves(s, e)
        hit, _ = orc.collide_obbtree(mo, mr, e)
        free, _, _ = orc.edges_free(meshes[on], meshes[rn], s, e, 0.1, 0, models=(mo, mr))
        np.testing.assert_array_equal(ok, (free.astype(bool) & ~hit.astype(bool)).astype(np.uint8))
        np.testing.assert_array_equal(ok, (env.isPathFree(s, e).astype(bool) & ~env.Collide(e).astype(bool)).astype(np.uint8))
    assert len(env.checkMoves(np.zeros((0, 6)), np.zeros((0, 6)))) == 0
    env.close()


def tube_soup(r):
    """~32 000 tiny triangles, cleared only from tubes of radius 0.5 around nine parallel lines along (1, 1, 1), and 27
    edges of length 5 * sqrt(3) per copy: along the tubes (free), half-way between them and out of the tubes into the soup"""
    u = np.ones(3) / np.sqrt(3)
    lines = np.array([(x, y, 0.0) for x in (-1.5, 0.0, 1.5) for y in (-1.5, 0.0, 1.5)])
    c = r.uniform(-2.5, 7.5, (36000, 3))
    rel = c[:, None, :] - lines[None]
    c = c[np.linalg.norm(rel - (rel @ u)[..., None] * u, axis=2).min(1) > 0.5]
    soup = c[:, None, :] + r.uniform(-0.02, 0.02, (len(c), 3, 3))
    copies = 256
    s = np.zeros((copies, 27, 6))
    s[..., :3] = np.concatenate([lines + 0.5, lines + [1.25, 1.25, 0.5], lines + 0.5])[None] + r.uniform(0, 0.5, (copies, 1, 1))
    e = s.copy()
    e[:, :18, :3] += 5.0
    e[:, 18:, :3] += [5.0, 5.0, 2.0]
    s[..., 3:] = e[..., 3:] = r.uniform(-np.pi, np.pi, (copies, 27, 3))   # constant angles: samples 0.1 apart in position
    return soup, s.reshape(-1, 6), e.reshape(-1, 6)


def test_edges_through_a_soup_that_overflows_the_swept_box_list(sff, orc, meshes):
    """the swept box of a 32-sample group holds more leaf triangles than its candidate list (192), so the kernel falls back
    to the per-sample walk for those groups; 6 912 edges so that each edge runs on one warp (a warp's share of a split
    edge is too short to overflow the list)"""
    rob = meshes["robot_small_s1"]   # a 0.5 x 0.5 plate: bounding radius 0.35 < tube radius 0.5
    soup, s, e = tube_soup(np.random.RandomState(5))
    env = sff.Environment(soup, rob)
    mo, mr = orc.ObbModel(soup), orc.ObbModel(rob)
    for mode in (sff.ROT_REFERENCE, sff.ROT_INTERPOLATE):
        free, first = env.isPathFree(s, e, 0.1, mode, want_first_hit=True)
        wf, wh, _ = orc.edges_free(soup, rob, s, e, 0.1, mode, models=(mo, mr))
        np.testing.assert_array_equal(free, wf)
        np.testing.assert_array_equal(first, wh)
        wf = wf.reshape(-1, 27)
        assert wf[:, :9].all() and wf[:, 9:].mean() < 0.1 and (wh > 32).sum() > 100
    env.close()
