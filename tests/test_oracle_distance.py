"""CPU checks of the reference separation distance (tests/distance_ref.py) that the GPU distance query is compared with:
closed-form triangle pairs, random pairs against an independent minimiser, and the SAT gap as a lower bound."""
import numpy as np
import pytest

import distance_ref as DR
from conftest import CASES, SEED

BASE = np.array([[0.0, 0.0, 0.0], [4.0, 0.0, 0.0], [0.0, 4.0, 0.0]])


def check_pair(P, Q, want):
    d, p, q = DR.tri_dist(P, Q)
    assert abs(d - want) <= 1e-12 * max(1.0, want), (d, want)
    assert abs(np.linalg.norm(p - q) - d) <= 1e-12
    assert DR.point_soup_distance(p, [P]) <= 1e-12 and DR.point_soup_distance(q, [Q]) <= 1e-12
    d2, _, _ = DR.tri_dist(Q, P)
    assert abs(d2 - d) <= 1e-12


def test_parallel_triangles_at_a_known_gap():
    check_pair(BASE, BASE + [0.5, 0.5, 2.5], 2.5)
    check_pair(BASE, BASE[::-1] + [1.0, 1.0, -0.75], 0.75)


def test_vertex_face():
    Q = np.array([[1.0, 1.0, 3.0], [1.0, 2.0, 9.0], [2.0, 1.0, 9.0]])   # vertex 0 above the interior of BASE
    check_pair(BASE, Q, 3.0)


def test_crossed_edges():
    P = np.array([[-2.0, 0.0, 0.0], [2.0, 0.0, 0.0], [0.0, 0.0, -5.0]])   # edge along x at z = 0, body below
    Q = np.array([[0.0, -2.0, 1.5], [0.0, 2.0, 1.5], [0.0, 0.0, 6.0]])    # edge along y at z = 1.5, body above
    check_pair(P, Q, 1.5)


def test_shared_vertex_and_offset_edges():
    Q = np.array([[4.0, 0.0, 0.0], [8.0, 0.0, 3.0], [8.0, 1.0, 3.0]])   # shares BASE's vertex 1
    check_pair(BASE, Q, 0.0)
    check_pair(BASE, Q + [3.0, 0.0, 0.0], 3.0)                          # beyond that vertex along x


def test_degenerate_triangles():
    seg = np.array([[1.0, 1.0, 2.0], [3.0, 3.0, 2.0], [2.0, 2.0, 2.0]])   # collinear, zero area, above BASE's interior
    d, _, _ = DR.tri_dist(BASE, seg)
    assert d == pytest.approx(2.0, abs=1e-12)
    pt = np.array([[6.0, 0.0, 0.0]] * 3)                                   # a point 2 beyond vertex 1
    check_pair(BASE, pt, 2.0)
    check_pair(seg, seg + [0.0, 0.0, 1.25], 1.25)                         # two parallel degenerate triangles


def _slsqp_distance(P, Q):
    from scipy.optimize import minimize

    def f(z):
        v = z[:3] @ P - z[3:] @ Q
        return float(v @ v)

    def g(z):
        v = z[:3] @ P - z[3:] @ Q
        return np.concatenate([2.0 * (P @ v), -2.0 * (Q @ v)])

    cons = [{"type": "eq", "fun": lambda z: z[:3].sum() - 1.0}, {"type": "eq", "fun": lambda z: z[3:].sum() - 1.0}]
    best = np.inf
    for z0 in (np.full(6, 1.0 / 3.0), np.array([1.0, 0, 0, 1.0, 0, 0]), np.array([0, 1.0, 0, 0, 0, 1.0])):
        r = minimize(f, z0, jac=g, bounds=[(0.0, 1.0)] * 6, constraints=cons, method="SLSQP",
                     options={"ftol": 1e-16, "maxiter": 500})
        best = min(best, f(np.clip(r.x, 0, 1)))
    return np.sqrt(max(best, 0.0))


def test_random_pairs_against_slsqp(orc):
    r = np.random.RandomState(7)
    n_checked = 0
    while n_checked < 200:
        P = r.uniform(-1, 1, (3, 3))
        Q = r.uniform(-1, 1, (3, 3)) + r.uniform(-1.5, 1.5, 3)
        if orc.tri_contact(P, Q):
            continue
        d, p, q = DR.tri_dist(P, Q)
        assert abs(d - _slsqp_distance(P, Q)) <= 1e-7, n_checked
        assert abs(np.linalg.norm(p - q) - d) <= 1e-12
        n_checked += 1


@pytest.mark.parametrize("case", ["T", "2D"])
def test_sat_gap_is_a_lower_bound(orc, meshes, case):
    """the oracle's SAT gap (pose_margin) of a free pose never exceeds its distance"""
    on, rn, rng = CASES[case]
    obst, robot = meshes[on], meshes[rn]
    if rng is None:
        r = np.random.RandomState(3)
        lo, hi = obst.reshape(-1, 3).min(0), obst.reshape(-1, 3).max(0)
        poses = np.zeros((300, 6))
        poses[:, :2] = r.uniform(lo[:2], hi[:2], (300, 2))
        poses[:, 3] = r.uniform(-np.pi, np.pi, 300)
    else:
        poses = orc.gen_poses(SEED, 0, 300, rng).astype(np.float64)
    hit = orc.collide_brute(obst, robot, poses)
    free = poses[hit == 0]
    assert len(free) > 50
    d, pts = DR.distance_batch(obst, robot, free)
    margin = orc.pose_margin(obst, robot, free)
    assert np.all(margin <= d * (1 + 1e-9) + 1e-9), np.max(margin - d)
    assert np.all(d > 0)
    np.testing.assert_allclose(np.linalg.norm(pts[:, :3] - pts[:, 3:], axis=1), d, rtol=0, atol=1e-9)
