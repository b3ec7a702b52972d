"""The motion of sffg_sweep_edges on the CPU (tests/sweep_motion.py): the motion bound mu really bounds how fast every
vertex of every golden robot moves, in both rotation modes, and the samples isPathFree checks lie on the motion."""
import numpy as np
import pytest

import distance_ref as DR
import edge_samples as ES
import sweep_motion as SM

ROBOTS = ("robot_small_s10", "robot_small_s1", "robot_cyl_small_s10")


def random_edges(seed, m, length, wide_angles):
    r = np.random.RandomState(seed)
    s = np.concatenate([r.uniform(-50, 50, (m, 3)), r.uniform(-np.pi, np.pi, (m, 3))], axis=1)
    e = s.copy()
    d = r.normal(size=(m, 3))
    e[:, :3] += r.uniform(0, length, (m, 1)) * d / np.linalg.norm(d, axis=1, keepdims=True)
    e[:, 3:] = r.uniform(-np.pi, np.pi, (m, 3))
    if wide_angles:   # differences beyond +-pi (wrapped) and angles up to 10 rad
        s[:, 3:] = r.uniform(-10, 10, (m, 3))
        e[:, 3:] = r.uniform(-10, 10, (m, 3))
    e[:4] = s[:4]               # motionless
    e[4:8, :3] = s[4:8, :3]     # rotation only
    return s, e


def vertices_at(robot, pose):
    """world positions of the robot's vertices [n][3] at pose [6]"""
    v = np.asarray(robot, dtype=np.float64).reshape(-1, 3)
    return v @ DR.rotation(pose[3], pose[4], pose[5]).T + pose[:3]


@pytest.mark.parametrize("rot_mode", [0, 1])
@pytest.mark.parametrize("robot_name", ROBOTS)
def test_motion_bound_is_lipschitz(meshes, robot_name, rot_mode):
    robot = meshes[robot_name]
    rho = SM.radius(robot)
    r = np.random.RandomState(11 + rot_mode)
    for wide in (False, True):
        s, e = random_edges(5 + rot_mode + 2 * wide, 60, 12.0, wide)
        mu = SM.motion_bound(s, e, rho, rot_mode)
        for i in range(len(s)):
            t1 = r.uniform(0, 1, 48)
            t2 = np.clip(t1 + r.normal(scale=r.choice([1e-4, 1e-2, 0.3]), size=48), 0, 1)
            p1 = SM.poses(s[i], e[i], t1, rot_mode)
            p2 = SM.poses(s[i], e[i], t2, rot_mode)
            for a, b, ta, tb in zip(p1, p2, t1, t2):
                moved = np.linalg.norm(vertices_at(robot, a) - vertices_at(robot, b), axis=1).max()
                assert moved <= mu[i] * abs(ta - tb) + 1e-12 * (1.0 + np.abs(a[:3]).max()), (i, ta, tb)
        if rot_mode == 0:   # translation only: the bound is attained
            i = 20
            a, b = SM.poses(s[i], e[i], [0.0, 1.0], rot_mode)
            assert np.isclose(np.linalg.norm(vertices_at(robot, a) - vertices_at(robot, b), axis=1).max(), mu[i])


@pytest.mark.parametrize("rot_mode", [0, 1])
def test_samples_lie_on_the_motion(rot_mode):
    for wide in (False, True):
        s, e = random_edges(21 + rot_mode, 200, 8.0, wide)
        for i in range(len(s)):
            smp = ES.edge_samples(s[i], e[i], 0.1, rot_mode)
            if len(smp) == 0:
                continue
            f = np.asarray(e[i])
            total = sum((s[i][k] - f[k]) ** 2 for k in range(3)) + sum(float(ES.wrap(f[3 + k] - s[i][3 + k])) ** 2 for k in range(3))
            parts = np.sqrt(total) / 0.1
            tau = np.arange(1, len(smp) + 1, dtype=np.float64) / parts
            got = SM.poses(s[i], e[i], tau, rot_mode)
            step = np.concatenate([f[:3] - s[i][:3], ES.wrap(f[3:] - s[i][3:])])
            scale = np.maximum(np.abs(smp), np.abs(step))
            assert np.all(np.abs(got - smp) <= 8 * np.spacing(scale)), i
            if rot_mode == 0:
                assert np.all(got[:, 3:] == 0) and np.all(smp[:, 3:] == 0)
