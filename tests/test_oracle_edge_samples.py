"""The host generator of edge sample poses (tests/edge_samples.py) against the CPU oracle's isPathFree: the same number of
samples, and the oracle's verdict and first hit recomputed from the generated poses, in both rotation modes."""
import numpy as np
import pytest

import edge_samples as ES
from conftest import SEED


def seeded_edges(orc, m, seed, length=4.0, wide_angles=False):
    s = orc.gen_poses(SEED + seed, 0, m, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
    r = np.random.RandomState(seed)
    d = r.normal(size=(m, 3))
    e = s.copy()
    e[:, :3] += length * d / np.linalg.norm(d, axis=1, keepdims=True)
    if wide_angles:   # angles that wrap: differences beyond +-pi, ends up to 10 rad
        s[:, 3:] = r.uniform(-10, 10, (m, 3))
        e[:, 3:] = r.uniform(-10, 10, (m, 3))
    return s, e


def test_sample_counts(orc):
    s, e = seeded_edges(orc, 400, 3, length=1.0, wide_angles=True)
    e[:5] = s[:5]                    # no samples
    e[5:10, 0] = s[5:10, 0] + 0.05   # shorter than sample_dist
    e[5:10, 1:] = s[5:10, 1:]
    for i in range(len(s)):
        assert len(ES.edge_samples(s[i], e[i], 0.1, 1)) == orc.edge_num_samples(s[i], e[i], 0.1), i
        assert len(ES.edge_samples(s[i], e[i], 0.1, 0)) == orc.edge_num_samples(s[i], e[i], 0.1), i


@pytest.mark.parametrize("rot_mode", [0, 1])
def test_verdicts_and_first_hits_match_the_oracle(orc, meshes, rot_mode):
    ob, rb = meshes["building_s10"], meshes["robot_small_s10"]
    s, e = seeded_edges(orc, 300, 7, wide_angles=rot_mode == 1)
    free, first, _ = orc.edges_free(ob, rb, s, e, 0.1, rot_mode, models=(orc.ObbModel(ob), orc.ObbModel(rb)))
    assert 0.1 < free.mean() < 0.9
    poses, edge, index = ES.all_samples(s, e, 0.1, rot_mode)
    hit = orc.collide_brute(ob, rb, poses).astype(bool)
    for i in range(len(s)):
        h = hit[edge == i]
        assert bool(free[i]) == (not h.any()), i
        assert first[i] == (index[edge == i][np.argmax(h)] if h.any() else 0), i
