"""GPU tests of the asynchronous forms of the C ABI (sffg_*_begin + sffg_index_end / sffg_env_end): calls on different
objects in flight together return exactly what the blocking calls return; the device-side scan of sffg_radius (one host
synchronisation) keeps the capacity protocol; appends enqueued without a wait are seen by the searches that follow."""
import ctypes as C

import numpy as np
import pytest

from conftest import CASES, SEED

pytestmark = pytest.mark.gpu


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _nodes(orc, n, seed):
    return orc.gen_poses(seed, 0, n, [-50, 50, -50, 50, 0, 100]).astype(np.float32)


def test_rounds_in_flight_match_blocking_calls(sff, orc, meshes):
    """one planner round's independent questions in flight together: radius over the global index, k nearest in three tree
    indices, the edges of the crowding rule -- bit-identical to the blocking calls, for small and for growing indices"""
    from space_filling_forest_star_b200 import _lib
    L = _lib.load()
    on, rn, rng = CASES["B"]
    env = sff.Environment(meshes[on], meshes[rn])
    for n in (300, 30000):       # exhaustive kernels / Morton-sorted view + tail
        glob = sff.Index(_nodes(orc, n, SEED + 1))
        trees = [sff.Index(_nodes(orc, n // 3 + 17 * t, SEED + 10 + t)) for t in range(3)]
        q = _nodes(orc, 700, SEED + 40)
        per = np.array([300, 0, 400], dtype=np.int64)
        k = 12
        r2 = 60.0 if n == 300 else 9.0
        s = orc.gen_poses(SEED + 41, 0, 900, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
        e = s.copy()
        e[:, :3] += np.random.RandomState(3).normal(size=(900, 3))
        # blocking answers
        cnt_w, off_w, ids_w, d2_w = glob.radiusSearch(q, r2)
        kid_w = np.empty((700, k), np.int32)
        kd2_w = np.empty((700, k), np.float32)
        hs = (C.c_void_p * 3)(*[t._h.value for t in trees])
        _lib.check(L.sffg_knn_multi(hs, _p(per), 3, _p(q), k, _p(kid_w), _p(kd2_w)))
        free_w, first_w = env.isPathFree(s, e, 0.1, 0, want_first_hit=True)
        ok_w = env.checkMoves(s, e)
        # the same questions in flight together
        cap = int(off_w[-1]) + 5
        cnt = np.zeros(700, np.int32)
        ids = np.full(cap, -7, np.int32)
        d2 = np.zeros(cap, np.float32)
        total = C.c_int64(-1)
        kid = np.empty((700, k), np.int32)
        kd2 = np.empty((700, k), np.float32)
        free = np.zeros(900, np.uint8)
        first = np.zeros(900, np.int32)
        _lib.check(L.sffg_knn_multi_begin(hs, _p(per), 3, _p(q), k, _p(kid), _p(kd2)))
        _lib.check(L.sffg_radius_begin(glob._h, _p(q), 700, r2, _p(cnt), _p(ids), _p(d2), cap, C.byref(total)))
        _lib.check(L.sffg_check_edges_begin(env._h, _p(s), _p(e), 900, 0.1, 0, _p(free), _p(first)))
        # a second host-pointer call on an object with a pending call is refused, nothing is lost
        assert L.sffg_radius(glob._h, _p(q), 700, r2, _p(cnt), None, None, 0, None) == 3
        assert L.sffg_knn(trees[0]._h, _p(q), 1, 1, _p(kid), _p(kd2)) == 3
        assert L.sffg_check_moves(env._h, _p(s), _p(e), 900, 0.1, 0, _p(free)) == 3
        _lib.check(L.sffg_env_end(env._h))
        _lib.check(L.sffg_index_end(glob._h))
        _lib.check(L.sffg_index_end(trees[0]._h))
        assert L.sffg_index_end(trees[0]._h) == 0    # nothing pending: no-op
        assert total.value == off_w[-1]
        np.testing.assert_array_equal(cnt, cnt_w)
        np.testing.assert_array_equal(ids[: total.value], ids_w)
        np.testing.assert_array_equal(d2[: total.value].view(np.uint32), d2_w.view(np.uint32))
        np.testing.assert_array_equal(kid, kid_w)
        np.testing.assert_array_equal(kd2.view(np.uint32), kd2_w.view(np.uint32))
        np.testing.assert_array_equal(free, free_w)
        np.testing.assert_array_equal(first, first_w)
        ok = np.zeros(900, np.uint8)
        _lib.check(L.sffg_check_moves_begin(env._h, _p(s), _p(e), 900, 0.1, 0, _p(ok)))
        _lib.check(L.sffg_env_end(env._h))
        np.testing.assert_array_equal(ok, ok_w)
        for t in trees:
            t.close()
        glob.close()
    env.close()


def test_obstacle_changes_are_refused_while_edges_are_pending(sff, orc, meshes):
    """refit and set-obstacles are host-pointer calls too: between sffg_check_edges_begin and sffg_env_end both are refused
    and the obstacle set stays as it was, so the pending results equal the blocking call's"""
    from space_filling_forest_star_b200 import _lib
    L = _lib.load()
    on, rn, _ = CASES["B"]
    env = sff.Environment(meshes[on], meshes[rn])
    s = orc.gen_poses(SEED + 42, 0, 500, [-45, 45, -45, 45, 0, 125]).astype(np.float64)
    e = s.copy()
    e[:, :3] += np.random.RandomState(4).normal(size=(500, 3))
    free_w, first_w = env.isPathFree(s, e, 0.1, 0, want_first_hit=True)
    free = np.zeros(500, np.uint8)
    first = np.zeros(500, np.int32)
    _lib.check(L.sffg_check_edges_begin(env._h, _p(s), _p(e), 500, 0.1, 0, _p(free), _p(first)))
    with pytest.raises(_lib.SffgError) as refit:
        env.refit_obstacles(meshes[on])
    assert refit.value.code == 3
    with pytest.raises(_lib.SffgError) as replace:
        env.set_obstacles(meshes[on][: len(meshes[on]) // 2])
    assert replace.value.code == 3
    _lib.check(L.sffg_env_end(env._h))
    np.testing.assert_array_equal(free, free_w)
    np.testing.assert_array_equal(first, first_w)
    env.close()


def test_radius_one_synchronisation_keeps_the_capacity_protocol(sff, orc):
    """device-side scan: rows that fit come back from the single pass; a caller buffer that is too small gives
    SFFG_ERR_CAPACITY with the needed size; results larger than the pinned staging area take the two-pass route"""
    from space_filling_forest_star_b200 import _lib
    L = _lib.load()
    nodes = _nodes(orc, 40000, SEED + 2)
    idx = sff.Index(nodes)
    q = _nodes(orc, 2500, SEED + 3)        # 60 KB of queries: a planner-sized (pinned staging) call
    for r2 in (4.0, 150.0):           # ~ a few / ~ 60+ hits per row (the second total exceeds the staging area)
        cnt_w, off_w, ids_w, d2_w = idx.radiusSearch(q, r2)
        want_c, _, want_ids, want_d2 = orc.radius_linear(nodes, q, r2)
        total_w = int(off_w[-1])
        assert total_w > 0
        np.testing.assert_array_equal(cnt_w, want_c)
        np.testing.assert_array_equal(ids_w, want_ids)
        np.testing.assert_array_equal(d2_w.view(np.uint32), want_d2.view(np.uint32))
        cnt = np.zeros(len(q), np.int32)
        total = C.c_int64(0)
        ids = np.empty(total_w, np.int32)
        d2 = np.empty(total_w, np.float32)
        # too small by one entry
        rc = L.sffg_radius(idx._h, _p(q), len(q), r2, _p(cnt), _p(ids), _p(d2), total_w - 1, C.byref(total))
        assert rc == 5 and total.value == total_w
        np.testing.assert_array_equal(cnt, cnt_w)
        # exact fit
        _lib.check(L.sffg_radius(idx._h, _p(q), len(q), r2, _p(cnt), _p(ids), _p(d2), total_w, C.byref(total)))
        assert total.value == total_w
        np.testing.assert_array_equal(ids, ids_w)
        np.testing.assert_array_equal(d2.view(np.uint32), d2_w.view(np.uint32))
        # every row sorted by (d2, id), strict radius
        for i in (0, 1, len(q) // 2, len(q) - 1):
            row = slice(off_w[i], off_w[i + 1])
            key = d2[row].astype(np.float64) * 2.0 ** 32 + ids[row]
            assert np.all(np.diff(key) > 0) and np.all(d2[row] < np.float32(r2))
    assert int(off_w[-1]) * 8 > (1 << 20)      # the large-radius case did not fit the staging area
    idx.close()


def test_appends_without_a_wait_are_seen_by_the_next_search(sff, orc):
    """sffg_index_add_multi_begin returns at once; searches on every index it appended to are ordered behind it"""
    from space_filling_forest_star_b200 import _lib
    L = _lib.load()
    base = _nodes(orc, 5000, SEED + 5)
    extra = _nodes(orc, 64, SEED + 6)
    glob, tree = sff.Index(base), sff.Index(base[:2000])
    hs = (C.c_void_p * 2)(glob._h.value, tree._h.value)
    rows = np.ascontiguousarray(np.concatenate([extra, extra[:40]]))
    per = np.array([64, 40], dtype=np.int64)
    _lib.check(L.sffg_index_add_multi_begin(hs, _p(per), 2, _p(rows)))
    assert glob.size() == 5064 and tree.size() == 2040
    # the tree index was not the lead: searching it needs no end call and must already see the new nodes
    ids, d2 = tree.knnSearch(extra[:40], 1)
    np.testing.assert_array_equal(ids[:, 0], 2000 + np.arange(40))
    assert np.all(d2[:, 0] == 0)
    # the lead's staging area is in use until its end call
    assert L.sffg_index_add(glob._h, _p(extra), 1) == 3
    _lib.check(L.sffg_index_end(glob._h))
    ids, d2 = glob.knnSearch(extra, 1)
    np.testing.assert_array_equal(ids[:, 0], 5000 + np.arange(64))
    glob.close()
    tree.close()


def test_one_kernel_radius_on_small_indices(sff, orc):
    """planner-sized searches on small indices run in one kernel (block per query, rows packed in completion order and put
    back into query order by the host); rows longer than its shared buffer or a full staging area fall back to the general
    path -- every case equals the oracle bit for bit, in 6-D (angles out of [-pi, pi) included) and in 2-D"""
    nodes = _nodes(orc, 6000, SEED + 7)
    nodes[:, 3:] *= 2.5
    q = _nodes(orc, 900, SEED + 8)
    idx = sff.Index(nodes[:4000])
    idx.addPoints(nodes[4000:])
    for r2 in (25.0, 400.0, 3000.0, 1.0e9):      # few hits / tens / hundreds (staging area overflows) / every node (row > buffer)
        for nq in (1, 37, 900):
            cnt, off, ids, d2 = idx.radiusSearch(q[:nq], r2)
            wc, woff, wi, wd = orc.radius_linear(nodes, q[:nq], r2)
            np.testing.assert_array_equal(cnt, wc)
            np.testing.assert_array_equal(ids, wi)
            np.testing.assert_array_equal(d2.view(np.uint32), wd.view(np.uint32))
    assert wc.min() == 6000
    idx.close()
    n2 = np.ascontiguousarray(_nodes(orc, 3000, SEED + 9)[:, :2]) * np.float32(10.0)
    q2 = np.ascontiguousarray(_nodes(orc, 200, SEED + 10)[:, :2]) * np.float32(10.0)
    idx2 = sff.Index(n2)
    for r2 in (900.0, 67600.0):                  # the planner's 2-D radius^2 is 67 600
        cnt, off, ids, d2 = idx2.radiusSearch(q2, r2)
        wc, woff, wi, wd = orc.radius_linear(n2, q2, r2)
        np.testing.assert_array_equal(cnt, wc)
        np.testing.assert_array_equal(ids, wi)
        np.testing.assert_array_equal(d2.view(np.uint32), wd.view(np.uint32))
    idx2.close()
    empty = sff.Index(dim=6)
    cnt, off, ids, d2 = empty.radiusSearch(q[:5], 10.0)
    assert cnt.sum() == 0 and len(ids) == 0
    empty.close()
