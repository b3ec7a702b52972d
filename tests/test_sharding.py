"""world_size-2 gloo test of the multi-GPU host logic (split -> local compute -> one all-gather)."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parents[1]


def test_shard_bounds_cover_everything():
    from space_filling_forest_star_b200.sharding import shard_bounds
    for n in (0, 1, 2, 7, 8, 9, 1000003):
        for world in (1, 2, 3, 8):
            seen = 0
            for r in range(world):
                b, e, per = shard_bounds(n, r, world)
                assert b == seen and e - b <= per and e <= n
                seen = e
            assert seen == n


def _init_gloo(rank, world, tmp):
    """rendezvous through a file in the test's own directory: no TCP port to pick, so no port another process may hold"""
    sys.path.insert(0, str(ROOT))
    dist.init_process_group("gloo", init_method=Path(tmp, "rendezvous").resolve().as_uri(), rank=rank, world_size=world)


def _worker(rank, world, n, tmp):
    _init_gloo(rank, world, tmp)
    from space_filling_forest_star_b200.sharding import shard_bounds, sharded_rows
    poses = torch.arange(n * 6, dtype=torch.float32).reshape(n, 6)

    def compute(b, e, out):     # stands in for env.collide_device on this rank's slice
        out[: e - b] = (poses[b:e, 0].to(torch.int64) // 6 % 3 == 0).to(torch.uint8)

    got = sharded_rows(n, (), torch.uint8, "cpu", compute)
    want = (torch.arange(n) % 3 == 0).to(torch.uint8)
    ok = torch.equal(got, want)

    def compute_rows(b, e, out):
        out[: e - b, :, 0] = torch.arange(b, e, dtype=torch.int32)[:, None]
        out[: e - b, :, 1] = rank

    rows = sharded_rows(n, (4, 2), torch.int32, "cpu", compute_rows)
    ok = ok and torch.equal(rows[:, 0, 0], torch.arange(n, dtype=torch.int32))
    b, e, _ = shard_bounds(n, rank, world)
    ok = ok and bool((rows[b:e, :, 1] == rank).all())
    Path(tmp, f"ok{rank}").write_text(str(ok))
    dist.destroy_process_group()


@pytest.mark.parametrize("n", [0, 5, 64, 1001])
def test_sharded_rows_gloo_world2(tmp_path, n):
    mp.spawn(_worker, args=(2, n, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").read_text() == "True" and (tmp_path / "ok1").read_text() == "True"


class _FakeIndex:
    """stands in for engine.Index.knn_device on CPU tensors: row i of the result is a function of query row i only"""

    def knn_device(self, queries, k, ids_out, d2_out):
        base = queries[:, 0].to(torch.int32)
        ids_out.copy_(base[:, None] * 100 + torch.arange(k, dtype=torch.int32)[None, :])
        d2_out.copy_(queries[:, 1:2] + torch.arange(k, dtype=torch.float32)[None, :])


def _knn_worker(rank, world, nq, k, tmp):
    _init_gloo(rank, world, tmp)
    from space_filling_forest_star_b200.sharding import sharded_knn
    q = torch.stack([torch.arange(nq, dtype=torch.float32), torch.arange(nq, dtype=torch.float32) * 0.5], 1).contiguous()
    ids, d2 = sharded_knn(_FakeIndex(), q, k)
    want_i = torch.arange(nq, dtype=torch.int32)[:, None] * 100 + torch.arange(k, dtype=torch.int32)[None, :]
    want_d = q[:, 1:2] + torch.arange(k, dtype=torch.float32)[None, :]
    ok = ids.shape == (nq, k) and torch.equal(ids, want_i) and torch.equal(d2, want_d)
    Path(tmp, f"ok{rank}").write_text(str(ok))
    dist.destroy_process_group()


@pytest.mark.parametrize("nq", [0, 1, 7, 64, 1001])
def test_sharded_knn_in_place_gather_gloo_world2(tmp_path, nq):
    """the search writes its rows into its slice of the gathered buffers and the all-gathers run in place on them"""
    mp.spawn(_knn_worker, args=(2, nq, 5, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").read_text() == "True" and (tmp_path / "ok1").read_text() == "True"


class _FakeRadiusIndex:
    """stands in for engine.Index.radiusSearch: row i holds (int(q[i,0]) % 5) entries derived from the query row alone"""

    def radiusSearch(self, queries, radius_sq):
        import numpy as np
        cnt = (queries[:, 0].astype(np.int64) % 5).astype(np.int32)
        off = np.zeros(len(queries) + 1, dtype=np.int64)
        np.cumsum(cnt, out=off[1:])
        ids = np.concatenate([np.arange(c, dtype=np.int32) + 10 * int(q0) for c, q0 in zip(cnt, queries[:, 0])] + [np.zeros(0, np.int32)])
        d2 = ids.astype(np.float32) * np.float32(0.25) + np.float32(radius_sq)
        return cnt, off, ids, d2


def _radius_worker(rank, world, nq, tmp):
    import numpy as np
    _init_gloo(rank, world, tmp)
    from space_filling_forest_star_b200.sharding import sharded_radius
    q = np.stack([np.arange(nq, dtype=np.float32) * 3 + 1, np.zeros(nq, dtype=np.float32)], 1)
    counts, offsets, ids, d2 = sharded_radius(_FakeRadiusIndex(), q, 2.0)
    wc, woff, wi, wd = _FakeRadiusIndex().radiusSearch(q, 2.0)
    ok = (np.array_equal(counts.numpy(), wc) and np.array_equal(offsets.numpy(), woff) and np.array_equal(ids.numpy(), wi)
          and np.array_equal(d2.numpy().view(np.uint32), wd.view(np.uint32)))
    Path(tmp, f"ok{rank}").write_text(str(ok))
    dist.destroy_process_group()


@pytest.mark.parametrize("nq", [0, 1, 2, 9, 500])
def test_sharded_radius_variable_rows_gloo_world2(tmp_path, nq):
    """counts first, then the packed rows padded to the largest per-rank total; every rank ends with the whole CSR result"""
    mp.spawn(_radius_worker, args=(2, nq, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").read_text() == "True" and (tmp_path / "ok1").read_text() == "True"
