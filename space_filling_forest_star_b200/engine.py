"""Host-side mirror of the reference interfaces that sit on the hot path, backed by libsffg.so (CUDA only).

Names follow the reference so that parity tests read like the reference's own call sites:

* :class:`Environment`  -- ``Environment<T>`` (src/environment.h:28-55): ``Collide`` (:306-316) over a batch of poses,
  ``isPathFree`` (``Solver<T,R>::isPathFree``, src/problemStruct.h:154-168) over a batch of edges
* :class:`Index`        -- ``flann::Index<D6Distance<float>>`` as the planner uses it (src/forest.h:72-73, :266, :317,
  :367): ``buildIndex``, ``addPoints``, ``knnSearch``, ``radiusSearch``
* :func:`load_mesh`     -- ``Obstacle<T>::ParseOBJFile`` / ``ParseMapFile`` (src/environment.h:125-223)

numpy arrays are host buffers (the call copies H2D, runs the kernels, copies D2H); the ``*_device`` methods take
torch CUDA tensors and only enqueue work on the current torch stream.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import BUILD_AUTO, BUILD_DEVICE, BUILD_HOST, ROT_INTERPOLATE, ROT_REFERENCE, SffgError, check  # noqa: F401

COLLISION_SAMPLE_SIZE = 0.1   # Solver::collisionSampleSize, src/problemStruct.h:121


def _ptr(a) -> int:
    return a.ctypes.data


def init(device: int = -1) -> None:
    """Bind the engine to a GPU (sffg_init).  Raises SffgError(NO_DEVICE) when there is none."""
    check(_lib.load().sffg_init(device))


def device_count() -> int:
    return _lib.load().sffg_device_count()


def load_mesh(path: str, is_obj, position: Sequence[float] = (0.0, 0.0, 0.0), scale: float = 1.0
              ) -> Tuple[np.ndarray, np.ndarray]:
    """-> (triangles float64 [n][3][3], bbox float64[6] = minX maxX minY maxY minZ maxZ).

    ``is_obj``: False/0 = 2-D .tri map, True/1 = OBJ as the reference reads it, 2 = repaired OBJ reading (opt-in)."""
    L = _lib.load()
    pos = np.asarray(position, dtype=np.float64)
    out = C.c_void_p()
    n = C.c_int64()
    bbox = np.zeros(6, dtype=np.float64)
    check(L.sffg_mesh_load(str(path).encode(), int(is_obj), _ptr(pos), float(scale), C.byref(out), C.byref(n), _ptr(bbox)))
    try:
        buf = (C.c_double * (9 * n.value)).from_address(out.value) if n.value else []
        tris = np.array(buf, dtype=np.float64).reshape(-1, 3, 3)
    finally:
        L.sffg_free(out)
    return tris, bbox


class Environment:
    """Obstacle BVH + robot mesh resident on one GPU."""

    def __init__(self, obstacle_tris, robot_tris, build: int = BUILD_AUTO):
        """``build``: where the obstacle hierarchy is built (BUILD_AUTO / BUILD_HOST / BUILD_DEVICE, include/sffg.h)"""
        self._L = _lib.load()
        self._h = C.c_void_p()
        o = np.ascontiguousarray(np.asarray(obstacle_tris, dtype=np.float64).reshape(-1, 9))
        r = np.ascontiguousarray(np.asarray(robot_tris, dtype=np.float64).reshape(-1, 9))
        check(self._L.sffg_env_create_ex(_ptr(o) if len(o) else None, len(o), _ptr(r), len(r), int(build), C.byref(self._h)))

    def set_obstacles(self, obstacle_tris, build: int = BUILD_AUTO) -> None:
        """replace the obstacle soup in place (moving obstacles): hierarchy, triangle arrays and clearance grid are rebuilt"""
        o = np.ascontiguousarray(np.asarray(obstacle_tris, dtype=np.float64).reshape(-1, 9))
        check(self._L.sffg_env_set_obstacles(self._h, _ptr(o) if len(o) else None, len(o), int(build)))

    def refit_obstacles(self, obstacle_tris) -> None:
        """the same triangles (count and order) at new positions: boxes, triangle arrays, top cut and clearance grid are
        recomputed, the topology of the hierarchy is kept (sffg_env_refit_obstacles)"""
        o = np.ascontiguousarray(np.asarray(obstacle_tris, dtype=np.float64).reshape(-1, 9))
        check(self._L.sffg_env_refit_obstacles(self._h, _ptr(o), len(o)))

    @classmethod
    def from_files(cls, robot_file: str, robot_is_obj: bool, obstacles: Sequence[Tuple[str, bool, Sequence[float]]],
                   scale: float = 1.0) -> "Environment":
        """Mirrors parseFile (src/main.cpp:161, :254): one robot Obstacle + a deque of obstacle meshes."""
        robot, _ = load_mesh(robot_file, robot_is_obj, (0, 0, 0), scale)
        soups = [load_mesh(f, io, pos, scale)[0] for (f, io, pos) in obstacles]
        obst = np.concatenate(soups) if soups else np.zeros((0, 3, 3))
        return cls(obst, robot)

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.sffg_env_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def info(self) -> dict:
        i = _lib.EnvInfo()
        check(self._L.sffg_env_info(self._h, C.byref(i)))
        return {k: getattr(i, k) for k, _ in i._fields_}

    # ---- Environment<T>::Collide ---------------------------------------------------------------------------
    def Collide(self, poses) -> np.ndarray:
        """poses [n][6] float32 or float64 (x y z yaw pitch roll) -> uint8[n], 1 = robot touches an obstacle."""
        p = np.asarray(poses)
        if p.dtype != np.float32:
            p = p.astype(np.float64, copy=False)
        p = np.ascontiguousarray(p.reshape(-1, 6))
        out = np.empty(len(p), dtype=np.uint8)
        fn = self._L.sffg_collide_poses_f32 if p.dtype == np.float32 else self._L.sffg_collide_poses_f64
        check(fn(self._h, _ptr(p) if len(p) else None, len(p), _ptr(out) if len(p) else None))
        return out

    def CollideTransforms(self, R, T) -> np.ndarray:
        """RAPID_Collide's own argument form: R [n][3][3] row-major rotation of the robot, T [n][3] -> uint8[n]."""
        R = np.asarray(R, dtype=np.float64).reshape(-1, 9)
        T = np.asarray(T, dtype=np.float64).reshape(-1, 3)
        rt = np.ascontiguousarray(np.concatenate([R, T], axis=1))
        out = np.empty(len(rt), dtype=np.uint8)
        check(self._L.sffg_collide_transforms_f64(self._h, _ptr(rt) if len(rt) else None, len(rt), _ptr(out) if len(rt) else None))
        return out

    def collide_host_buffers(self, poses_ptr: int, is_f64: bool, n: int, out_ptr: int) -> None:
        """Raw host-pointer form of Collide (pinned buffers from the caller), used by bench.py's e2e leg."""
        fn = self._L.sffg_collide_poses_f64 if is_f64 else self._L.sffg_collide_poses_f32
        check(fn(self._h, poses_ptr, n, out_ptr))

    def edges_host_buffers(self, starts_ptr: int, ends_ptr: int, m: int, free_ptr: int, sample_dist: float = COLLISION_SAMPLE_SIZE,
                           rot_mode: int = ROT_REFERENCE) -> None:
        """Raw host-pointer form of isPathFree (pinned float64 [m][6] buffers from the caller), used by bench.py's e2e leg."""
        check(self._L.sffg_check_edges(self._h, starts_ptr, ends_ptr, m, float(sample_dist), rot_mode, free_ptr, None))

    def collide_device(self, poses, out=None, stream: Optional[int] = None):
        """poses: torch CUDA tensor [n][6] float32/float64; returns a torch uint8 tensor (enqueued, not synchronised)."""
        import torch
        assert poses.is_cuda and poses.is_contiguous() and poses.shape[-1] == 6
        n = poses.numel() // 6
        if out is None:
            out = torch.empty(n, dtype=torch.uint8, device=poses.device)
        st = torch.cuda.current_stream(poses.device).cuda_stream if stream is None else stream
        check(self._L.sffg_collide_poses_device(self._h, poses.data_ptr(), int(poses.dtype == torch.float64), n, out.data_ptr(), st))
        return out

    # ---- separation distance (sffg_distance_poses) -----------------------------------------------------------
    def Distance(self, poses, max_dist: float = np.inf, points: bool = False):
        """poses [n][6] float32 or float64 -> dist float64[n]: distance robot <-> obstacles capped at max_dist, 0 exactly
        where Collide says 1; with ``points`` also float64 [n][6] (nearest robot point, nearest obstacle point, world
        frame; NaN unless 0 < dist < max_dist)."""
        p = np.asarray(poses)
        if p.dtype != np.float32:
            p = p.astype(np.float64, copy=False)
        p = np.ascontiguousarray(p.reshape(-1, 6))
        n = len(p)
        dist = np.empty(n, dtype=np.float64)
        pts = np.empty((n, 6), dtype=np.float64) if points else None
        check(self._L.sffg_distance_poses(self._h, _ptr(p) if n else None, int(p.dtype == np.float64), n, float(max_dist),
                                          _ptr(dist) if n else None, _ptr(pts) if (points and n) else None))
        return (dist, pts) if points else dist

    def distance_device(self, poses, max_dist: float = np.inf, out=None, points=None, stream: Optional[int] = None):
        """poses: torch CUDA tensor [n][6] float32/float64 -> torch float64 [n] (enqueued, not synchronised); ``points``
        (optional torch float64 [n][6] on the same device) receives the nearest points."""
        import torch
        assert poses.is_cuda and poses.is_contiguous() and poses.shape[-1] == 6
        n = poses.numel() // 6
        if out is None:
            out = torch.empty(n, dtype=torch.float64, device=poses.device)
        assert out.dtype == torch.float64 and out.is_contiguous() and out.numel() == n
        if points is not None:
            assert points.dtype == torch.float64 and points.is_contiguous() and points.numel() == 6 * n
        st = torch.cuda.current_stream(poses.device).cuda_stream if stream is None else stream
        check(self._L.sffg_distance_poses_device(self._h, poses.data_ptr(), int(poses.dtype == torch.float64), n, float(max_dist),
                                                 out.data_ptr(), points.data_ptr() if points is not None else None, st))
        return out

    def EdgeDistance(self, starts, ends, max_dist: float = np.inf, sample_dist: float = COLLISION_SAMPLE_SIZE,
                     rot_mode: int = ROT_REFERENCE, points: bool = False):
        """edges start -> end ([m][6] float64) -> (dist float64[m], index int32[m]): the minimum over the samples isPathFree
        checks of the pose distance capped at max_dist (0 exactly where isPathFree says 0) and the lowest sample reporting
        it (the first hit on contact, 0 when dist == max_dist); with ``points`` also float64 [m][6] (nearest robot point at
        that sample, nearest obstacle point; NaN unless 0 < dist < max_dist).  The end points are not samples."""
        s = np.ascontiguousarray(np.asarray(starts, dtype=np.float64).reshape(-1, 6))
        e = np.ascontiguousarray(np.asarray(ends, dtype=np.float64).reshape(-1, 6))
        assert len(s) == len(e)
        m = len(s)
        dist = np.empty(m, dtype=np.float64)
        index = np.empty(m, dtype=np.int32)
        pts = np.empty((m, 6), dtype=np.float64) if points else None
        check(self._L.sffg_distance_edges(self._h, _ptr(s) if m else None, _ptr(e) if m else None, m, float(sample_dist), rot_mode,
                                          float(max_dist), _ptr(dist) if m else None, _ptr(index) if m else None,
                                          _ptr(pts) if (points and m) else None))
        return (dist, index, pts) if points else (dist, index)

    def edge_distance_device(self, starts, ends, max_dist: float = np.inf, sample_dist: float = COLLISION_SAMPLE_SIZE,
                             rot_mode: int = ROT_REFERENCE, out=None, index_out=None, points=None, stream: Optional[int] = None):
        """starts, ends: torch CUDA float64 [m][6] -> torch float64 [m] (enqueued, not synchronised); ``index_out`` (int32
        [m]) and ``points`` (float64 [m][6]) on the same device are optional."""
        import torch
        assert starts.is_cuda and starts.dtype == torch.float64 and ends.dtype == torch.float64
        assert starts.is_contiguous() and ends.is_contiguous() and starts.shape == ends.shape
        m = starts.numel() // 6
        if out is None:
            out = torch.empty(m, dtype=torch.float64, device=starts.device)
        assert out.dtype == torch.float64 and out.is_contiguous() and out.numel() == m
        if index_out is not None:
            assert index_out.dtype == torch.int32 and index_out.is_contiguous() and index_out.numel() == m
        if points is not None:
            assert points.dtype == torch.float64 and points.is_contiguous() and points.numel() == 6 * m
        st = torch.cuda.current_stream(starts.device).cuda_stream if stream is None else stream
        check(self._L.sffg_distance_edges_device(self._h, starts.data_ptr(), ends.data_ptr(), m, float(sample_dist), rot_mode,
                                                 float(max_dist), out.data_ptr(),
                                                 index_out.data_ptr() if index_out is not None else None,
                                                 points.data_ptr() if points is not None else None, st))
        return out

    # ---- continuous edge check (sffg_sweep_edges) ------------------------------------------------------------
    def SweepEdges(self, starts, ends, margin: float, rot_mode: int = ROT_REFERENCE):
        """edges start -> end ([m][6] float64) -> (clear uint8[m], t float64[m], dist float64[m]): clear = 1 certifies every
        pose of the motion start + t (end - start), t in [0, 1], at distance >= margin / 2 (t = 1, dist = margin);
        otherwise the motion is certified on [0, t) and dist < margin is the pose distance at t (0 on contact)."""
        s = np.ascontiguousarray(np.asarray(starts, dtype=np.float64).reshape(-1, 6))
        e = np.ascontiguousarray(np.asarray(ends, dtype=np.float64).reshape(-1, 6))
        assert len(s) == len(e)
        m = len(s)
        clear = np.empty(m, dtype=np.uint8)
        t = np.empty(m, dtype=np.float64)
        dist = np.empty(m, dtype=np.float64)
        check(self._L.sffg_sweep_edges(self._h, _ptr(s) if m else None, _ptr(e) if m else None, m, rot_mode, float(margin),
                                       _ptr(clear) if m else None, _ptr(t) if m else None, _ptr(dist) if m else None))
        return clear, t, dist

    def sweep_edges_device(self, starts, ends, margin: float, rot_mode: int = ROT_REFERENCE, clear_out=None, t_out=None,
                           dist_out=None, stream: Optional[int] = None):
        """starts, ends: torch CUDA float64 [m][6] -> torch uint8 [m] clear flags (enqueued, not synchronised); ``t_out`` and
        ``dist_out`` (float64 [m] on the same device) are optional."""
        import torch
        assert starts.is_cuda and starts.dtype == torch.float64 and ends.dtype == torch.float64
        assert starts.is_contiguous() and ends.is_contiguous() and starts.shape == ends.shape
        m = starts.numel() // 6
        if clear_out is None:
            clear_out = torch.empty(m, dtype=torch.uint8, device=starts.device)
        assert clear_out.dtype == torch.uint8 and clear_out.is_contiguous() and clear_out.numel() == m
        for o in (t_out, dist_out):
            if o is not None:
                assert o.dtype == torch.float64 and o.is_contiguous() and o.numel() == m
        st = torch.cuda.current_stream(starts.device).cuda_stream if stream is None else stream
        check(self._L.sffg_sweep_edges_device(self._h, starts.data_ptr(), ends.data_ptr(), m, rot_mode, float(margin),
                                              clear_out.data_ptr(), t_out.data_ptr() if t_out is not None else None,
                                              dist_out.data_ptr() if dist_out is not None else None, st))
        return clear_out

    # ---- Solver<T,R>::isPathFree ---------------------------------------------------------------------------
    def isPathFree(self, starts, ends, sample_dist: float = COLLISION_SAMPLE_SIZE, rot_mode: int = ROT_REFERENCE,
                   want_first_hit: bool = False):
        s = np.ascontiguousarray(np.asarray(starts, dtype=np.float64).reshape(-1, 6))
        e = np.ascontiguousarray(np.asarray(ends, dtype=np.float64).reshape(-1, 6))
        assert len(s) == len(e)
        free = np.empty(len(s), dtype=np.uint8)
        first = np.empty(len(s), dtype=np.int32) if want_first_hit else None
        m = len(s)
        check(self._L.sffg_check_edges(self._h, _ptr(s) if m else None, _ptr(e) if m else None, m, float(sample_dist), rot_mode,
                                       _ptr(free) if m else None, _ptr(first) if (want_first_hit and m) else None))
        return (free, first) if want_first_hit else free

    def checkMoves(self, starts, ends, sample_dist: float = COLLISION_SAMPLE_SIZE, rot_mode: int = ROT_REFERENCE) -> np.ndarray:
        """``!env.Collide(end) && isPathFree(start, end)`` per row: the validity test of an expansion step
        (src/forest.h:246, src/rrt.h:149) in one engine call -> uint8[m], 1 = valid"""
        s = np.ascontiguousarray(np.asarray(starts, dtype=np.float64).reshape(-1, 6))
        e = np.ascontiguousarray(np.asarray(ends, dtype=np.float64).reshape(-1, 6))
        assert len(s) == len(e)
        ok = np.empty(len(s), dtype=np.uint8)
        m = len(s)
        check(self._L.sffg_check_moves(self._h, _ptr(s) if m else None, _ptr(e) if m else None, m, float(sample_dist), rot_mode,
                                       _ptr(ok) if m else None))
        return ok

    def edges_device(self, starts, ends, sample_dist: float = COLLISION_SAMPLE_SIZE, rot_mode: int = ROT_REFERENCE,
                     free_out=None, first_hit_out=None, stream: Optional[int] = None):
        import torch
        assert starts.is_cuda and starts.dtype == torch.float64 and starts.is_contiguous() and ends.is_contiguous()
        m = starts.numel() // 6
        if free_out is None:
            free_out = torch.empty(m, dtype=torch.uint8, device=starts.device)
        st = torch.cuda.current_stream(starts.device).cuda_stream if stream is None else stream
        check(self._L.sffg_check_edges_device(self._h, starts.data_ptr(), ends.data_ptr(), m, float(sample_dist), rot_mode,
                                              free_out.data_ptr(), first_hit_out.data_ptr() if first_hit_out is not None else None, st))
        return free_out

    def sync_check(self) -> None:
        check(self._L.sffg_env_sync_check(self._h))

    def enable_counters(self, on: bool = True) -> None:
        check(self._L.sffg_env_enable_counters(self._h, int(on)))

    def read_counters(self) -> dict:
        c = _lib.Counters()
        check(self._L.sffg_env_read_counters(self._h, C.byref(c)))
        return {k: getattr(c, k) for k, _ in c._fields_}


def gen_poses_device(seed: int, first_index: int, n: int, rng: Sequence[float], out=None):
    """Philox pose stream generated on the GPU (torch float32 [n][6]); bit-identical to oracle.gen_poses."""
    import torch
    L = _lib.load()
    if out is None:
        out = torch.empty((n, 6), dtype=torch.float32, device="cuda")
    r = np.asarray(rng, dtype=np.float32)
    check(L.sffg_gen_poses_device(seed, first_index, n, _ptr(r), out.data_ptr(), torch.cuda.current_stream().cuda_stream))
    return out


class Index:
    """Exact neighbour index over 2-D or 6-D nodes: the planner-facing subset of flann::Index<D6Distance<float>>.

    ``Index(points)`` + ``buildIndex()`` + ``addPoints(rows)`` reproduce src/forest.h:72-73 / :367; ids are insertion
    order; distances are squared; ``knnSearch`` rows ascend by (d2, id); ``radiusSearch`` is strict (d2 < r2).
    """

    def __init__(self, points=None, dim: Optional[int] = None):
        self._L = _lib.load()
        self._h = C.c_void_p()
        if points is not None:
            points = np.ascontiguousarray(np.asarray(points, dtype=np.float32))
            points = points.reshape(-1, points.shape[-1])
            dim = points.shape[1]
        if dim is None:
            raise ValueError("Index needs points or dim")
        self.dim = int(dim)
        check(self._L.sffg_index_create(self.dim, C.byref(self._h)))
        if points is not None and len(points):
            self.addPoints(points)

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.sffg_index_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def buildIndex(self) -> None:
        """No tree to build: the node set is scanned exactly (kept for call-site compatibility, src/forest.h:73)."""

    def addPoints(self, points) -> None:
        p = np.ascontiguousarray(np.asarray(points, dtype=np.float32).reshape(-1, self.dim))
        check(self._L.sffg_index_add(self._h, _ptr(p) if len(p) else None, len(p)))

    def add_device(self, points, stream: Optional[int] = None) -> None:
        import torch
        assert points.is_cuda and points.dtype == torch.float32 and points.is_contiguous()
        st = torch.cuda.current_stream(points.device).cuda_stream if stream is None else stream
        check(self._L.sffg_index_add_device(self._h, points.data_ptr(), points.numel() // self.dim, st))

    def size(self) -> int:
        return int(self._L.sffg_index_size(self._h))

    def knnSearch(self, queries, knn: int) -> Tuple[np.ndarray, np.ndarray]:
        """-> (ids int32 [nq][k] (-1 padded), d2 float32 [nq][k] (+inf padded))"""
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32).reshape(-1, self.dim))
        ids = np.empty((len(q), knn), dtype=np.int32)
        d2 = np.empty((len(q), knn), dtype=np.float32)
        nq = len(q)
        check(self._L.sffg_knn(self._h, _ptr(q) if nq else None, nq, int(knn), _ptr(ids) if nq else None, _ptr(d2) if nq else None))
        return ids, d2

    def knn_device(self, queries, knn: int, ids_out=None, d2_out=None, stream: Optional[int] = None):
        import torch
        assert queries.is_cuda and queries.dtype == torch.float32 and queries.is_contiguous()
        nq = queries.numel() // self.dim
        if ids_out is None:
            ids_out = torch.empty((nq, knn), dtype=torch.int32, device=queries.device)
        if d2_out is None:
            d2_out = torch.empty((nq, knn), dtype=torch.float32, device=queries.device)
        st = torch.cuda.current_stream(queries.device).cuda_stream if stream is None else stream
        check(self._L.sffg_knn_device(self._h, queries.data_ptr(), nq, int(knn), ids_out.data_ptr(), d2_out.data_ptr(), st))
        return ids_out, d2_out

    def radiusSearch(self, queries, radius_sq: float):
        """-> (counts int32[nq], offsets int64[nq+1], ids int32[total], d2 float32[total]); row i = ids[offsets[i]:offsets[i+1]]"""
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32).reshape(-1, self.dim))
        nq = len(q)
        counts = np.zeros(nq, dtype=np.int32)
        total = C.c_int64(0)
        if nq == 0:
            return counts, np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.float32)
        check(self._L.sffg_radius(self._h, _ptr(q), nq, float(radius_sq), _ptr(counts), None, None, 0, C.byref(total)))
        ids = np.empty(max(total.value, 1), dtype=np.int32)
        d2 = np.empty(max(total.value, 1), dtype=np.float32)
        check(self._L.sffg_radius(self._h, _ptr(q), nq, float(radius_sq), _ptr(counts), _ptr(ids), _ptr(d2), total.value, C.byref(total)))
        offsets = np.zeros(nq + 1, dtype=np.int64)
        np.cumsum(counts, out=offsets[1:])
        return counts, offsets, ids[: total.value], d2[: total.value]
