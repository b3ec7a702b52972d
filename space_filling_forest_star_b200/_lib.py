"""ctypes binding of libsffg.so -- the C ABI declared in include/sffg.h.

There is no Python/CPU implementation behind these symbols: if the shared object is missing it is built with nvcc,
and if no sm_100 GPU is present every compute call raises :class:`SffgError` (SFFG_ERR_NO_DEVICE).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

SFFG_OK = 0
ERR_NAMES = {1: "NO_DEVICE", 2: "CUDA", 3: "ARG", 4: "IO", 5: "CAPACITY", 6: "DOMAIN", 7: "INTERNAL"}
ROT_REFERENCE, ROT_INTERPOLATE = 0, 1
BUILD_AUTO, BUILD_HOST, BUILD_DEVICE = 0, 1, 2
MAX_K = 128


class SffgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"SFFG_ERR_{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


class EnvInfo(C.Structure):
    _fields_ = [("n_obst_tris", C.c_int64), ("n_robot_tris", C.c_int64), ("n_nodes", C.c_int64), ("depth", C.c_int32),
                ("device_bytes", C.c_int64), ("build_ms", C.c_double), ("grid_cells", C.c_int64), ("grid_cell_size", C.c_double),
                ("built_on_device", C.c_int32)]


class Counters(C.Structure):
    _fields_ = [("poses", C.c_int64), ("poses_past_root", C.c_int64), ("box_tests", C.c_int64), ("pair_tests", C.c_int64),
                ("exact_tests", C.c_int64), ("traversal_steps", C.c_int64), ("triangle_passes", C.c_int64),
                ("triangles_transformed", C.c_int64), ("exact_run", C.c_int64), ("poses_past_grid", C.c_int64)]


# name -> (restype, argtypes); mirrors include/sffg.h one to one (tests/test_abi.py checks the header against this)
_p = C.c_void_p
SIGNATURES = {
    "sffg_version": (C.c_int, []),
    "sffg_last_error": (C.c_char_p, []),
    "sffg_init": (C.c_int, [C.c_int]),
    "sffg_device_count": (C.c_int, []),
    "sffg_mesh_load": (C.c_int, [C.c_char_p, C.c_int, _p, C.c_double, C.POINTER(_p), C.POINTER(C.c_int64), _p]),
    "sffg_free": (None, [_p]),
    "sffg_env_create": (C.c_int, [_p, C.c_int64, _p, C.c_int64, C.POINTER(_p)]),
    "sffg_env_destroy": (C.c_int, [_p]),
    "sffg_env_create_ex": (C.c_int, [_p, C.c_int64, _p, C.c_int64, C.c_int, C.POINTER(_p)]),
    "sffg_env_set_obstacles": (C.c_int, [_p, _p, C.c_int64, C.c_int]),
    "sffg_env_refit_obstacles": (C.c_int, [_p, _p, C.c_int64]),
    "sffg_env_info": (C.c_int, [_p, C.POINTER(EnvInfo)]),
    "sffg_collide_poses_f32": (C.c_int, [_p, _p, C.c_int64, _p]),
    "sffg_collide_poses_f64": (C.c_int, [_p, _p, C.c_int64, _p]),
    "sffg_collide_transforms_f64": (C.c_int, [_p, _p, C.c_int64, _p]),
    "sffg_collide_poses_device": (C.c_int, [_p, _p, C.c_int, C.c_int64, _p, _p]),
    "sffg_distance_poses": (C.c_int, [_p, _p, C.c_int, C.c_int64, C.c_double, _p, _p]),
    "sffg_distance_poses_device": (C.c_int, [_p, _p, C.c_int, C.c_int64, C.c_double, _p, _p, _p]),
    "sffg_distance_edges": (C.c_int, [_p, _p, _p, C.c_int64, C.c_double, C.c_int, C.c_double, _p, _p, _p]),
    "sffg_distance_edges_device": (C.c_int, [_p, _p, _p, C.c_int64, C.c_double, C.c_int, C.c_double, _p, _p, _p, _p]),
    "sffg_sweep_edges": (C.c_int, [_p, _p, _p, C.c_int64, C.c_int, C.c_double, _p, _p, _p]),
    "sffg_sweep_edges_device": (C.c_int, [_p, _p, _p, C.c_int64, C.c_int, C.c_double, _p, _p, _p, _p]),
    "sffg_peer_buffer_create": (C.c_int, [C.c_int64, C.POINTER(_p), _p]),
    "sffg_peer_buffer_open": (C.c_int, [_p, C.POINTER(_p)]),
    "sffg_peer_buffer_close": (C.c_int, [_p]),
    "sffg_peer_buffer_destroy": (C.c_int, [_p]),
    "sffg_collide_poses_gather_device": (C.c_int, [_p, _p, C.c_int, C.c_int64, _p, C.c_int, _p]),
    "sffg_collide_poses_gather_sync_device": (C.c_int, [_p, _p, C.c_int, C.c_int64, _p, _p, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                                       _p, _p]),
    "sffg_peer_wait_device": (C.c_int, [_p, _p, C.c_int, C.c_int, C.c_uint32, _p]),
    "sffg_peer_barrier_device": (C.c_int, [_p, _p, C.c_int, C.c_int, C.c_uint32, _p]),
    "sffg_check_edges": (C.c_int, [_p, _p, _p, C.c_int64, C.c_double, C.c_int, _p, _p]),
    "sffg_check_moves": (C.c_int, [_p, _p, _p, C.c_int64, C.c_double, C.c_int, _p]),
    "sffg_check_edges_device": (C.c_int, [_p, _p, _p, C.c_int64, C.c_double, C.c_int, _p, _p, _p]),
    "sffg_env_enable_counters": (C.c_int, [_p, C.c_int]),
    "sffg_env_sync_check": (C.c_int, [_p]),
    "sffg_env_read_counters": (C.c_int, [_p, C.POINTER(Counters)]),
    "sffg_gen_poses_device": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, _p, _p, _p]),
    "sffg_index_create": (C.c_int, [C.c_int, C.POINTER(_p)]),
    "sffg_index_destroy": (C.c_int, [_p]),
    "sffg_index_add": (C.c_int, [_p, _p, C.c_int64]),
    "sffg_index_add_device": (C.c_int, [_p, _p, C.c_int64, _p]),
    "sffg_index_add_multi": (C.c_int, [_p, _p, C.c_int, _p]),
    "sffg_index_size": (C.c_int64, [_p]),
    "sffg_knn": (C.c_int, [_p, _p, C.c_int64, C.c_int, _p, _p]),
    "sffg_knn_device": (C.c_int, [_p, _p, C.c_int64, C.c_int, _p, _p, _p]),
    "sffg_knn_gather_device": (C.c_int, [_p, _p, C.c_int64, C.c_int, _p, _p, C.c_int, _p]),
    "sffg_knn_multi": (C.c_int, [_p, _p, C.c_int, _p, C.c_int, _p, _p]),
    "sffg_radius": (C.c_int, [_p, _p, C.c_int64, C.c_float, _p, _p, _p, C.c_int64, C.POINTER(C.c_int64)]),
    # asynchronous forms (begin enqueues, the matching end completes)
    "sffg_radius_begin": (C.c_int, [_p, _p, C.c_int64, C.c_float, _p, _p, _p, C.c_int64, C.POINTER(C.c_int64)]),
    "sffg_knn_multi_begin": (C.c_int, [_p, _p, C.c_int, _p, C.c_int, _p, _p]),
    "sffg_index_add_multi_begin": (C.c_int, [_p, _p, C.c_int, _p]),
    "sffg_index_end": (C.c_int, [_p]),
    "sffg_check_edges_begin": (C.c_int, [_p, _p, _p, C.c_int64, C.c_double, C.c_int, _p, _p]),
    "sffg_check_moves_begin": (C.c_int, [_p, _p, _p, C.c_int64, C.c_double, C.c_int, _p]),
    "sffg_env_end": (C.c_int, [_p]),
}

_lib = None


def lib_path() -> Path:
    return _build.LIB


def load() -> C.CDLL:
    """Load (building first if needed) libsffg.so.  Raises if it cannot be built -- never falls back."""
    global _lib
    if _lib is None:
        import os
        variant = os.environ.get("SFFG_LIB")   # another build for A/B measurements; the default is the in-tree library
        path = Path(variant) if variant else _build.build_native()
        L = C.CDLL(str(path))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError here = header and library out of sync
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != SFFG_OK:
        raise SffgError(rc, load().sffg_last_error().decode("utf-8", "replace"))
