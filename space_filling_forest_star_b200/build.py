"""In-tree build of libsffg.so (hand-written CUDA for sm_100a + the C++ host side) with plain nvcc.

The shared object lands next to this file so that it travels with the repository snapshot; nothing is JIT-compiled
and nothing is installed into site-packages.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libsffg.so"
SOURCES = ["sffg_api.cu", "collide_kernels.cu", "clearance_grid.cu", "knn_kernels.cu", "knn_pruned.cu", "bvh_device.cu", "bvh_build.cpp", "mesh_loader.cpp"]
HEADERS = ["common.h", "collide_kernels.cuh", "clearance_grid.cuh", "cuda_handles.h", "knn_kernels.cuh", "knn_common.cuh", "knn_pruned.cuh", "bvh_device.cuh", "../../include/sffg.h"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: libsffg.so cannot be built (there is no CPU fallback)")


def is_stale() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    return any((CSRC / f).resolve().stat().st_mtime > t for f in SOURCES + HEADERS)


def build_native(force: bool = False, verbose: bool = False) -> Path:
    """Compile every CUDA/C++ source of the engine for sm_100a into space_filling_forest_star_b200/libsffg.so."""
    if not force and not is_stale():
        return LIB
    host_cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++"
    cmd = [_nvcc(), "-O3", "-std=c++17", *ARCH, "-lineinfo", "-ccbin", host_cxx,
           "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-cudart", "static",
           "-o", str(LIB), *[str(CSRC / s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB


HOST_SRC = PKG / "host" / "sff_planner.cpp"
HOST_BIN = PKG / "host" / "sff_planner"


def build_host(force: bool = False) -> Path:
    """The restructured (batched) planner host: plain C++17 on top of the C ABI, linked against libsffg.so."""
    lib = build_native()
    newest = max([f.stat().st_mtime for f in HOST_SRC.parent.glob("*.h")] + [HOST_SRC.stat().st_mtime, lib.stat().st_mtime])
    if not force and HOST_BIN.exists() and HOST_BIN.stat().st_mtime > newest:
        return HOST_BIN
    cxx = "/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++"
    cmd = [cxx, "-std=c++17", "-O2", "-Wall", "-I", str(PKG.parent / "include"), str(HOST_SRC), "-L", str(PKG), "-l:libsffg.so",
           "-Wl,-rpath,$ORIGIN/..", "-o", str(HOST_BIN)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build failed:\n" + res.stdout + res.stderr)
    return HOST_BIN


if __name__ == "__main__":
    import sys
    print(build_native(force=True, verbose="-v" in sys.argv))
    print(build_host(force=True))
