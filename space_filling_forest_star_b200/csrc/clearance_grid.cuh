// clearance_grid.cuh -- the clearance grid of an environment: its sizing, its build and its device arrays (implemented in
// clearance_grid.cu).  The pose and edge kernels read it through GridDev (collide_kernels.cuh).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "collide_kernels.cuh"
#include "cuda_handles.h"

namespace sffg {

// Owner of one clearance grid.  A default-constructed owner holds no grid (view.n[0] == 0).
struct ClearanceGrid {
  DevPtr<unsigned> bits, planes;
  DevPtr<int2> witness;
  GridDev view{};
  size_t bytes = 0;     // device memory held
  int64_t cells = 0;
  double h = 0;         // cell edge
};

// Builds the clearance grid of the obstacle triangles `d_tris32` (n_tris records of 3 float4, leaf order) inside the box
// [root_lo, root_hi] for a robot of bounding radius `rho`, on `stream`, and waits for it.  The grid covers the box
// dilated by rho with cubic cells of edge rho / 4, grown until there are at most 2^24 cells.  Every cell gets its bit and
// its plane record and, unless SFFG_WITNESS=0, its two contact witnesses.  There is no grid without obstacles or with
// SFFG_CLEARANCE_GRID=0.  `*out` receives the grid on success and is left alone otherwise.
cudaError_t build_clearance_grid(const float4 *d_tris32, int64_t n_tris, const double root_lo[3], const double root_hi[3],
                                 double rho, cudaStream_t stream, ClearanceGrid *out);

}  // namespace sffg
