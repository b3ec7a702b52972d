// collide_kernels.cuh -- device-side view of an environment + launch wrappers (implemented in collide_kernels.cu)
#pragma once
#include <cuda_runtime.h>

#include "common.h"

namespace sffg {

// Device view of the clearance grid (built by clearance_grid.cu): n[0] * n[1] * n[2] cubic cells of edge h from the
// corner o, cell (ix, iy, iz) at index (iz * n[1] + iy) * n[0] + ix.  n[0] == 0 means "no grid": every other field is
// then unset.
//   bits     1 bit per cell: set when some obstacle triangle may lie within the robot's bounding radius of a robot origin
//            in the cell; clear proves every pose with its origin in the cell collision free
//   planes   1 word per cell: a separating-plane record (direction index in the low 5 bits, offset above them, see
//            plane_says_free); kNoPlane for unmarked cells
//   witness  1 int2 per cell: the two triangles (leaf order, -1 for none) that mark the cell with their points nearest
//            its centre, which phase B tries before the walk (contact probe); null when the probe is off
//   plane_pad  absolute part of the plane test's margin, rounded up (see clearance_margins in clearance_grid.cu)
// (The fields the pose kernels read keep the order they had as loose EnvDev fields: that order leaves their code as it was.)
struct GridDev {
  const unsigned *bits;
  float o[3];
  float inv_h;   // float(1 / h), rounded from double
  int n[3];
  const unsigned *planes;
  float plane_pad;
  float h;
  const int2 *witness;
};

__host__ __device__ __forceinline__ long long cell_count(const GridDev &g) { return (long long)g.n[0] * g.n[1] * g.n[2]; }
// The index of cell (ix, iy, iz).
__device__ __forceinline__ unsigned cell_index(const GridDev &g, unsigned ix, unsigned iy, unsigned iz) {
  return (iz * (unsigned)g.n[1] + iy) * (unsigned)g.n[0] + ix;
}
// The cell that holds position (x, y, z), or -1 outside the grid.
__device__ __forceinline__ int grid_cell(const GridDev &g, float x, float y, float z) {
  const float fx = (x - g.o[0]) * g.inv_h, fy = (y - g.o[1]) * g.inv_h, fz = (z - g.o[2]) * g.inv_h;
  if (!(fx >= 0.f && fy >= 0.f && fz >= 0.f && fx < (float)g.n[0] && fy < (float)g.n[1] && fz < (float)g.n[2])) return -1;
  return (int)cell_index(g, (unsigned)fx, (unsigned)fy, (unsigned)fz);
}
// The centre of cell (ix, iy, iz), and of the cell at `cell`.
__device__ __forceinline__ void cell_centre(const GridDev &g, int ix, int iy, int iz, float p[3]) {
  p[0] = g.o[0] + (ix + 0.5f) * g.h;
  p[1] = g.o[1] + (iy + 0.5f) * g.h;
  p[2] = g.o[2] + (iz + 0.5f) * g.h;
}
__device__ __forceinline__ void cell_centre(const GridDev &g, long long cell, float p[3]) {
  cell_centre(g, (int)(cell % g.n[0]), (int)(cell / g.n[0] % g.n[1]), (int)(cell / ((long long)g.n[0] * g.n[1])), p);
}

// Plane records: the 26 integer directions m in {-1,0,1}^3 \ {0}, d = 9 (mz + 1) + 3 (my + 1) + (mx + 1); d = 13 (m = 0)
// is the "no plane" record, whose offset is -FLT_MAX so that no pose passes it.
constexpr int kNoPlaneDir = 13;
constexpr unsigned kNoPlane = 0x80800000u | kNoPlaneDir;   // float_to_ordered(-FLT_MAX) = 0x80800000, low 5 bits clear
__device__ __forceinline__ void plane_dir(int d, float *m) {
  m[0] = (float)(d % 3 - 1);
  m[1] = (float)(d / 3 % 3 - 1);
  m[2] = (float)(d / 9 - 1);
}

struct EnvDev {
  const float4 *slots;      // 2 float4 per child slot, kWide slots per node
  const float4 *top;        // <= 32 slots: a cut through the top of the hierarchy, tested by all lanes in step 0
  int n_top;
  int n_stage_max;          // leading nodes (breadth-first order) a CTA may stage in shared memory; fixes the smem layout
  const float4 *tris32;     // 3 float4 per obstacle triangle (BVH leaf order); p[0].w = representation error bound
  const double *tris64;     // 9 doubles per obstacle triangle (BVH leaf order) -- exact stage
  const RobotTri *robot;    // n_robot records (FP32, robot frame)
  const double *robot64;    // 9 doubles per robot triangle -- exact stage
  int n_robot;
  int n_obst;
  float root_c[3], root_h[3];   // obstacle AABB, centre / half extents (outward rounded)
  float rob_c[3], rob_h[3];     // robot AABB in the robot frame (outward rounded)
  float rob_radius;             // max |robot vertex| about the robot origin (rounded up)
  GridDev grid;                 // clearance grid over the obstacle AABB dilated by rob_radius
  const float4 *rob_verts;      // distinct robot vertices (nearest floats); null above kPlaneVertCap: the robot box stands in
  int n_rob_verts;
  unsigned long long *counters; // 5 x u64 (may be null): poses, past_root, box_tests, pair_tests, exact_tests
  int *status;                  // device int, set non-zero on traversal-stack overflow
  unsigned int *work_counter;   // persistent-kernel work distribution: never reset, units are (fetched value - work_base)
  unsigned int work_base;
};

// destinations of a verdict: the local output plus (multi-GPU) the same offset in every peer's gathered buffer, mapped into
// this process through CUDA IPC -- the kernel stores each verdict to all of them, so the result all-gather rides on the
// kernel's own stores over NVLink instead of being a separate collective
constexpr int kMaxPeers = 8;
struct OutSet {
  uint8_t *p[kMaxPeers];
  int n;
};
struct FlagSet {
  unsigned *p[kMaxPeers];   // p[r] = rank r's flag array (kMaxPeers words), p[me] is local
  int n, me;
};
// completion signalling fused into the gather kernel: before touching the destinations every CTA waits until all ranks
// have published an epoch >= wait_epoch (their earlier results have been consumed, see sffg.h); the last CTA to finish
// publishes signal_epoch to every rank.  flags.n == 0 disables both.
struct GatherSync {
  FlagSet flags;
  unsigned signal_epoch, wait_epoch;
  unsigned *done_counter;   // local word, zero between launches
};

struct LaunchCfg {
  int sm_count;
  int blocks_per_sm;
};

// verdict_out[i] = 1 if the robot at poses[i] touches the obstacle soup
// pose_fmt: 0 = float [n][6] x y z yaw pitch roll, 1 = double [n][6], 2 = double [n][12] (R row-major, then T)
cudaError_t launch_collide_poses(const EnvDev &env, const void *d_poses, int pose_fmt, int64_t n,
                                 uint8_t *d_verdict, cudaStream_t stream, const LaunchCfg &cfg, bool count,
                                 unsigned *work_base_io);
// same, verdict i goes to outs.p[r][i] for every r < outs.n (peer-store gather)
cudaError_t launch_collide_poses_gather(const EnvDev &env, const void *d_poses, int pose_fmt, int64_t n, const OutSet &outs,
                                        const GatherSync &sync, cudaStream_t stream, const LaunchCfg &cfg, bool count,
                                        unsigned *work_base_io);
// all ranks' stores of the kernels enqueued before this call are visible on every rank once the barrier kernel has run on
// every rank: signal (st.release.sys into every peer's flag word) + wait (ld.acquire.sys on the own flag words), bounded
// by a 10 s timeout that raises the env status instead of hanging the GPU
cudaError_t launch_peer_barrier(const FlagSet &flags, unsigned epoch, bool signal, int *d_status, cudaStream_t stream);

// dist[i] = separation distance robot <-> obstacle soup of poses[i], capped at max_dist (0 exactly on contact); points
// (optional, [n][6]) = nearest robot point then nearest obstacle point, world frame, NaN unless 0 < dist < max_dist.
// pose_fmt 0 or 1 (the matrix form is not supported: cudaErrorInvalidValue)
cudaError_t launch_distance_poses(const EnvDev &env, const void *d_poses, int pose_fmt, int64_t n, double max_dist,
                                  double *d_dist, double *d_points, cudaStream_t stream, const LaunchCfg &cfg,
                                  unsigned *work_base_io);

cudaError_t launch_check_edges(const EnvDev &env, const double *d_starts, const double *d_ends, int64_t m,
                               double sample_dist, int rot_mode, uint8_t *d_free, int32_t *d_first_hit,
                               cudaStream_t stream, const LaunchCfg &cfg, bool count, unsigned *work_base_io,
                               int *d_fh_scratch /* m ints, or null to force one warp per edge */);

// dist[e] = minimum over the samples of edge e (those launch_check_edges tests) of the pose distance capped at max_dist,
// index[e] (optional) = the lowest sample reporting it (the first hit on contact, 0 when dist == max_dist), points
// (optional, [m][6]) as for launch_distance_poses at that sample.  Enqueues launch_check_edges into the scratch first.
struct EdgeDistScratch {
  uint8_t *free;        // m free flags of the verdict launch
  int32_t *first_hit;   // m first hits of the verdict launch
  int *fh;              // m ints for the verdict launch's split edges, or null (one warp per edge)
  void *recs;           // distance_edges_rec_bytes(m, cfg) bytes for the distance kernel's split edges, or null
};
size_t distance_edges_rec_bytes(int64_t m, const LaunchCfg &cfg);
cudaError_t launch_distance_edges(const EnvDev &env, const double *d_starts, const double *d_ends, int64_t m, double sample_dist,
                                  int rot_mode, double max_dist, double *d_dist, int32_t *d_index, double *d_points,
                                  cudaStream_t stream, const LaunchCfg &cfg, unsigned *work_base_io,
                                  const EdgeDistScratch &scr);

// continuous check of the motion start -> end of every edge by conservative advancement on the pose distance
// (include/sffg.h): clear[e] = 1 when every pose of the motion is certified at distance >= margin / 2; otherwise t[e] is
// where the lowest stopped piece stopped and dist[e] the pose distance there (< margin).  t and dist may be null.
struct SweepScratch {
  int *stop;    // m ints for the edges split over several warps, or null (one warp per edge)
  void *recs;   // sweep_edges_rec_bytes(m, cfg) bytes for the split edges' per-warp records, or null
};
size_t sweep_edges_rec_bytes(int64_t m, const LaunchCfg &cfg);
cudaError_t launch_sweep_edges(const EnvDev &env, const double *d_starts, const double *d_ends, int64_t m, int rot_mode,
                               double margin, uint8_t *d_clear, double *d_t, double *d_dist, cudaStream_t stream,
                               const LaunchCfg &cfg, unsigned *work_base_io, const SweepScratch &scr);

cudaError_t launch_gen_poses(uint64_t seed, uint64_t first, int64_t n, const float range[6], float *d_out,
                             cudaStream_t stream);

size_t collide_smem_bytes(int n_robot, int n_stage_max);
// Staged hierarchy per CTA at most: the first three levels (1 + 8 + 64 nodes, 18.7 KB).  Shared memory and L1 come out
// of the same 256 KB per SM; 384 staged nodes (96 KB) measured no faster than 73 because L1 holds the deeper levels
// and the triangles (profiles/r02_collide_variants.md).
#ifndef SFFG_STAGE_NODES
#define SFFG_STAGE_NODES 73
#endif
constexpr int kStageNodesCap = SFFG_STAGE_NODES;

// Robots with more distinct vertices than this take the support of their box in the plane test (robot_small has 8,
// robot_cyl_small 64).  One FMA chain per vertex per pose past the grid bit.
constexpr int kPlaneVertCap = 16;

}  // namespace sffg
