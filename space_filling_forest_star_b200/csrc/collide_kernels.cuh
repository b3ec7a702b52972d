// collide_kernels.cuh -- device-side view of an environment + launch wrappers (implemented in collide_kernels.cu)
#pragma once
#include <cuda_runtime.h>

#include "common.h"

namespace sffg {

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
  // free-space (clearance) grid: bit = 1 -> some obstacle triangle may be within rob_radius of a robot origin placed in
  // that cell; bit = 0 -> every pose with its origin in the cell is collision free.  grid_n[0] == 0 disables it.
  const unsigned *clear_bits;
  float grid_o[3];
  float grid_inv_h;
  int grid_n[3];
  // one separating plane per grid cell (word = direction index in the low 5 bits, offset above them, see plane_says_free),
  // set whenever clear_bits is
  const unsigned *planes;
  float plane_pad;              // absolute part of the plane test's margin, rounded up
  const float4 *rob_verts;      // distinct robot vertices (nearest floats); null above kPlaneVertCap: the robot box stands in
  int n_rob_verts;
  // per grid cell, the two triangles (leaf order, -1 for none) that mark it with their points nearest the cell centre:
  // phase B tries them before the walk (contact probe).  Null when the grid or the probe is off.
  const int2 *witness;
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

cudaError_t launch_check_edges(const EnvDev &env, const double *d_starts, const double *d_ends, int64_t m,
                               double sample_dist, int rot_mode, uint8_t *d_free, int32_t *d_first_hit,
                               cudaStream_t stream, const LaunchCfg &cfg, bool count, unsigned *work_base_io,
                               int *d_fh_scratch /* m ints, or null to force one warp per edge */);

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

// Marks every cell whose centre is within `reach` of an obstacle triangle (one warp per triangle) in `d_bits`, and picks
// each marked cell's plane record (`d_planes`, one word per cell).  `d_scratch` holds `scratch_words` ints (at least one
// per cell); the 26 plane directions take ceil(26 / (scratch_words / cells)) passes over the triangles.
// With `d_witness` (one int2 per cell) it then stores each cell's two contact witnesses -- of the triangles that mark the cell,
// the two nearest its centre -- in two more passes over the triangles; that needs scratch_words >= 2 * cells.
cudaError_t launch_build_clearance(const float4 *d_tris32, int n_tris, const float origin[3], float h, const int n[3], float reach,
                                   unsigned *d_bits, unsigned *d_planes, int2 *d_witness, int *d_scratch, size_t scratch_words,
                                   cudaStream_t stream);

// Robots with more distinct vertices than this take the support of their box in the plane test (robot_small has 8,
// robot_cyl_small 64).  One FMA chain per vertex per pose past the grid bit.
constexpr int kPlaneVertCap = 16;

}  // namespace sffg
