// common.h -- internal declarations shared by the host-side C++ and the CUDA translation units of libsffg.so
#pragma once
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/sffg.h"

namespace sffg {

// ---- error reporting (thread-local text behind sffg_last_error) ------------------------------------------
void set_error(const std::string &msg);
int fail(int code, const std::string &msg);

// ---- device-side flattened structures ---------------------------------------------------------------------
constexpr int kWide = 8;              // children per BVH node
constexpr int32_t kEmptyChild = 0x7fffffff;

// One child slot of a wide node = two float4 (32 B).  8 slots of one node are contiguous (256 B), so the 8 lanes
// that test one node issue two fully-coalesced 128-B loads.
//   a = (cx, cy, cz, bits(child))      child >= 0: wide-node index; child < 0: ~triangle index; kEmptyChild: unused
//   b = (hx, hy, hz, 0)                half extents, rounded outward
struct ChildSlot {
  float cx, cy, cz;
  int32_t child;
  float hx, hy, hz;
  float pad;
};
static_assert(sizeof(ChildSlot) == 32, "ChildSlot must be 32 bytes");

// FP32 obstacle triangle for the conservative SAT stage: 3 x float4 (48 B).
//   w of vertex 0 = representation error bound (max |double - float| over the 9 coordinates, rounded up)
struct TriF32 {
  float p[3][4];
};

// Robot triangle record, robot frame, FP32 (precomputed from double on the host).
struct RobotTri {
  float q[3][3];      // vertices (nearest float of the double vertices)
  float f[3][3];      // edges  f1 = q2-q1, f2 = q3-q2, f3 = q1-q3
  float m[3];         // normal f1 x f2
  float h[3][3];      // in-plane edge normals f_k x m
  float m_lo, m_hi;   // projection interval of the TRUE (double) triangle on the float axis m, rounded outward
  float h_lo[3], h_hi[3];   // same for the three h axes
  float lo[3], hi[3]; // AABB in the robot frame (rounded outward)
  float qmax;         // max |coordinate| of the three vertices (rounded up)
  float pad[7];       // 52 words per record: stride 20 mod 32 banks -> 6 consecutive records never share a bank
};
static_assert(sizeof(RobotTri) % 16 == 0, "RobotTri must be 16-byte granular");

struct HostBvh {
  std::vector<ChildSlot> slots;       // n_nodes * kWide
  std::vector<int32_t> tri_order;     // BVH leaf order -> original triangle index
  int depth = 0;
  double root_lo[3] = {0, 0, 0}, root_hi[3] = {0, 0, 0};
  std::vector<int> level_base, level_count;   // nodes are stored breadth-first: level l = [level_base[l], +level_count[l])
};

// picks <= 32 slots forming a cut through the top of the hierarchy (largest boxes expanded first)
void top_cut(const HostBvh &bvh, std::vector<ChildSlot> *out);

// builds an 8-wide AABB BVH over a double triangle soup; leaves are single triangles; slots refer to triangles by
// their position in tri_order
void build_wide_bvh(const double *tris, int64_t n, HostBvh *out);

// mesh loader (reference semantics), returns SFFG_* status
int load_mesh(const char *path, int is_obj, const double position[3], double scale, std::vector<double> *tris,
              double bbox[6]);

float round_up_f32(double v);     // smallest float >= v
float round_down_f32(double v);   // largest float <= v

#ifdef __CUDACC__
// Order-preserving float <-> int: the ints compare as the (non-NaN) floats do, so integer min / max reductions and
// atomics can bound floats.  Non-negative floats keep their bits, negative ones flip their magnitude bits.
__host__ __device__ __forceinline__ int float_to_ordered(float f) {
  int i;
  memcpy(&i, &f, sizeof i);
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__host__ __device__ __forceinline__ float ordered_to_float(int i) {
  i = i >= 0 ? i : i ^ 0x7fffffff;
  float f;
  memcpy(&f, &i, sizeof f);
  return f;
}
#endif

}  // namespace sffg
