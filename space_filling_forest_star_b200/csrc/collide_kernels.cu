// collide_kernels.cu -- sm_100a kernels for pose and edge collision verdicts.
//
// Replaces the inside of Environment<T>::Collide -> Obstacle<T>::Collide -> RAPID_Collide
// (reference src/environment.h:306-316, :269-276) and of Solver<T,R>::isPathFree (src/problemStruct.h:154-168).
//
// Execution model (one warp = one pose at a time):
//   phase A  lane-per-pose: load 32 poses, cull the robot's bounding sphere against the obstacle AABB and the clearance
//            grid's cell bit, build R, test the robot against the cell's separating plane
//   phase B  warp-per-pose for the survivors:
//            - 8-wide AABB BVH (breadth-first node order); the top of the hierarchy -- a <=32-box cut tested by all lanes
//              in step 0 and the first three levels of nodes -- is staged in shared memory once per CTA; warp-shared DFS
//              stack in shared memory; each step pops up to 4 nodes and the 32 lanes test the 4x8 child boxes against
//              the robot's oriented box (6-axis conservative SAT)
//            - surviving leaf triangles are transformed into the robot frame (as RAPID does) lane-per-triangle,
//              then lane-per-(obstacle triangle, robot triangle) pair runs the 17-axis separating-axis test in FP32
//              as a *certificate* test: an axis only counts when its gap exceeds a rigorous rounding bound
//            - pairs the lane-per-pair stage leaves open get the 9 edge x edge axes (three pairs per pass on ten lanes
//              each) and the 6 contact certificates cooperatively: the certificates first (five pairs per pass on six
//              lanes each) in the pose verdict kernel, the axes first in every other kernel
//            - pairs without an FP32 certificate are decided by the exact stage: the same 17 axes in FP64 with the
//              operation order of the CPU oracle, one axis per lane; __all_sync gives the pair verdict
//            - __ballot/__any early-out on the first confirmed contact (verdict-equivalent to RAPID's ALL_CONTACTS
//              because the caller only looks at num_contacts != 0)
// The result equals "OR over all triangle pairs of the double-precision SAT" -- the oracle's ground truth.
#include <algorithm>
#include <cfloat>
#include <cstdint>
#include <mutex>

#include <math_constants.h>

#include "collide_kernels.cuh"

namespace sffg {
namespace {

constexpr int kWarpsPerBlock = 16;
constexpr int kThreads = kWarpsPerBlock * 32;
constexpr int kMinBlocksPerSm = 1;   // __launch_bounds__ of the pose and edge kernels
constexpr int kStackCap = 384;   // node ids pending for one pose
constexpr int kTriCap = 64;      // candidate triangles pending for one pose
constexpr int kCandCap = 192;    // candidate triangles of one group of edge samples (swept-box traversal)
constexpr unsigned kFull = 0xffffffffu;
constexpr float kEpsBox = 1.52587890625e-05f;   // 2^-16, relative slack of the box culls   (>= 140 ulp, see DESIGN.md)
constexpr float kEpsSat = 1.52587890625e-05f;   // 2^-16, relative position error of the FP32 SAT stage
// Both budgets include the FP32 rotation's error against FillRotationMatrix of the pose's own angles: every sin / cos
// within 2^-21 of the exact value (sincosf <= 2 ulp, plus up to 2^-23 from narrowing a double angle |a| <= float(pi) to
// float; wider double angles are never narrowed, see sincos_narrow), every entry of R within 2^-19.  Unbounded, the
// narrowing alone would be 2^-15 at |a| ~ 1000 rad, and an FP32 certificate could be issued for the wrong pose.

struct XTri {        // obstacle triangle in the robot frame (FP32); 13 words = odd stride, bank-conflict free
  float v[9];
  float err;         // absolute position error bound of these 9 values
  float mabs;        // max |v|
  int tri;           // triangle index (leaf order) for the exact stage
  int pad;
};

struct WarpScratch {
  int stack[kStackCap];
  int tri[kTriCap];
  union {              // the swept-box candidate list serves only the kernels without the contact probe, and vice versa
    int cand[kCandCap];
    int2 wit[32];      // each lane's contact witnesses from phase A ({-1, -1}: none), read by phase B's probe
  };
  XTri xt[32];
};

// what a CTA stages once: the robot records, the top cut and the first nodes of the (breadth-first) hierarchy
struct CtaShared {
  const RobotTri *rob;
  const float4 *top;     // 2 float4 per slot, E.n_top slots
  const float4 *nodes;   // 16 float4 per node, n_stage nodes
  int n_stage;
};
constexpr int kTopSlots = 32;

// ---------------------------------------------------------------------------------------------------------
// FP32 certificate SAT
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float min3f(float a, float b, float c) { return fminf(a, fminf(b, c)); }
__device__ __forceinline__ float max3f(float a, float b, float c) { return fmaxf(a, fmaxf(b, c)); }

// true when axis (ax,ay,az) separates the two triangles by more than the rounding bound
__device__ __forceinline__ bool axis_certifies(float ax, float ay, float az, const float *p, const float (*q)[3],
                                               float errpos) {
  float P1 = ax * p[0] + ay * p[1] + az * p[2];
  float P2 = ax * p[3] + ay * p[4] + az * p[5];
  float P3 = ax * p[6] + ay * p[7] + az * p[8];
  float Q1 = ax * q[0][0] + ay * q[0][1] + az * q[0][2];
  float Q2 = ax * q[1][0] + ay * q[1][1] + az * q[1][2];
  float Q3 = ax * q[2][0] + ay * q[2][1] + az * q[2][2];
  float gap = fmaxf(min3f(P1, P2, P3) - max3f(Q1, Q2, Q3), min3f(Q1, Q2, Q3) - max3f(P1, P2, P3));
  float bound = (fabsf(ax) + fabsf(ay) + fabsf(az)) * errpos;
  return gap > bound;
}

// axis with a host-precomputed (outward rounded) projection interval of the robot triangle
__device__ __forceinline__ bool axis_certifies_pre(const float *a, const float *p, float qlo, float qhi, float errpos) {
  float P1 = a[0] * p[0] + a[1] * p[1] + a[2] * p[2];
  float P2 = a[0] * p[3] + a[1] * p[4] + a[2] * p[5];
  float P3 = a[0] * p[6] + a[1] * p[7] + a[2] * p[8];
  float gap = fmaxf(min3f(P1, P2, P3) - qhi, qlo - max3f(P1, P2, P3));
  float bound = (fabsf(a[0]) + fabsf(a[1]) + fabsf(a[2])) * errpos;
  return gap > bound;
}

// Stage P1, lane-per-pair: the 8 most selective certificates -- AABB in the robot frame, the two face normals and the
// six in-plane edge normals (robot-side intervals precomputed on the host).
// Returns true when the pair is PROVEN disjoint; false = still open (stage P2 looks at it).
__device__ bool pair_quick_disjoint(const XTri &x, const RobotTri &rt) {
  const float *p = x.v;
  const float errpos = 2.0f * x.err + kEpsSat * fmaxf(x.mabs, rt.qmax);
  {
    float lo0 = min3f(p[0], p[3], p[6]) - errpos, hi0 = max3f(p[0], p[3], p[6]) + errpos;
    float lo1 = min3f(p[1], p[4], p[7]) - errpos, hi1 = max3f(p[1], p[4], p[7]) + errpos;
    float lo2 = min3f(p[2], p[5], p[8]) - errpos, hi2 = max3f(p[2], p[5], p[8]) + errpos;
    if (lo0 > rt.hi[0] || hi0 < rt.lo[0] || lo1 > rt.hi[1] || hi1 < rt.lo[1] || lo2 > rt.hi[2] || hi2 < rt.lo[2])
      return true;
  }
  if (axis_certifies_pre(rt.m, p, rt.m_lo, rt.m_hi, errpos)) return true;
  const float e0[3] = {p[3] - p[0], p[4] - p[1], p[5] - p[2]}, e1[3] = {p[6] - p[3], p[7] - p[4], p[8] - p[5]};
  const float n0 = e0[1] * e1[2] - e0[2] * e1[1], n1 = e0[2] * e1[0] - e0[0] * e1[2], n2 = e0[0] * e1[1] - e0[1] * e1[0];
  if (axis_certifies(n0, n1, n2, p, rt.q, errpos)) return true;
#pragma unroll
  for (int k = 0; k < 3; ++k)
    if (axis_certifies_pre(rt.h[k], p, rt.h_lo[k], rt.h_hi[k], errpos)) return true;
  // obstacle in-plane edge normals e_i x n: what separates a robot lying in the plane of a big triangle but beyond an edge
  const float e2[3] = {p[0] - p[6], p[1] - p[7], p[2] - p[8]};
  if (axis_certifies(e0[1] * n2 - e0[2] * n1, e0[2] * n0 - e0[0] * n2, e0[0] * n1 - e0[1] * n0, p, rt.q, errpos)) return true;
  if (axis_certifies(e1[1] * n2 - e1[2] * n1, e1[2] * n0 - e1[0] * n2, e1[0] * n1 - e1[1] * n0, p, rt.q, errpos)) return true;
  if (axis_certifies(e2[1] * n2 - e2[2] * n1, e2[2] * n0 - e2[0] * n2, e2[0] * n1 - e2[1] * n0, p, rt.q, errpos)) return true;
  return false;
}

// ---------------------------------------------------------------------------------------------------------
// FP32 contact certificate.  A pair the separating-axis stage could not clear is usually a deep contact; proving it
// in FP32 saves the FP64 stage.  Sufficient condition: an edge of one triangle pierces the interior of the other --
// its endpoints lie strictly on opposite sides of the other triangle's plane and the three signed volumes
// [(c_k - a) x (c_{k+1} - a)] . (b - a) share a sign -- with every quantity clear of a rigorous error bound
// (positions are off by at most errpos; a bilinear / trilinear form of vectors bounded by 2M then moves by less than
// 150 * errpos * M^2, allotted 256).  Lane j < 6 checks one (edge, triangle) combination; any lane suffices.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool edge_pierces(const float *a, const float *b, const float *c0, const float *c1, const float *c2,
                                             float bound) {
  const float u[3] = {c1[0] - c0[0], c1[1] - c0[1], c1[2] - c0[2]}, v[3] = {c2[0] - c0[0], c2[1] - c0[1], c2[2] - c0[2]};
  const float n[3] = {u[1] * v[2] - u[2] * v[1], u[2] * v[0] - u[0] * v[2], u[0] * v[1] - u[1] * v[0]};
  const float da = n[0] * (a[0] - c0[0]) + n[1] * (a[1] - c0[1]) + n[2] * (a[2] - c0[2]);
  const float db = n[0] * (b[0] - c0[0]) + n[1] * (b[1] - c0[1]) + n[2] * (b[2] - c0[2]);
  if (!((da > bound && db < -bound) || (da < -bound && db > bound))) return false;
  const float d[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]};
  const float w0[3] = {c0[0] - a[0], c0[1] - a[1], c0[2] - a[2]}, w1[3] = {c1[0] - a[0], c1[1] - a[1], c1[2] - a[2]},
              w2[3] = {c2[0] - a[0], c2[1] - a[1], c2[2] - a[2]};
  const float v0 = (w0[1] * w1[2] - w0[2] * w1[1]) * d[0] + (w0[2] * w1[0] - w0[0] * w1[2]) * d[1] + (w0[0] * w1[1] - w0[1] * w1[0]) * d[2];
  const float v1 = (w1[1] * w2[2] - w1[2] * w2[1]) * d[0] + (w1[2] * w2[0] - w1[0] * w2[2]) * d[1] + (w1[0] * w2[1] - w1[1] * w2[0]) * d[2];
  const float v2 = (w2[1] * w0[2] - w2[2] * w0[1]) * d[0] + (w2[2] * w0[0] - w2[0] * w0[2]) * d[1] + (w2[0] * w0[1] - w2[1] * w0[0]) * d[2];
  return (v0 > bound && v1 > bound && v2 > bound) || (v0 < -bound && v1 < -bound && v2 < -bound);
}

// Stage P2, the pairs the lane-per-pair stage left open, in two kinds of cooperative pass (order: see triangle_stage):
//   pass c  six lanes per pair, up to five pairs per pass (lane 6g + c): the six edge-pierces-triangle contact certificates
//                                                                            -> any one proves the pose's contact
//   pass a  ten lanes per pair, three pairs per pass (lanes 0..9, 10..19, 20..29; k = lane % 10): lanes k < 9 evaluate
//           the nine edge x edge axes e_i x f_j                              -> pairs proven disjoint
// what neither decides goes to the FP64 exact stage
__device__ __forceinline__ bool open_pair_axis(const XTri &x, const RobotTri &rt, int k) {
  const float *p = x.v;
  const float errpos = 2.0f * x.err + kEpsSat * fmaxf(x.mabs, rt.qmax);
  const int i = k / 3, j = k - 3 * i, i1 = i == 2 ? 0 : i + 1;
  const float e[3] = {p[3 * i1] - p[3 * i], p[3 * i1 + 1] - p[3 * i + 1], p[3 * i1 + 2] - p[3 * i + 2]};
  const float ax = e[1] * rt.f[j][2] - e[2] * rt.f[j][1], ay = e[2] * rt.f[j][0] - e[0] * rt.f[j][2],
              az = e[0] * rt.f[j][1] - e[1] * rt.f[j][0];
  return axis_certifies(ax, ay, az, p, rt.q, errpos);
}
__device__ __forceinline__ bool open_pair_pierce(const XTri &x, const RobotTri &rt, int c) {
  const float M = fmaxf(x.mabs, rt.qmax);
  const float bound = 256.0f * (2.0f * x.err + kEpsSat * M) * M * M;
  const int ed = c < 3 ? c : c - 3, ed1 = ed == 2 ? 0 : ed + 1;
  const bool obst_edge = c < 3;
  const float *a = obst_edge ? x.v + 3 * ed : rt.q[ed], *b = obst_edge ? x.v + 3 * ed1 : rt.q[ed1];
  const float *c0 = obst_edge ? rt.q[0] : x.v, *c1 = obst_edge ? rt.q[1] : x.v + 3, *c2 = obst_edge ? rt.q[2] : x.v + 6;
  return edge_pierces(a, b, c0, c1, c2, bound);
}

// ---------------------------------------------------------------------------------------------------------
// FP64 exact stage -- operation order of oracle/sff_oracle.c (make_xform, xform_point, orc_tri_contact).
// Explicit *_rn intrinsics keep ptxas from contracting a*b+c into an FMA, which the CPU oracle does not do.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double ddot(const double *a, const double *b) {
  return dadd(dadd(dmul(a[0], b[0]), dmul(a[1], b[1])), dmul(a[2], b[2]));
}
__device__ __forceinline__ void dcross(double *r, const double *a, const double *b) {
  r[0] = dsub(dmul(a[1], b[2]), dmul(a[2], b[1]));
  r[1] = dsub(dmul(a[2], b[0]), dmul(a[0], b[2]));
  r[2] = dsub(dmul(a[0], b[1]), dmul(a[1], b[0]));
}

// Point<T>::FillRotationMatrix (reference src/primitives.h:252-262), double.  The three sincos calls are spread over
// lanes 0..2 (every lane runs one call) and exchanged by shuffle; all lanes return the same matrix.
__device__ void rotation_f64_warp(double yaw, double pitch, double roll, double *m, int lane) {
  const int sel = lane % 3;
  const double ang = sel == 0 ? yaw : (sel == 1 ? pitch : roll);
  double s, c;
  sincos(ang, &s, &c);
  const double sy = __shfl_sync(kFull, s, 0), cy = __shfl_sync(kFull, c, 0);
  const double sp = __shfl_sync(kFull, s, 1), cp = __shfl_sync(kFull, c, 1);
  const double sr = __shfl_sync(kFull, s, 2), cr = __shfl_sync(kFull, c, 2);
  m[0] = dmul(cy, cp);
  m[1] = dsub(dmul(dmul(cy, sp), sr), dmul(sy, cr));
  m[2] = dadd(dmul(dmul(cy, sp), cr), dmul(sy, sr));
  m[3] = dmul(sy, cp);
  m[4] = dadd(dmul(dmul(sy, sp), sr), dmul(cy, cr));
  m[5] = dsub(dmul(dmul(sy, sp), cr), dmul(cy, sr));
  m[6] = -sp;
  m[7] = dmul(cp, sr);
  m[8] = dmul(cp, cr);
}

// all 32 lanes call this with identical arguments; lane k < 17 evaluates axis k.  Returns the pair verdict.
__device__ __noinline__ bool exact_pair_contact(const double *R2, const double *T2, const double *ot, const double *rq,
                                                int lane) {
  // mT = R2^T * (0 - T2); vertex = (R2^T row . p) * 1.0 + mT
  double u[3] = {dsub(0.0, T2[0]), dsub(0.0, T2[1]), dsub(0.0, T2[2])};
  double mT[3], P[3][3];
#pragma unroll
  for (int i = 0; i < 3; ++i) mT[i] = dadd(dadd(dmul(R2[0 + i], u[0]), dmul(R2[3 + i], u[1])), dmul(R2[6 + i], u[2]));
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double s = dadd(dadd(dmul(R2[0 + i], ot[3 * v]), dmul(R2[3 + i], ot[3 * v + 1])), dmul(R2[6 + i], ot[3 * v + 2]));
      P[v][i] = dadd(dmul(1.0, s), mT[i]);
    }
  // everything relative to P[0]
  double p[3][3], q[3][3], vec[8][3];   // vec: e1 e2 e3 f1 f2 f3 n1 m1
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    p[0][k] = dsub(P[0][k], P[0][k]);
    p[1][k] = dsub(P[1][k], P[0][k]);
    p[2][k] = dsub(P[2][k], P[0][k]);
    q[0][k] = dsub(rq[k], P[0][k]);
    q[1][k] = dsub(rq[3 + k], P[0][k]);
    q[2][k] = dsub(rq[6 + k], P[0][k]);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    vec[0][k] = dsub(p[1][k], p[0][k]);
    vec[1][k] = dsub(p[2][k], p[1][k]);
    vec[2][k] = dsub(p[0][k], p[2][k]);
    vec[3][k] = dsub(q[1][k], q[0][k]);
    vec[4][k] = dsub(q[2][k], q[1][k]);
    vec[5][k] = dsub(q[0][k], q[2][k]);
  }
  dcross(vec[6], vec[0], vec[1]);
  dcross(vec[7], vec[3], vec[4]);
  // axis table: 0: n1, 1: m1, 2..10: e_i x f_j, 11..13: e_i x n1, 14..16: f_j x m1
  bool overlaps = true;
  if (lane < 17) {
    double ax[3];
    if (lane == 0) { ax[0] = vec[6][0]; ax[1] = vec[6][1]; ax[2] = vec[6][2]; }
    else if (lane == 1) { ax[0] = vec[7][0]; ax[1] = vec[7][1]; ax[2] = vec[7][2]; }
    else {
      int a, b;
      if (lane < 11) { a = (lane - 2) / 3; b = 3 + (lane - 2) % 3; }
      else if (lane < 14) { a = lane - 11; b = 6; }
      else { a = 3 + (lane - 14); b = 7; }
      dcross(ax, vec[a], vec[b]);
    }
    double P1 = ddot(ax, p[0]), P2 = ddot(ax, p[1]), P3 = ddot(ax, p[2]);
    double Q1 = ddot(ax, q[0]), Q2 = ddot(ax, q[1]), Q3 = ddot(ax, q[2]);
    double mx1 = fmax(P1, fmax(P2, P3)), mn1 = fmin(P1, fmin(P2, P3));
    double mx2 = fmax(Q1, fmax(Q2, Q3)), mn2 = fmin(Q1, fmin(Q2, Q3));
    if (mn1 > mx2) overlaps = false;
    if (mn2 > mx1) overlaps = false;
  }
  return __all_sync(kFull, overlaps);
}

// ---------------------------------------------------------------------------------------------------------
// pose formats.  Each lane keeps its own pose in the narrowest form that loses nothing; the exact stage fetches the
// double pose of lane `src` on demand (rare), so the FP32 fast path of an f32 batch never touches the FP64 pipe.
// ---------------------------------------------------------------------------------------------------------
enum { kFmtEulerF32 = 0, kFmtEulerF64 = 1, kFmtMatrixF64 = 2 };

template <int FMT> struct LanePose;

template <> struct LanePose<kFmtEulerF32> {
  float t[3], a[3];
  __device__ __forceinline__ void load(const void *base, long long i) {
    const float2 *p = reinterpret_cast<const float2 *>(base) + 3 * i;
    const float2 x = p[0], y = p[1], z = p[2];
    t[0] = x.x; t[1] = x.y; t[2] = y.x; a[0] = y.y; a[1] = z.x; a[2] = z.y;
  }
  __device__ __forceinline__ void clear() { t[0] = t[1] = t[2] = a[0] = a[1] = a[2] = 0.f; }
  __device__ __forceinline__ void split(float *hi, float *lo) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) { hi[k] = t[k]; lo[k] = 0.f; }
  }
  __device__ __forceinline__ void rot32(float *R) const;
  __device__ __forceinline__ void exact(int src, double *R2, double *T2, int lane) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) T2[k] = (double)__shfl_sync(kFull, t[k], src);
    rotation_f64_warp((double)__shfl_sync(kFull, a[0], src), (double)__shfl_sync(kFull, a[1], src),
                      (double)__shfl_sync(kFull, a[2], src), R2, lane);
  }
};

template <> struct LanePose<kFmtEulerF64> {
  double t[3], a[3];
  bool identity;   // edge samples in reference mode: R = I exactly, no trigonometry anywhere
  __device__ __forceinline__ void load(const void *base, long long i) {
    const double2 *p = reinterpret_cast<const double2 *>(base) + 3 * i;
    const double2 x = p[0], y = p[1], z = p[2];
    t[0] = x.x; t[1] = x.y; t[2] = y.x; a[0] = y.y; a[1] = z.x; a[2] = z.y;
    identity = false;
  }
  __device__ __forceinline__ void clear() { t[0] = t[1] = t[2] = a[0] = a[1] = a[2] = 0.0; identity = false; }
  __device__ __forceinline__ void split(float *hi, float *lo) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) { hi[k] = (float)t[k]; lo[k] = (float)(t[k] - (double)hi[k]); }
  }
  __device__ __forceinline__ void rot32(float *R) const;
  __device__ __forceinline__ void exact(int src, double *R2, double *T2, int lane) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) T2[k] = __shfl_sync(kFull, t[k], src);
    if (__shfl_sync(kFull, (int)identity, src)) {
      // FillRotationMatrix at zero angles: identity with m[2][0] = -sin(0) = -0.0
      R2[0] = 1.0; R2[1] = 0.0; R2[2] = 0.0; R2[3] = 0.0; R2[4] = 1.0; R2[5] = 0.0; R2[6] = -0.0; R2[7] = 0.0; R2[8] = 1.0;
    } else {
      rotation_f64_warp(__shfl_sync(kFull, a[0], src), __shfl_sync(kFull, a[1], src), __shfl_sync(kFull, a[2], src), R2, lane);
    }
  }
};

template <> struct LanePose<kFmtMatrixF64> {
  double t[3], r[9];   // RAPID_Collide's own arguments: R2 row-major, T2
  __device__ __forceinline__ void load(const void *base, long long i) {
    const double *p = reinterpret_cast<const double *>(base) + 12 * i;
#pragma unroll
    for (int k = 0; k < 9; ++k) r[k] = p[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) t[k] = p[9 + k];
  }
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int k = 0; k < 9; ++k) r[k] = 0.0;
    t[0] = t[1] = t[2] = 0.0;
  }
  __device__ __forceinline__ void split(float *hi, float *lo) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) { hi[k] = (float)t[k]; lo[k] = (float)(t[k] - (double)hi[k]); }
  }
  __device__ __forceinline__ void rot32(float *R) const {
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = (float)r[k];
  }
  __device__ __forceinline__ void exact(int src, double *R2, double *T2, int) const {
#pragma unroll
    for (int k = 0; k < 3; ++k) T2[k] = __shfl_sync(kFull, t[k], src);
#pragma unroll
    for (int k = 0; k < 9; ++k) R2[k] = __shfl_sync(kFull, r[k], src);
  }
};

// Point<T>::FillRotationMatrix in FP32 (certificate stage only), from the sines and cosines of yaw, pitch and roll
__device__ __forceinline__ void rotation_f32_sc(float sy, float cy, float sp, float cp, float sr, float cr, float *m) {
  m[0] = cy * cp;
  m[1] = cy * sp * sr - sy * cr;
  m[2] = cy * sp * cr + sy * sr;
  m[3] = sy * cp;
  m[4] = sy * sp * sr + cy * cr;
  m[5] = sy * sp * cr - cy * sr;
  m[6] = -sp;
  m[7] = cp * sr;
  m[8] = cp * cr;
}
__device__ __forceinline__ void LanePose<kFmtEulerF32>::rot32(float *R) const {
  float sy, cy, sp, cp, sr, cr;
  sincosf(a[0], &sy, &cy);
  sincosf(a[1], &sp, &cp);
  sincosf(a[2], &sr, &cr);
  rotation_f32_sc(sy, cy, sp, cp, sr, cr, R);
}
// sin and cos of a double angle for the FP32 rotation.  Narrowing the angle to float moves it by up to half an ulp of the
// angle: at most 2^-23 while |a| <= float(pi), which the error budget covers (see kEpsSat), but 2^-15 at 1000 rad, more
// than the whole budget.  Angles beyond float(pi) therefore take sincos(double) of the angle itself, rounded to float
// (within 2^-25 plus sincos's 1 ulp in double, for every finite angle); in-range angles keep the FP32 path.
__device__ __forceinline__ void sincos_narrow(double a, float *s, float *c) {
  const float af = (float)a;
  if (fabsf(af) <= 3.14159274f) {
    sincosf(af, s, c);
  } else {
    double sd, cd;
    sincos(a, &sd, &cd);
    *s = (float)sd;
    *c = (float)cd;
  }
}
__device__ __forceinline__ void LanePose<kFmtEulerF64>::rot32(float *R) const {
  if (identity) {
    R[0] = 1.f; R[1] = 0.f; R[2] = 0.f; R[3] = 0.f; R[4] = 1.f; R[5] = 0.f; R[6] = 0.f; R[7] = 0.f; R[8] = 1.f;
  } else {
    float sy, cy, sp, cp, sr, cr;
    sincos_narrow(a[0], &sy, &cy);
    sincos_narrow(a[1], &sp, &cp);
    sincos_narrow(a[2], &sr, &cr);
    rotation_f32_sc(sy, cy, sp, cp, sr, cr, R);
  }
}

// ---------------------------------------------------------------------------------------------------------
// per-pose warp traversal
// ---------------------------------------------------------------------------------------------------------
struct PoseU {          // warp-uniform copy of one pose
  float R[9];           // row-major, world <- robot
  float Thi[3], Tlo[3]; // T = Thi + Tlo (+ negligible)
};

struct Tally { unsigned long long past_root, box, pair, exact, steps, tri_passes, tris, exact_run, past_grid; };

struct BoxTest {        // per-pose constants of the oriented-box test
  float o[3], ra[3], rob_sz;
};

__device__ __forceinline__ BoxTest make_box_test(const EnvDev &E, const PoseU &P) {
  BoxTest bt;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    bt.o[k] = P.R[3 * k] * E.rob_c[0] + P.R[3 * k + 1] * E.rob_c[1] + P.R[3 * k + 2] * E.rob_c[2] + P.Tlo[k];
    bt.ra[k] = fabsf(P.R[3 * k]) * E.rob_h[0] + fabsf(P.R[3 * k + 1]) * E.rob_h[1] + fabsf(P.R[3 * k + 2]) * E.rob_h[2];
  }
  bt.rob_sz = 2.0f * E.rob_radius + fabsf(P.Tlo[0]) + fabsf(P.Tlo[1]) + fabsf(P.Tlo[2]);
  return bt;
}

// robot oriented box (centre T + R c, axes R, half extents h) against an AABB slot; conservative.  Straight-line code:
// lanes of one step almost never agree on an early exit, so all six axes are evaluated and combined without branches.
__device__ __forceinline__ bool slot_overlaps(const EnvDev &E, const PoseU &P, const BoxTest &bt, const float4 a, const float4 b) {
  const float tx = (a.x - P.Thi[0]) - bt.o[0], ty = (a.y - P.Thi[1]) - bt.o[1], tz = (a.z - P.Thi[2]) - bt.o[2];
  const float pad = kEpsBox * (fabsf(tx) + fabsf(ty) + fabsf(tz) + b.x + b.y + b.z + bt.rob_sz);
  const float s0 = P.R[0] * tx + P.R[3] * ty + P.R[6] * tz, s1 = P.R[1] * tx + P.R[4] * ty + P.R[7] * tz,
              s2 = P.R[2] * tx + P.R[5] * ty + P.R[8] * tz;
  const float r0 = fabsf(P.R[0]) * b.x + fabsf(P.R[3]) * b.y + fabsf(P.R[6]) * b.z,
              r1 = fabsf(P.R[1]) * b.x + fabsf(P.R[4]) * b.y + fabsf(P.R[7]) * b.z,
              r2 = fabsf(P.R[2]) * b.x + fabsf(P.R[5]) * b.y + fabsf(P.R[8]) * b.z;
  // the largest excess over the allowed distance on any axis; overlap iff none is positive
  const float ex = fmaxf(fmaxf(fabsf(tx) - (b.x + bt.ra[0]), fabsf(ty) - (b.y + bt.ra[1])), fabsf(tz) - (b.z + bt.ra[2]));
  const float eb = fmaxf(fmaxf(fabsf(s0) - (E.rob_h[0] + r0), fabsf(s1) - (E.rob_h[1] + r1)), fabsf(s2) - (E.rob_h[2] + r2));
  return !(fmaxf(ex, eb) > pad);
}

// state of the pair stages of one pose: the verdict so far and the pose's double-precision transform (built on first use)
// (the flags stay separate scalars: the transform arrays are handed to the non-inlined exact stage by address, and a struct
// holding both would drag the flags into local memory with them -- measured +2.4 % on the pose kernel)
struct PairCtx {
  double R2[9], T2[3];
};

// obstacle triangle t (leaf order) into the robot frame of pose P (what RAPID does: x = R^T (p - T)), tagged with the lane
// `tag` its pose came from; returns false when its box, padded by the position error bound, misses the robot's box
__device__ __forceinline__ bool transform_triangle(const EnvDev &E, const PoseU &P, int t, int tag, XTri &x) {
  const float4 v0 = __ldg(E.tris32 + 3 * (size_t)t), v1 = __ldg(E.tris32 + 3 * (size_t)t + 1),
               v2 = __ldg(E.tris32 + 3 * (size_t)t + 2);
  const float w[9] = {(v0.x - P.Thi[0]) - P.Tlo[0], (v0.y - P.Thi[1]) - P.Tlo[1], (v0.z - P.Thi[2]) - P.Tlo[2],
                      (v1.x - P.Thi[0]) - P.Tlo[0], (v1.y - P.Thi[1]) - P.Tlo[1], (v1.z - P.Thi[2]) - P.Tlo[2],
                      (v2.x - P.Thi[0]) - P.Tlo[0], (v2.y - P.Thi[1]) - P.Tlo[1], (v2.z - P.Thi[2]) - P.Tlo[2]};
  float mabs = 0.f;
#pragma unroll
  for (int v = 0; v < 3; ++v)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float val = P.R[c] * w[3 * v] + P.R[3 + c] * w[3 * v + 1] + P.R[6 + c] * w[3 * v + 2];
      x.v[3 * v + c] = val;
      mabs = fmaxf(mabs, fabsf(val));
    }
  x.err = v0.w;
  x.mabs = mabs;
  x.tri = t;
  x.pad = tag;
  const float padT = 2.0f * x.err + kEpsSat * fmaxf(mabs, E.rob_radius);
  bool keep = true;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float lo = min3f(x.v[c], x.v[3 + c], x.v[6 + c]) - padT, hi = max3f(x.v[c], x.v[3 + c], x.v[6 + c]) + padT;
    const float rc = c == 0 ? E.rob_c[0] : (c == 1 ? E.rob_c[1] : E.rob_c[2]);
    const float rh = c == 0 ? E.rob_h[0] : (c == 1 ? E.rob_h[1] : E.rob_h[2]);
    if (lo > rc + rh || hi < rc - rh) keep = false;
  }
  return keep;
}

// m without its n lowest set bits
__device__ __forceinline__ unsigned drop_lowest(unsigned m, int n) {
#pragma unroll
  for (int k = 0; k < n; ++k) m &= m - 1;
  return m;
}
// the lane of the n-th lowest set bit of m (n = 0..4), -1 when m has no more than n
__device__ __forceinline__ int nth_lane(unsigned m, int n) {
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (k < n) m &= m - 1;
  return __ffs(m) - 1;
}

// Triangle stage of one pose over the candidate triangles ws.tri[0, ntri): transform into the robot frame, cull, pair stages
// P1 (lane-per-pair), P2 and the FP64 exact stage; stops at the first confirmed contact.  CONTACT_FIRST selects the P2 order:
// the contact certificates of five pairs before their separating axes (the pose verdict kernel, whose open pairs mostly
// touch), or the axes of three pairs first and the certificates of what they leave open (every other kernel: edge samples
// are mostly free, and the distance and sweep kernels keep their registers).  Either order gives every pair that no
// certificate proves in contact all nine axes, then FP64, so the verdict of every call is the same.
template <int FMT, bool COUNT, bool CONTACT_FIRST>
__device__ __forceinline__ void triangle_stage(const EnvDev &E, WarpScratch &ws, const RobotTri *srob, const PoseU &P,
                                               const LanePose<FMT> &lp, int src, int lane, int ntri, bool &hit, bool &have_R2,
                                               PairCtx &pc, Tally &tally) {
  const unsigned lt = (1u << lane) - 1u;
  const int grp10 = lane / 10, k10 = lane - 10 * grp10, grp6 = lane / 6, k6 = lane - 6 * grp6;
  const float inv_n_robot = 1.0f / (float)E.n_robot;
  for (int base = 0; base < ntri && !hit; base += 32) {
    const int cnt = (ntri - base) < 32 ? (ntri - base) : 32;
    bool keep = false;
    XTri x;
    if (lane < cnt) keep = transform_triangle(E, P, ws.tri[base + lane], 0, x);
    const unsigned km = __ballot_sync(kFull, keep);
    const int nx = __popc(km);
    if (COUNT) { tally.tri_passes += 1; tally.tris += cnt; }
    if (keep) ws.xt[__popc(km & lt)] = x;
    __syncwarp();
    const int npairs = nx * E.n_robot;
    for (int pb = 0; pb < npairs && !hit; pb += 32) {
      const int pidx = pb + lane;
      bool undecided = false;
      // (triangle, robot triangle) of this lane's pair; the quotient by float reciprocal is exact for pidx < 2^20
      const int xi_l = (int)(((float)pidx + 0.5f) * inv_n_robot), r_l = pidx - xi_l * E.n_robot;
      if (pidx < npairs) undecided = !pair_quick_disjoint(ws.xt[xi_l], srob[r_l]);
      unsigned um = __ballot_sync(kFull, undecided);
      if (COUNT) {
        const int np = (npairs - pb) < 32 ? (npairs - pb) : 32;
        tally.pair += np;
        tally.exact += __popc(um);   // pairs the lane-per-pair stage P1 left open
      }
      if constexpr (CONTACT_FIRST) {
        // the pair of lane l, computed again where needed: cheaper in registers than shuffling it from its lane
        const auto pair_of = [&](int l, int &xi, int &r) {
          xi = (int)(((float)(pb + l) + 0.5f) * inv_n_robot);
          r = pb + l - xi * E.n_robot;
        };
        while (um && !hit) {
          const unsigned five = um ^ drop_lowest(um, 5);   // the next five open pairs
          um ^= five;
          const int lc = grp6 < 5 ? nth_lane(five, grp6) : -1;   // pass c: lane 6g + c, certificate c of pair g
          int xi, r;
          bool con = false;
          if (lc >= 0) {
            pair_of(lc, xi, r);
            con = open_pair_pierce(ws.xt[xi], srob[r], k6);
          }
          if (__any_sync(kFull, con)) {
            hit = true;
            break;
          }
          // none of the five touches provably: pass a, three pairs at a time, and FP64 for what it leaves open
          unsigned left = five;
#pragma unroll 1
          while (left && !hit) {
            const unsigned three = left ^ drop_lowest(left, 3);
            left ^= three;
            const int la = grp10 < 3 ? nth_lane(three, grp10) : -1;
            bool sep = false;
            if (la >= 0 && k10 < 9) {
              pair_of(la, xi, r);
              sep = open_pair_axis(ws.xt[xi], srob[r], k10);
            }
            const unsigned bs = __ballot_sync(kFull, sep);
#pragma unroll 1
            for (int g = 0; g < 3; ++g) {
              const int lg = nth_lane(three, g);
              if (lg < 0) break;
              if ((bs >> (10 * g)) & 0x3ffu) continue;
              if (COUNT) tally.exact_run += 1;
              if (!have_R2) {
                lp.exact(src, pc.R2, pc.T2, lane);
                have_R2 = true;
              }
              pair_of(lg, xi, r);
              const int t = ws.xt[xi].tri;
              if (exact_pair_contact(pc.R2, pc.T2, E.tris64 + 9 * (size_t)t, E.robot64 + 9 * (size_t)r, lane)) {
                hit = true;
                break;
              }
            }
          }
        }
      } else {
        while (um && !hit) {
          const int l0 = __ffs(um) - 1;
          um &= um - 1;
          const int l1 = um ? __ffs(um) - 1 : -1;
          um &= um - 1;   // (0 stays 0)
          const int l2 = um ? __ffs(um) - 1 : -1;
          um &= um - 1;
          const int lmine = grp10 == 0 ? l0 : (grp10 == 1 ? l1 : (grp10 == 2 ? l2 : -1));
          const int xim = __shfl_sync(kFull, xi_l, lmine & 31), rm = __shfl_sync(kFull, r_l, lmine & 31);
          bool sep = false;
          if (lmine >= 0 && k10 < 9) sep = open_pair_axis(ws.xt[xim], srob[rm], k10);
          const unsigned bs = __ballot_sync(kFull, sep);
          unsigned open_g = 0;
          if (!(bs & 0x3ffu)) open_g |= 1u;
          if (l1 >= 0 && !(bs & (0x3ffu << 10))) open_g |= 2u;
          if (l2 >= 0 && !(bs & (0x3ffu << 20))) open_g |= 4u;
          if (open_g == 0) continue;
          // pass c on the lanes of the axes, for the pairs no axis separated
          bool con = false;
          if (lmine >= 0 && k10 < 6 && ((open_g >> grp10) & 1u)) con = open_pair_pierce(ws.xt[xim], srob[rm], k10);
          if (__any_sync(kFull, con)) {
            hit = true;
            break;
          }
          while (open_g) {
            const int g = __ffs(open_g) - 1;
            open_g &= open_g - 1;
            const int lg = g == 0 ? l0 : (g == 1 ? l1 : l2);
            const int xg = __shfl_sync(kFull, xi_l, lg), rg = __shfl_sync(kFull, r_l, lg);
            if (COUNT) tally.exact_run += 1;
            if (!have_R2) {
              lp.exact(src, pc.R2, pc.T2, lane);
              have_R2 = true;
            }
            const int t = ws.xt[xg].tri;
            if (exact_pair_contact(pc.R2, pc.T2, E.tris64 + 9 * (size_t)t, E.robot64 + 9 * (size_t)rg, lane)) {
              hit = true;
              break;
            }
          }
        }
      }
    }
    __syncwarp();
  }
}

// what one step of the hierarchy walk found: the ballot of lanes holding an accepted leaf, and this lane's triangle
struct StepLeaves {
  unsigned mask;
  bool mine;
  int tri;
};

// One step of the warp-cooperative walk of the hierarchy.  Step 0 (`first`) tests the precomputed <= 32-slot cut of the
// top of the hierarchy with all lanes (top_cut emits no empty slot).  Every later step pops up to 4 nodes from the stack,
// 8 lanes per node; near the cap it pops 1 (strict depth-first grows the stack by at most 7 per level), which keeps any
// hierarchy of depth <= 45 inside the stack.  Interior children that `overlaps(a, b)` accepts are pushed; `sp` may end
// above kStackCap (those pushes are dropped), and the caller decides what that means.  Accepted leaves are returned for
// the caller to append where it keeps them.
template <bool COUNT, class Overlaps>
__device__ __forceinline__ StepLeaves walk_step(const EnvDev &E, WarpScratch &ws, const CtaShared &cs, bool first, int &sp,
                                                int lane, const Overlaps &overlaps, Tally &tally) {
  bool ov = false;
  int child = kEmptyChild;
  bool active;
  if (first) {
    active = lane < E.n_top;
    if (active) {
      const float4 a = cs.top[lane], b = cs.top[kTopSlots + lane];
      child = __float_as_int(a.w);
      ov = overlaps(a, b);
    }
  } else {
    const int take = sp > kStackCap - 64 ? 1 : (sp < 4 ? sp : 4);
    const int grp = lane >> 3;
    active = grp < take;
    const int node = active ? ws.stack[sp - 1 - grp] : 0;
    __syncwarp();
    sp -= take;
    if (active) {
      float4 a, b;
      if (node < cs.n_stage) {   // (nodes of one step are popped together: mostly one side of this branch)
        const int si = node * kWide + (lane & 7);
        a = cs.nodes[si];                             // staged as two arrays (all `a` halves, then all `b` halves):
        b = cs.nodes[cs.n_stage * kWide + si];        // 8 lanes read 128 contiguous bytes, no bank conflicts
      } else {
        const float4 *gn = E.slots + ((size_t)node * kWide + (lane & 7)) * 2;
        a = __ldg(gn);
        b = __ldg(gn + 1);
      }
      child = __float_as_int(a.w);
      if (child != kEmptyChild) ov = overlaps(a, b);
    }
  }
  const unsigned m_int = __ballot_sync(kFull, ov && child >= 0);
  const unsigned m_leaf = __ballot_sync(kFull, ov && child < 0);
  if (COUNT) { tally.box += __popc(__ballot_sync(kFull, active && child != kEmptyChild)); tally.steps += 1; }
  if (ov && child >= 0) {
    const int pos = sp + __popc(m_int & ((1u << lane) - 1u));
    if (pos < kStackCap) ws.stack[pos] = child;
  }
  sp += __popc(m_int);
  return {m_leaf, ov && child < 0, ~child};
}

// PROBE: the contact probe (every kernel but the edge verdict kernel); CONTACT_FIRST: triangle_stage's P2 order
template <int FMT, bool COUNT, bool PROBE, bool CONTACT_FIRST>
__device__ bool warp_pose_hit(const EnvDev &E, WarpScratch &ws, const CtaShared &cs, const PoseU &P,
                              const LanePose<FMT> &lp, int src, int lane, Tally &tally) {
  const RobotTri *srob = cs.rob;
  const BoxTest bt = make_box_test(E, P);
  const auto overlaps = [&](const float4 a, const float4 b) { return slot_overlaps(E, P, bt, a, b); };
  const unsigned lt = (1u << lane) - 1u;

  int sp = 0, ntri = 0;
  bool hit = false, have_R2 = false;
  PairCtx pc;
  if (COUNT) tally.past_root += 1;

  // Contact probe: a pose that reaches phase B mostly collides, and mostly with one of its cell's two witnesses (the
  // triangles that mark the cell nearest its centre).  The first pass of the loop below runs the triangle stage over them
  // alone; a confirmed contact ends the pose without a walk, anything else walks from the root as if there were no probe.
  // (Phase A fetched the witnesses of every lane's cell with its plane, into ws.wit.)
  // The edge kernel is built without it (PROBE = false): its samples mostly share the swept-box candidate list, and the
  // probe's code alone cost its per-sample loop 2 % of the edge rate in spills.
  bool probe = false;
  if (PROBE) {
    const int2 w = ws.wit[src];
    if (lane < 2) ws.tri[lane] = lane ? w.y : w.x;
    ntri = (w.x >= 0) + (w.y >= 0);   // (w.y >= 0 only with w.x >= 0)
    probe = ntri > 0;
    __syncwarp();
  }

  bool first = true;
  while (true) {
    // walk until a candidate triangle is pending, then run the triangle stage over what the last step found
    if (!probe && (first || (sp > 0 && ntri <= kTriCap - 32))) {
      const StepLeaves lv = walk_step<COUNT>(E, ws, cs, first, sp, lane, overlaps, tally);
      first = false;
      if (lv.mine) ws.tri[ntri + __popc(lv.mask & lt)] = lv.tri;
      ntri += __popc(lv.mask);
      if (sp > kStackCap) {     // never silently drop work: flag the launch as failed
        if (lane == 0) *reinterpret_cast<volatile int *>(E.status) = 1;
        sp = kStackCap;
      }
      __syncwarp();
      if (sp > 0 && ntri == 0) continue;
    }
    if (ntri == 0) {
      if (sp == 0) break;
      continue;
    }
    // ---------------- triangle stage ----------------
    triangle_stage<FMT, COUNT, CONTACT_FIRST>(E, ws, srob, P, lp, src, lane, ntri, hit, have_R2, pc, tally);
    if (hit) break;
    ntri = 0;
    if (probe) {   // no contact with the witnesses: the walk starts (it may deliver them again, which is harmless)
      probe = false;
      continue;
    }
    if (sp == 0) break;
  }
  return hit;
}

// ---------------------------------------------------------------------------------------------------------
// Edge samples in reference mode all carry the identity rotation (src/problemStruct.h:157-163), so the robot's box at a
// sample is the axis-aligned box T + [rob_c - rob_h, rob_c + rob_h] and the boxes of the surviving samples of one
// 32-sample group lie in one slightly larger axis-aligned box.  ONE traversal with that swept box collects every triangle
// any of the samples could touch; each sample then runs only the triangle stage over that list.  (The per-sample
// traversal was 63 % of the edge kernel's instructions.)  The list is a superset of what the per-sample traversal would
// deliver and every stage after it is unchanged, so the verdicts are the same.
// ---------------------------------------------------------------------------------------------------------
// every leaf triangle whose slot box meets [lo, hi] -> ws.cand; returns their number, or -1 when the list would overflow
template <bool COUNT>
__device__ int collect_box_candidates(const EnvDev &E, WarpScratch &ws, const CtaShared &cs, const float *lo, const float *hi, int lane,
                                      Tally &tally) {
  // slot box [c - h, c + h] against [lo, hi], directed rounding keeps the test conservative
  const auto overlaps = [&](const float4 a, const float4 b) {
    return __fadd_ru(a.x, b.x) >= lo[0] && __fsub_rd(a.x, b.x) <= hi[0] && __fadd_ru(a.y, b.y) >= lo[1] &&
           __fsub_rd(a.y, b.y) <= hi[1] && __fadd_ru(a.z, b.z) >= lo[2] && __fsub_rd(a.z, b.z) <= hi[2];
  };
  const unsigned lt = (1u << lane) - 1u;
  int sp = 0, ncand = 0;
  bool first = true;
  while (first || sp > 0) {
    const StepLeaves lv = walk_step<COUNT>(E, ws, cs, first, sp, lane, overlaps, tally);
    first = false;
    if (ncand + __popc(lv.mask) > kCandCap || sp > kStackCap) {
      __syncwarp();   // the caller falls back to the per-sample traversal (which reports stack overflows) on this stack
      return -1;
    }
    if (lv.mine) ws.cand[ncand + __popc(lv.mask & lt)] = lv.tri;
    ncand += __popc(lv.mask);
    __syncwarp();
  }
  return ncand;
}

// one sample against the shared candidate list
template <int FMT, bool COUNT>
__device__ bool pose_hits_candidates(const EnvDev &E, WarpScratch &ws, const CtaShared &cs, const PoseU &P, const LanePose<FMT> &lp,
                                     int src, int lane, int ncand, Tally &tally) {
  bool hit = false, have_R2 = false;
  PairCtx pc;
  if (COUNT) tally.past_root += 1;
  for (int base = 0; base < ncand && !hit; base += 32) {
    const int cnt = (ncand - base) < 32 ? (ncand - base) : 32;
    if (lane < cnt) ws.tri[lane] = ws.cand[base + lane];
    __syncwarp();
    triangle_stage<FMT, COUNT, false>(E, ws, cs.rob, P, lp, src, lane, cnt, hit, have_R2, pc, tally);
  }
  return hit;
}

// A clear bit proves that no obstacle triangle comes within the robot's bounding radius of any point of the cell (the
// build inflates the reach by the cell's half diagonal plus rounding margins), so the pose is free whatever its orientation.
__device__ __forceinline__ bool cell_marked(const EnvDev &E, int cell) {
  return ((__ldg(E.grid.bits + (cell >> 5)) >> (cell & 31)) & 1u) != 0u;
}

// O(1) free-space test for a marked cell: its plane record `word` holds a direction m and an offset c with m.p >= c for every
// vertex p of every obstacle triangle that marks the cell (the build's own predicate, so every triangle that can touch a
// robot whose origin lies in the cell, by the argument of the clear bit).  A convex robot hull strictly below the plane
// (m.x < c for every robot point x = R v + T) meets none of those triangles, so the pose is free.
//
// The test computes s = m.thi + max_v (R^T m).v in FP32 and clears the pose when s + margin < c, c rounded down.  The
// margin bounds |s - m.(R_o v + T)| for the oracle's FP64 rotation R_o of the pose's own angles (or its matrix):
//   - R: every entry of the FP32 rotation within 2^-19 of R_o (see kEpsSat); w = R^T m has |m|_1 <= 3 exact terms per
//     entry, so |w - R_o^T m| <= 3 * 2^-19 + 2^-21 < 2^-17 per entry, times |v|_1 <= sqrt(3) rho; the nearest-float
//     vertices and the FP32 dot product add < 12 * 2^-24 rho.  The box support (w.c + sum |w_j| h_j, |c_j| + h_j <= rho)
//     moves by < 3 * 2^-17 rho + 12 * 2^-24 rho.  Allotted 2^-15 rho (plane_pad).
//   - T = thi + tlo: |m.tlo| <= |tlo|_1, added as is; m.thi and the final sums round by < 2^-22 (|thi|_1 + 3 rho),
//     allotted 2^-20 |thi|_1 (and the 2^-15 rho above).
//   - the grid's absolute slack (stated once, in clearance_margins of clearance_grid.cu, which adds it to the reach too),
//     carried in plane_pad so that a plane never clears a pose that the grid's own rounding allowances would hold back.
// With these the robot stays below the plane by a positive gap in exact arithmetic, and the oracle's FP64 SAT finds
// separated triangles separated -- the same ground the clear bit and the FP32 certificates stand on (DESIGN.md 4.1).
__device__ __forceinline__ bool plane_says_free(const EnvDev &E, unsigned word, const float *R, const float *thi, float tlo_mag) {
  const float c = ordered_to_float((int)(word & ~31u));
  float m[3];
  plane_dir((int)(word & 31u), m);
  const float w0 = m[0] * R[0] + m[1] * R[3] + m[2] * R[6], w1 = m[0] * R[1] + m[1] * R[4] + m[2] * R[7],
              w2 = m[0] * R[2] + m[1] * R[5] + m[2] * R[8];
  float sup;
  if (E.rob_verts) {
    sup = -FLT_MAX;
#pragma unroll 1   // (unrolled, the loop costs the edge kernel extra spill reloads)
    for (int i = 0; i < E.n_rob_verts; ++i) {
      const float4 v = __ldg(E.rob_verts + i);
      sup = fmaxf(sup, w0 * v.x + w1 * v.y + w2 * v.z);
    }
  } else {
    sup = w0 * E.rob_c[0] + w1 * E.rob_c[1] + w2 * E.rob_c[2] + fabsf(w0) * E.rob_h[0] + fabsf(w1) * E.rob_h[1] +
          fabsf(w2) * E.rob_h[2];
  }
  const float s = m[0] * thi[0] + m[1] * thi[1] + m[2] * thi[2] + sup;
  const float margin = E.grid.plane_pad + 9.5367431640625e-07f * (fabsf(thi[0]) + fabsf(thi[1]) + fabsf(thi[2])) + tlo_mag;
  return s + margin < c;
}

// lane-per-pose cull: robot bounding sphere (about the robot origin) against the obstacle AABB
__device__ __forceinline__ bool sphere_hits_root(const EnvDev &E, float tx, float ty, float tz, float tlo_mag) {
  const float dx = fmaxf(fabsf(tx - E.root_c[0]) - E.root_h[0], 0.f);
  const float dy = fmaxf(fabsf(ty - E.root_c[1]) - E.root_h[1], 0.f);
  const float dz = fmaxf(fabsf(tz - E.root_c[2]) - E.root_h[2], 0.f);
  const float pad = kEpsBox * (fabsf(tx) + fabsf(ty) + fabsf(tz) + fabsf(E.root_c[0]) + fabsf(E.root_c[1]) +
                               fabsf(E.root_c[2]) + E.root_h[0] + E.root_h[1] + E.root_h[2] + E.rob_radius) + tlo_mag;
  const float r = E.rob_radius + pad;
  return dx * dx + dy * dy + dz * dz <= r * r * 1.000001f;
}

// robot records, top cut and the first `n_stage` nodes of the hierarchy -> shared memory (once per CTA)
__device__ __forceinline__ CtaShared stage_cta(const EnvDev &E, unsigned char *smem, int n_stage) {
  RobotTri *srob = reinterpret_cast<RobotTri *>(smem);
  float4 *stop = reinterpret_cast<float4 *>(smem + (size_t)E.n_robot * sizeof(RobotTri));
  float4 *snodes = stop + 2 * kTopSlots;
  {
    const int words = E.n_robot * (int)(sizeof(RobotTri) / 4);
    const float *g = reinterpret_cast<const float *>(E.robot);
    float *d = reinterpret_cast<float *>(srob);
    for (int i = threadIdx.x; i < words; i += blockDim.x) d[i] = __ldg(g + i);
  }
  // slot = 2 float4 (a, b) in global memory; shared memory keeps all `a` halves first, then all `b` halves
  for (int i = threadIdx.x; i < 2 * E.n_top; i += blockDim.x) stop[(i & 1) * kTopSlots + (i >> 1)] = __ldg(E.top + i);
  const int nv = n_stage * kWide * 2;
  for (int i = threadIdx.x; i < nv; i += blockDim.x) snodes[(i & 1) * n_stage * kWide + (i >> 1)] = __ldg(E.slots + i);
  __syncthreads();
  CtaShared cs;
  cs.rob = srob;
  cs.top = stop;
  cs.nodes = snodes;
  cs.n_stage = n_stage;
  return cs;
}
__device__ __forceinline__ WarpScratch &warp_scratch(const EnvDev &E, unsigned char *smem, int warp) {
  unsigned char *base = smem + (size_t)E.n_robot * sizeof(RobotTri) + (size_t)2 * kTopSlots * sizeof(float4) +
                        (size_t)E.n_stage_max * kWide * 2 * sizeof(float4);
  return reinterpret_cast<WarpScratch *>(base)[warp];
}

__device__ __forceinline__ void flush_tally(const EnvDev &E, const Tally &t, unsigned long long poses, int lane) {
  if (lane == 0 && E.counters) {
    atomicAdd(E.counters + 0, poses);
    atomicAdd(E.counters + 1, t.past_root);
    atomicAdd(E.counters + 2, t.box);
    atomicAdd(E.counters + 3, t.pair);
    atomicAdd(E.counters + 4, t.exact);
    atomicAdd(E.counters + 8, t.exact_run);
    atomicAdd(E.counters + 9, t.past_grid);
    atomicAdd(E.counters + 5, t.steps);
    atomicAdd(E.counters + 6, t.tri_passes);
    atomicAdd(E.counters + 7, t.tris);
  }
}

// phase A (lane-per-pose cull + rotation) then phase B over the surviving lanes; returns the mask of colliding lanes
// (stops at the first hit when `first_only`, which is what an edge needs)
// CONTACT_FIRST: the P2 order of the triangle stage (see triangle_stage); only the pose verdict kernel takes the
// certificates first
template <int FMT, bool COUNT, bool SWEPT_CAPABLE = false, bool CONTACT_FIRST = false>
__device__ __forceinline__ unsigned check_32_poses(const EnvDev &E, WarpScratch &ws, const CtaShared &cs, bool valid,
                                                   const LanePose<FMT> &lp, int lane, bool first_only, Tally &tally,
                                                   bool swept = false, bool swept_identity = true) {
  float thi[3], tlo[3], R[9];
  lp.split(thi, tlo);
  const float tlo_mag = fabsf(tlo[0]) + fabsf(tlo[1]) + fabsf(tlo[2]);
  bool alive = valid && E.n_obst > 0 && sphere_hits_root(E, thi[0], thi[1], thi[2], tlo_mag);
  constexpr bool kProbe = !SWEPT_CAPABLE;   // (warp_pose_hit's PROBE)
  unsigned plane = kNoPlane;   // (loaded before the rotation is built, which hides the load)
  int2 wit = make_int2(-1, -1);   // the contact witnesses of the cell, loaded with its plane
  if (alive && E.grid.n[0] > 0) {
    const int cell = grid_cell(E.grid, thi[0], thi[1], thi[2]);
    alive = cell < 0 || cell_marked(E, cell);
    if (alive && cell >= 0) {
      plane = __ldg(E.grid.planes + cell);
      if (kProbe && E.grid.witness) wit = __ldg(E.grid.witness + cell);
    }
  }
  if (alive) lp.rot32(R);
  if (alive && plane != kNoPlane) alive = !plane_says_free(E, plane, R, thi, tlo_mag);
  if (kProbe) {
    ws.wit[lane] = wit;
    __syncwarp();
  }
  if (COUNT) tally.past_grid += __popc(__ballot_sync(kFull, alive));
  unsigned todo = __ballot_sync(kFull, alive);
  unsigned hitmask = 0;
  int ncand = -1;   // >= 0: every sample runs the triangle stage over the swept-box candidate list ws.cand[0, ncand)
  if (SWEPT_CAPABLE && swept && __popc(todo) >= 2) {
    // one traversal with the box that holds the robot at every surviving sample, outward rounded: with the identity
    // rotation (reference mode) the robot's own axis-aligned box, with interpolated angles the cube around its bounding
    // sphere (any rotation keeps the robot inside it)
    int blo[3], bhi[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float c = __fadd_rd(thi[k], tlo[k]), cu = __fadd_ru(thi[k], tlo[k]);
      const float pad = kEpsBox * (fabsf(cu) + E.rob_radius);
      const float rl = swept_identity ? __fsub_rd(E.rob_c[k], E.rob_h[k]) : -E.rob_radius;
      const float rh = swept_identity ? __fadd_ru(E.rob_c[k], E.rob_h[k]) : E.rob_radius;
      const float l = __fsub_rd(__fadd_rd(c, rl), pad);
      const float h = __fadd_ru(__fadd_ru(cu, rh), pad);
      blo[k] = __reduce_min_sync(kFull, alive ? float_to_ordered(l) : 0x7fffffff);
      bhi[k] = __reduce_max_sync(kFull, alive ? float_to_ordered(h) : (int)0x80000000);
    }
    const float lo[3] = {ordered_to_float(blo[0]), ordered_to_float(blo[1]), ordered_to_float(blo[2])},
                hi[3] = {ordered_to_float(bhi[0]), ordered_to_float(bhi[1]), ordered_to_float(bhi[2])};
    ncand = collect_box_candidates<COUNT>(E, ws, cs, lo, hi, lane, tally);   // -1 (overflow): per-sample traversal
    if (ncand == 0) return 0;
  }
  while (todo) {
    const int src = __ffs(todo) - 1;
    todo &= todo - 1;
    PoseU P;
#pragma unroll
    for (int k = 0; k < 9; ++k) P.R[k] = __shfl_sync(kFull, R[k], src);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      P.Thi[k] = __shfl_sync(kFull, thi[k], src);
      P.Tlo[k] = FMT == kFmtEulerF32 ? 0.f : __shfl_sync(kFull, tlo[k], src);
    }
    if (SWEPT_CAPABLE && ncand > 0 ? pose_hits_candidates<FMT, COUNT>(E, ws, cs, P, lp, src, lane, ncand, tally)
                                   : warp_pose_hit<FMT, COUNT, kProbe, CONTACT_FIRST>(E, ws, cs, P, lp, src, lane, tally)) {
      hitmask |= 1u << src;
      if (first_only) break;
    }
  }
  return hitmask;
}


// spins (one thread) until every rank has published an epoch >= `epoch` in the local flag words; bounded by a 10 s timeout
__device__ __forceinline__ void wait_flags(const FlagSet &f, unsigned epoch, int *status) {
  unsigned long long t0, t1;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  for (int r = 0; r < f.n; ++r) {
    const unsigned *mine = f.p[f.me] + r;
    for (;;) {
      unsigned v;
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(mine) : "memory");
      if ((int)(v - epoch) >= 0) break;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > 10000000000ull) {   // a peer died or never launched -- flag it, never hang the GPU
        if (status) atomicExch(status, 3);
        else __trap();                  // no status word to raise (barrier without an environment): fail the launch loudly
        return;
      }
      __nanosleep(100);
    }
  }
}

template <int FMT, bool COUNT>
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSm) collide_poses_kernel(EnvDev E, const void *poses, long long n,
                                                                                  OutSet outs, GatherSync gs, int chunk) {
  extern __shared__ __align__(16) unsigned char smem[];
  if (gs.flags.n > 0 && gs.wait_epoch != 0 && threadIdx.x == 0) wait_flags(gs.flags, gs.wait_epoch, E.status);
  const CtaShared cs = stage_cta(E, smem, E.n_stage_max);   // (its __syncthreads also releases the CTA from the wait above)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpScratch &ws = warp_scratch(E, smem, warp);
  // a work unit is `chunk` (1..32) consecutive poses: 32 for large batches (full lanes in phase A), fewer when the
  // batch is too small to give every resident warp a unit (planner-sized calls are latency-, not throughput-bound)
  const long long nchunks = (n + chunk - 1) / chunk;
  Tally tally = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  unsigned long long nposes = 0;
  while (true) {
    unsigned c = 0;
    if (lane == 0) c = atomicAdd(E.work_counter, 1u) - E.work_base;
    c = __shfl_sync(kFull, c, 0);
    if ((long long)c >= nchunks) break;
    const long long i = (long long)c * chunk + lane;
    const bool mine = lane < chunk && i < n;
    LanePose<FMT> lp;
    if (mine) lp.load(poses, i);
    else lp.clear();
    if (COUNT) nposes += mine ? 1 : 0;
    const unsigned hitmask = check_32_poses<FMT, COUNT, false, true>(E, ws, cs, mine, lp, lane, false, tally);
    if (outs.n == 1) {
      if (mine) outs.p[0][i] = (uint8_t)((hitmask >> lane) & 1u);
    } else if (chunk == 32 && (long long)c * 32 + 32 <= n) {
      // peer-store gather: the 32 verdict bytes of this unit are 8 words; lane = 8 * destination + word, so one store
      // instruction serves four destinations with one full 32-byte segment each (local HBM or a peer over NVLink)
      const unsigned nib = (hitmask >> (4 * (lane & 7))) & 0xFu;
      const unsigned word = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
      for (int r0 = 0; r0 < outs.n; r0 += 4) {
        const int r = r0 + (lane >> 3);
        if (r < outs.n) reinterpret_cast<unsigned *>(outs.p[r] + (long long)c * 32)[lane & 7] = word;
      }
    } else if (mine) {
      const uint8_t v = (uint8_t)((hitmask >> lane) & 1u);
      for (int r = 0; r < outs.n; ++r) outs.p[r][i] = v;
    }
  }
  if (COUNT) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) nposes += __shfl_xor_sync(kFull, nposes, s);
    flush_tally(E, tally, nposes, lane);
  }
  if (gs.flags.n > 0) {
    // completion signal of the fused gather: the last CTA to get here publishes the epoch to every rank
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence_system();
      if (atomicAdd(gs.done_counter, 1u) == gridDim.x - 1) {
        *gs.done_counter = 0;
        __threadfence_system();
        for (int r = 0; r < gs.flags.n; ++r)
          asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(gs.flags.p[r] + gs.flags.me), "r"(gs.signal_epoch) : "memory");
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// edges: Solver<T,R>::isPathFree (reference src/problemStruct.h:154-168), one warp per edge
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double wrap_pi(double a) {
  const double pi = 3.14159265358979323846;
  if (a < -pi) return dadd(a, dmul(2.0, pi));
  else if (a >= pi) return dsub(a, dmul(2.0, pi));
  return a;
}

// `split` (power of two) warps share one edge: warp j of an edge takes the j-th contiguous 1/split of the sample indices
// (neighbouring samples share one swept box), so a planner-sized batch still occupies the whole GPU.
// With split > 1 the per-edge minimum colliding index is combined with atomicMin in `fh` (pre-set to kNoHit) and warps
// stop as soon as an earlier hit than anything they could still find is published; finalize_edges_kernel then writes
// the outputs.  split == 1 writes them directly.
constexpr int kNoHit = 0x7f7f7f7f;   // what cudaMemsetAsync(..., 0x7f, ...) produces
// work units (edge, range) a planner-sized batch is cut into per resident warp.  Measured with the swept-box traversal
// (profiles/r02_edges_swept.md): 1 beats 2 / 4 / 8 for the planner's short edges (2 048 edges of length 4: 41.6 us per call
// against 44.9 / 50.9 / 69.6), long edges lose a little (length 12: 68 against 62 us at 4).
constexpr int kEdgeUnitsPerWarp = 1;

// The samples of one edge as Solver<T,R>::isPathFree visits them: indices 1 .. S with (double)index < parts.  The edge
// verdict and the edge distance kernels both take their poses from here, so the two see the same samples.
struct EdgeSamples {
  double s[6], dir[3], adir[3];
  double parts;
  long long S;
};
__device__ __forceinline__ EdgeSamples edge_samples(const double *starts, const double *ends, unsigned eidx, double sample) {
  EdgeSamples es;
  double f[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    es.s[k] = __ldg(starts + 6 * (size_t)eidx + k);
    f[k] = __ldg(ends + 6 * (size_t)eidx + k);
  }
  // Point<T>::distance, src/primitives.h:224-235
  double sum = 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double d = dsub(es.s[k], f[k]);
    sum = dadd(sum, dmul(d, d));
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    es.adir[k] = wrap_pi(dsub(f[3 + k], es.s[3 + k]));
    sum = dadd(sum, dmul(es.adir[k], es.adir[k]));
  }
  const double total = sqrt(sum);
  es.parts = __ddiv_rn(total, sample);
#pragma unroll
  for (int k = 0; k < 3; ++k) es.dir[k] = dsub(f[k], es.s[k]);
  es.S = 0;
  if (es.parts > 1.0) {
    const double cl = ceil(es.parts);
    es.S = (cl > 2.0e9 ? 2000000000LL : (long long)cl) - 1;
  }
  return es;
}
// sample `idx` of the edge: start + (idx * dir) / parts, the angles interpolated the same way or (reference mode) the
// identity rotation
__device__ __forceinline__ void edge_sample_pose(const EdgeSamples &es, long long idx, int rot_mode, LanePose<kFmtEulerF64> &lp) {
  const double di = (double)idx;
  lp.clear();
  lp.identity = rot_mode != SFFG_ROT_INTERPOLATE;
#pragma unroll
  for (int k = 0; k < 3; ++k) lp.t[k] = dadd(es.s[k], __ddiv_rn(dmul(di, es.dir[k]), es.parts));
  if (rot_mode == SFFG_ROT_INTERPOLATE) {
#pragma unroll
    for (int k = 0; k < 3; ++k) lp.a[k] = dadd(es.s[3 + k], __ddiv_rn(dmul(di, es.adir[k]), es.parts));
  }
}

template <bool COUNT>
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSm) check_edges_kernel(EnvDev E, const double *starts,
                                                                           const double *ends, long long m, double sample,
                                                                           int rot_mode, uint8_t *free_out,
                                                                           int32_t *first_hit, int split, int *fh) {
  extern __shared__ __align__(16) unsigned char smem[];
  const CtaShared cs = stage_cta(E, smem, E.n_stage_max);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpScratch &ws = warp_scratch(E, smem, warp);
  Tally tally = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  unsigned long long nposes = 0;
  const long long units = m * split;
  while (true) {
    unsigned u = 0;
    if (lane == 0) u = atomicAdd(E.work_counter, 1u) - E.work_base;
    u = __shfl_sync(kFull, u, 0);
    if ((long long)u >= units) break;
    const unsigned eidx = u / (unsigned)split;
    const int part = (int)(u - eidx * (unsigned)split);
    const EdgeSamples es = edge_samples(starts, ends, eidx, sample);
    int hit_index = 0;
    // warp `part` of the edge takes a CONTIGUOUS range of the sample indices (neighbouring samples share one swept box)
    const long long range_len = (es.S + split - 1) / split;
    const long long first_idx = 1 + (long long)part * range_len;
    const long long last_idx = first_idx + range_len - 1 < es.S ? first_idx + range_len - 1 : es.S;
    for (long long base = first_idx; base <= last_idx && hit_index == 0; base += 32) {
      if (split > 1 && *reinterpret_cast<volatile int *>(fh + eidx) < base) break;   // an earlier hit is already known
      const long long idx = base + lane;
      const bool valid = idx <= last_idx;
      LanePose<kFmtEulerF64> lp;
      edge_sample_pose(es, idx, rot_mode, lp);
      if (COUNT) nposes += valid ? 1 : 0;
      const unsigned hm = check_32_poses<kFmtEulerF64, COUNT, true>(E, ws, cs, valid, lp, lane, true, tally, true,
                                                                    rot_mode != SFFG_ROT_INTERPOLATE);
      if (hm) hit_index = (int)(base + (long long)(__ffs(hm) - 1));
    }
    if (lane == 0) {
      if (split > 1) {
        if (hit_index) atomicMin(fh + eidx, hit_index);
      } else {
        free_out[eidx] = hit_index == 0 ? 1 : 0;
        if (first_hit) first_hit[eidx] = hit_index;
      }
    }
  }
  if (COUNT) {
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) nposes += __shfl_xor_sync(kFull, nposes, sft);
    flush_tally(E, tally, nposes, lane);
  }
}

__global__ void finalize_edges_kernel(const int *fh, long long m, uint8_t *free_out, int32_t *first_hit) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int v = fh[i];
  free_out[i] = v == kNoHit ? 1 : 0;
  if (first_hit) first_hit[i] = v == kNoHit ? 0 : v;
}

// ---------------------------------------------------------------------------------------------------------
// synthetic pose stream: Philox4x32-10, bit-identical to oracle/sff_oracle.c::orc_gen_poses
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox10(unsigned long long seed, unsigned long long index, unsigned stream, unsigned *o) {
  unsigned c0 = (unsigned)index, c1 = (unsigned)(index >> 32), c2 = stream, c3 = 0;
  unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}
__device__ __forceinline__ float u01(unsigned bits) { return __fmul_rn((float)(bits >> 8), 5.9604644775390625e-08f); }
__device__ __forceinline__ float acos_poly(float x) {
  const float ax = fabsf(x);
  float p = -0.0012624911f;
  p = __fadd_rn(__fmul_rn(p, ax), 0.0066700901f);
  p = __fadd_rn(__fmul_rn(p, ax), -0.0170881256f);
  p = __fadd_rn(__fmul_rn(p, ax), 0.0308918810f);
  p = __fadd_rn(__fmul_rn(p, ax), -0.0501743046f);
  p = __fadd_rn(__fmul_rn(p, ax), 0.0889789874f);
  p = __fadd_rn(__fmul_rn(p, ax), -0.2145988016f);
  p = __fadd_rn(__fmul_rn(p, ax), 1.5707963050f);
  const float r = __fmul_rn(__fsqrt_rn(__fsub_rn(1.0f, ax)), p);
  return x < 0.0f ? __fsub_rn(3.14159274f, r) : r;
}

__global__ void gen_poses_kernel(unsigned long long seed, unsigned long long first, long long n, float r0, float r1,
                                 float r2, float r3, float r4, float r5, float *out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned a[4], b[4];
  philox10(seed, first + (unsigned long long)i, 0, a);
  philox10(seed, first + (unsigned long long)i, 1, b);
  float *o = out + 6 * i;
  o[0] = __fadd_rn(r0, __fmul_rn(u01(a[0]), __fsub_rn(r1, r0)));
  o[1] = __fadd_rn(r2, __fmul_rn(u01(a[1]), __fsub_rn(r3, r2)));
  o[2] = __fadd_rn(r4, __fmul_rn(u01(a[2]), __fsub_rn(r5, r4)));
  o[3] = __fadd_rn(-3.14159274f, __fmul_rn(u01(a[3]), 6.28318548f));
  float phi = __fadd_rn(acos_poly(__fsub_rn(1.0f, __fmul_rn(2.0f, u01(b[0])))), 1.57079637f);
  if (u01(b[1]) < 0.5f) phi = __fsub_rn(phi, 3.14159274f);
  o[4] = phi;
  o[5] = __fadd_rn(-3.14159274f, __fmul_rn(u01(b[2]), 6.28318548f));
}

// ---------------------------------------------------------------------------------------------------------
// separation distance per pose (sffg_distance_poses).  Contact is decided by check_32_poses, the verdict path itself; a
// free pose then runs a branch-and-bound walk of the hierarchy whose bound `best` starts at max_dist and shrinks with every
// triangle pair evaluated in FP64.  Every cull below is a rigorous lower bound on a distance, so nothing nearer than the
// final `best` is ever dropped and the result is the minimum over all pairs, whatever the hierarchy.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ double clamp01(double x) { return fmin(fmax(x, 0.0), 1.0); }
__device__ __forceinline__ double dist2(const double *a, const double *b) {
  const double d[3] = {dsub(a[0], b[0]), dsub(a[1], b[1]), dsub(a[2], b[2])};
  return ddot(d, d);
}

// closest points a on [p0, p0 + d1] and b on [q0, q0 + d2] (Ericson, Real-Time Collision Detection 5.1.9, with exact
// zero tests for degenerate segments); returns |a - b|^2
__device__ double seg_seg(const double *p0, const double *d1, const double *q0, const double *d2, double *a, double *b) {
  const double r[3] = {dsub(p0[0], q0[0]), dsub(p0[1], q0[1]), dsub(p0[2], q0[2])};
  const double A = ddot(d1, d1), E = ddot(d2, d2), F = ddot(d2, r);
  double s = 0.0, t = 0.0;
  if (A == 0.0) {
    if (E != 0.0) t = clamp01(ddiv(F, E));
  } else {
    const double C = ddot(d1, r);
    if (E == 0.0) {
      s = clamp01(ddiv(-C, A));
    } else {
      const double B = ddot(d1, d2);
      const double den = dsub(dmul(A, E), dmul(B, B));
      s = den != 0.0 ? clamp01(ddiv(dsub(dmul(B, F), dmul(C, E)), den)) : 0.0;
      t = ddiv(dadd(dmul(B, s), F), E);
      if (t < 0.0) {
        t = 0.0;
        s = clamp01(ddiv(-C, A));
      } else if (t > 1.0) {
        t = 1.0;
        s = clamp01(ddiv(dsub(B, C), A));
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    a[k] = dadd(p0[k], dmul(d1[k], s));
    b[k] = dadd(q0[k], dmul(d2[k], t));
  }
  return dist2(a, b);
}

// foot b of x on the plane of triangle c (9 doubles) when it lies inside the triangle; returns |x - b|^2, or +inf when the
// foot lies outside or the triangle has no area (an edge term of the pair then bounds the distance from below)
__device__ double point_face(const double *x, const double *c, double *b) {
  double u[3], v[3], n[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { u[k] = dsub(c[3 + k], c[k]); v[k] = dsub(c[6 + k], c[k]); b[k] = x[k]; }
  dcross(n, u, v);
  const double nn = ddot(n, n);
  if (nn == 0.0) return CUDART_INF;
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const double *c0 = c + 3 * e, *c1 = c + 3 * (e == 2 ? 0 : e + 1);
    const double ed[3] = {dsub(c1[0], c0[0]), dsub(c1[1], c0[1]), dsub(c1[2], c0[2])};
    const double w[3] = {dsub(x[0], c0[0]), dsub(x[1], c0[1]), dsub(x[2], c0[2])};
    double m[3];
    dcross(m, ed, w);
    if (ddot(m, n) < 0.0) return CUDART_INF;
  }
  const double w[3] = {dsub(x[0], c[0]), dsub(x[1], c[1]), dsub(x[2], c[2])};
  const double s = ddiv(ddot(n, w), nn);
#pragma unroll
  for (int k = 0; k < 3; ++k) b[k] = dsub(x[k], dmul(n[k], s));
  return dist2(x, b);
}

// Sub-problem k of a triangle pair, q = robot triangle and p = obstacle triangle (world frame): k < 9 robot edge k % 3
// against obstacle edge k / 3, k = 9..11 robot vertex k - 9 against the obstacle face, k = 12..14 obstacle vertex k - 12
// against the robot face.  For two disjoint triangles a nearest pair of points lies on an edge of each or is a vertex
// facing the other's interior, so the minimum over the 15 is their distance.  a = robot point, b = obstacle point.
__device__ __noinline__ double pair_subproblem(const double *q, const double *p, int k, double *a, double *b) {
  if (k < 9) {
    const int i = k / 3, j = k - 3 * i, i1 = i == 2 ? 0 : i + 1, j1 = j == 2 ? 0 : j + 1;
    const double dq[3] = {dsub(q[3 * j1], q[3 * j]), dsub(q[3 * j1 + 1], q[3 * j + 1]), dsub(q[3 * j1 + 2], q[3 * j + 2])};
    const double dp[3] = {dsub(p[3 * i1], p[3 * i]), dsub(p[3 * i1 + 1], p[3 * i + 1]), dsub(p[3 * i1 + 2], p[3 * i + 2])};
    return seg_seg(q + 3 * j, dq, p + 3 * i, dp, a, b);
  }
  if (k < 12) {
    const double *x = q + 3 * (k - 9);
    a[0] = x[0]; a[1] = x[1]; a[2] = x[2];
    return point_face(x, p, b);
  }
  const double *x = p + 3 * (k - 12);
  b[0] = x[0]; b[1] = x[1]; b[2] = x[2];
  return point_face(x, q, a);
}

// Lower bound on the distance between obstacle triangle x (robot frame, FP32) and the box [lo, hi]: the gap of the two
// boxes less the position error of x (errpos per coordinate, sqrt(3) errpos in length, allotted 2 errpos; the FP32
// subtractions and the square root are covered by the rest of the allowance and the factor).
__device__ __forceinline__ float tri_box_distance_lb(const XTri &x, const float *lo, const float *hi, float errpos) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float g = fmaxf(fmaxf(min3f(x.v[c], x.v[3 + c], x.v[6 + c]) - hi[c], lo[c] - max3f(x.v[c], x.v[3 + c], x.v[6 + c])), 0.f);
    s += g * g;
  }
  return sqrtf(s) * 0.99999f - 2.0f * errpos;
}

// Lower bound on the distance between a slot box and the robot's oriented box: the largest axis excess of slot_overlaps
// less twice its pad (which covers the FP32 rotation against the pose's FP64 one), the robot-axis excess scaled down for
// the rows of the FP32 R, which are unit only to within 2^-17.
__device__ __forceinline__ float slot_distance_lb(const EnvDev &E, const PoseU &P, const BoxTest &bt, const float4 a, const float4 b) {
  const float tx = (a.x - P.Thi[0]) - bt.o[0], ty = (a.y - P.Thi[1]) - bt.o[1], tz = (a.z - P.Thi[2]) - bt.o[2];
  const float pad = kEpsBox * (fabsf(tx) + fabsf(ty) + fabsf(tz) + b.x + b.y + b.z + bt.rob_sz);
  const float s0 = P.R[0] * tx + P.R[3] * ty + P.R[6] * tz, s1 = P.R[1] * tx + P.R[4] * ty + P.R[7] * tz,
              s2 = P.R[2] * tx + P.R[5] * ty + P.R[8] * tz;
  const float r0 = fabsf(P.R[0]) * b.x + fabsf(P.R[3]) * b.y + fabsf(P.R[6]) * b.z,
              r1 = fabsf(P.R[1]) * b.x + fabsf(P.R[4]) * b.y + fabsf(P.R[7]) * b.z,
              r2 = fabsf(P.R[2]) * b.x + fabsf(P.R[5]) * b.y + fabsf(P.R[8]) * b.z;
  const float ex = fmaxf(fmaxf(fabsf(tx) - (b.x + bt.ra[0]), fabsf(ty) - (b.y + bt.ra[1])), fabsf(tz) - (b.z + bt.ra[2]));
  const float eb = fmaxf(fmaxf(fabsf(s0) - (E.rob_h[0] + r0), fabsf(s1) - (E.rob_h[1] + r1)), fabsf(s2) - (E.rob_h[2] + r2));
  return fmaxf(ex, eb * 0.99999f) - 2.0f * pad;
}

// Lower bound on the distance from the robot (inside its bounding sphere about T) to the obstacle AABB: the arithmetic of
// sphere_hits_root, its pad and a relative allowance taken off.
__device__ __forceinline__ float sphere_root_distance_lb(const EnvDev &E, const float *t, float tlo_mag) {
  const float dx = fmaxf(fabsf(t[0] - E.root_c[0]) - E.root_h[0], 0.f);
  const float dy = fmaxf(fabsf(t[1] - E.root_c[1]) - E.root_h[1], 0.f);
  const float dz = fmaxf(fabsf(t[2] - E.root_c[2]) - E.root_h[2], 0.f);
  const float pad = kEpsBox * (fabsf(t[0]) + fabsf(t[1]) + fabsf(t[2]) + fabsf(E.root_c[0]) + fabsf(E.root_c[1]) +
                               fabsf(E.root_c[2]) + E.root_h[0] + E.root_h[1] + E.root_h[2] + E.rob_radius) + tlo_mag;
  return sqrtf(dx * dx + dy * dy + dz * dz) * 0.99999f - (E.rob_radius + pad);
}

// the float that the slot and pair culls compare with: sqrt(best2) rounded up
__device__ __forceinline__ float cull_bound(double best2) { return __double2float_ru(__dsqrt_ru(best2)); }

// what the branch and bound of one pose has found: the squared distance bound and its two points (warp-uniform)
struct DistBest {
  double d2;
  float cull;
  double pts[6];   // robot point, obstacle point (world frame)
};

// Pair stage of one pose over the candidate triangles ws.tri[0, ntri): transform into the robot frame (FP32), drop those
// whose box is farther than `best` from the robot's box, then lane-per-pair box bounds against each robot triangle; the
// pairs they leave are evaluated in FP64, two pairs per pass on 15 lanes each (lanes 0..14 and 16..30).  The warp minimum
// on (squared distance, lane) makes the outcome independent of timing.
__device__ void distance_pair_stage(const EnvDev &E, WarpScratch &ws, const RobotTri *srob, const PoseU &P, const double *R2,
                                    const double *T2, int lane, int ntri, DistBest &best) {
  const unsigned lt = (1u << lane) - 1u;
  const int half = lane >> 4, k = lane & 15;
  const float inv_n_robot = 1.0f / (float)E.n_robot;
  float rlo[3], rhi[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    rlo[c] = __fsub_rd(E.rob_c[c], E.rob_h[c]);
    rhi[c] = __fadd_ru(E.rob_c[c], E.rob_h[c]);
  }
  for (int base = 0; base < ntri; base += 32) {
    const int cnt = (ntri - base) < 32 ? (ntri - base) : 32;
    bool keep = false;
    XTri x;
    if (lane < cnt) {
      transform_triangle(E, P, ws.tri[base + lane], 0, x);   // (its overlap verdict is no use here)
      keep = !(tri_box_distance_lb(x, rlo, rhi, 2.0f * x.err + kEpsSat * fmaxf(x.mabs, E.rob_radius)) > best.cull);
    }
    const unsigned km = __ballot_sync(kFull, keep);
    if (keep) ws.xt[__popc(km & lt)] = x;
    __syncwarp();
    const int npairs = __popc(km) * E.n_robot;
    for (int pb = 0; pb < npairs; pb += 32) {
      const int pidx = pb + lane;
      const int xi_l = (int)(((float)pidx + 0.5f) * inv_n_robot), r_l = pidx - xi_l * E.n_robot;
      bool open = false;
      if (pidx < npairs) {
        const XTri &xp = ws.xt[xi_l];
        const RobotTri &rt = srob[r_l];
        open = !(tri_box_distance_lb(xp, rt.lo, rt.hi, 2.0f * xp.err + kEpsSat * fmaxf(xp.mabs, rt.qmax)) > best.cull);
      }
      unsigned um = __ballot_sync(kFull, open);
      while (um) {
        const int l0 = __ffs(um) - 1;
        um &= um - 1;
        const int l1 = um ? __ffs(um) - 1 : -1;
        um &= um - 1;   // (0 stays 0)
        const int lmine = half == 0 ? l0 : l1;
        const int xim = __shfl_sync(kFull, xi_l, lmine & 31), rm = __shfl_sync(kFull, r_l, lmine & 31);
        double d2 = CUDART_INF, a[3] = {0.0, 0.0, 0.0}, b[3] = {0.0, 0.0, 0.0};
        if (lmine >= 0 && k < 15) {
          const double *ot = E.tris64 + 9 * (size_t)ws.xt[xim].tri, *rq = E.robot64 + 9 * (size_t)rm;
          double p[9], q[9];
#pragma unroll
          for (int j = 0; j < 9; ++j) p[j] = __ldg(ot + j);
#pragma unroll
          for (int v = 0; v < 3; ++v)   // robot vertex into the world frame: R2 r + T2
#pragma unroll
            for (int i = 0; i < 3; ++i)
              q[3 * v + i] = dadd(dadd(dadd(dmul(R2[3 * i], __ldg(rq + 3 * v)), dmul(R2[3 * i + 1], __ldg(rq + 3 * v + 1))),
                                       dmul(R2[3 * i + 2], __ldg(rq + 3 * v + 2))), T2[i]);
          d2 = pair_subproblem(q, p, k, a, b);
        }
        int wl = lane;
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
          const double od = __shfl_xor_sync(kFull, d2, s);
          const int ol = __shfl_xor_sync(kFull, wl, s);
          if (od < d2 || (od == d2 && ol < wl)) { d2 = od; wl = ol; }
        }
        if (d2 < best.d2) {   // (warp-uniform)
          best.d2 = d2;
          best.cull = cull_bound(d2);
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            best.pts[c] = __shfl_sync(kFull, a[c], wl);
            best.pts[3 + c] = __shfl_sync(kFull, b[c], wl);
          }
        }
      }
    }
    __syncwarp();
  }
}

// branch and bound of one free pose: walk_step with the distance cull, the pair stage after every step that found leaves
template <int FMT>
__device__ void warp_pose_distance(const EnvDev &E, WarpScratch &ws, const CtaShared &cs, const PoseU &P, const LanePose<FMT> &lp,
                                   int src, int lane, DistBest &best) {
  const BoxTest bt = make_box_test(E, P);
  double R2[9], T2[3];
  lp.exact(src, R2, T2, lane);
  const auto near = [&](const float4 a, const float4 b) { return !(slot_distance_lb(E, P, bt, a, b) > best.cull); };
  const unsigned lt = (1u << lane) - 1u;
  Tally tally = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int sp = 0;
  bool first = true;
  while (first || sp > 0) {
    const StepLeaves lv = walk_step<false>(E, ws, cs, first, sp, lane, near, tally);
    first = false;
    if (lv.mine) ws.tri[__popc(lv.mask & lt)] = lv.tri;
    if (sp > kStackCap) {     // never silently drop work: flag the launch as failed
      if (lane == 0) *reinterpret_cast<volatile int *>(E.status) = 1;
      sp = kStackCap;
    }
    __syncwarp();
    if (lv.mask) distance_pair_stage(E, ws, cs.rob, P, R2, T2, lane, __popc(lv.mask), best);
  }
}

template <int FMT>
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSm) distance_poses_kernel(EnvDev E, const void *poses, long long n,
                                                                                   double max_dist, double *dist_out,
                                                                                   double *points_out, int chunk) {
  extern __shared__ __align__(16) unsigned char smem[];
  const CtaShared cs = stage_cta(E, smem, E.n_stage_max);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpScratch &ws = warp_scratch(E, smem, warp);
  const long long nchunks = (n + chunk - 1) / chunk;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  const double max2 = __dmul_ru(max_dist, max_dist);
  Tally tally = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  while (true) {
    unsigned c = 0;
    if (lane == 0) c = atomicAdd(E.work_counter, 1u) - E.work_base;
    c = __shfl_sync(kFull, c, 0);
    if ((long long)c >= nchunks) break;
    const long long i = (long long)c * chunk + lane;
    const bool mine = lane < chunk && i < n;
    LanePose<FMT> lp;
    if (mine) lp.load(poses, i);
    else lp.clear();
    // contact: exactly the verdict of the pose kernel
    const bool hit = (check_32_poses<FMT, false>(E, ws, cs, mine, lp, lane, false, tally) >> lane) & 1u;
    float thi[3], tlo[3], R[9];
    lp.split(thi, tlo);
    const float tlo_mag = fabsf(tlo[0]) + fabsf(tlo[1]) + fabsf(tlo[2]);
    // lane-per-pose cap: a robot whose bounding sphere stays max_dist away from the obstacle box gets max_dist
    const bool open = mine && !hit && E.n_obst > 0 && !((double)sphere_root_distance_lb(E, thi, tlo_mag) >= max_dist);
    double d = hit ? 0.0 : max_dist, pt[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) pt[k] = nan;
    if (open) lp.rot32(R);
    unsigned todo = __ballot_sync(kFull, open);
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      PoseU P;
#pragma unroll
      for (int k = 0; k < 9; ++k) P.R[k] = __shfl_sync(kFull, R[k], src);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        P.Thi[k] = __shfl_sync(kFull, thi[k], src);
        P.Tlo[k] = FMT == kFmtEulerF32 ? 0.f : __shfl_sync(kFull, tlo[k], src);
      }
      DistBest best;
      best.d2 = max2;
      best.cull = cull_bound(max2);
      warp_pose_distance<FMT>(E, ws, cs, P, lp, src, lane, best);
      if (lane == src && best.d2 < max2) {
        const double dd = __dsqrt_rn(best.d2);
        if (dd < max_dist) {
          d = dd > 0.0 ? dd : 4.9406564584124654e-324;   // a free pose never reports contact
#pragma unroll
          for (int k = 0; k < 6; ++k) pt[k] = best.pts[k];
        }
      }
    }
    if (mine) {
      dist_out[i] = d;
      if (points_out) {
#pragma unroll
        for (int k = 0; k < 6; ++k) points_out[6 * i + k] = pt[k];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// separation distance per edge (sffg_distance_edges): the minimum of the pose distance over the samples isPathFree
// checks.  Contact comes from the verdict launch that runs first (free flags and first hits), so this kernel does distance
// work for free edges only.  A warp visits its range of an edge in index order; each sample's branch and bound starts
// from the smallest squared distance found so far on that range, and a sample replaces the record only when its
// reported (rounded) distance is strictly smaller.  A sample that finds nothing below the seed cannot lower the minimum,
// so the record is the minimum over the samples and the lowest index that reports it.
// ---------------------------------------------------------------------------------------------------------
// one warp's result for its range of an edge (split > 1: finalize_distance_edges_kernel reduces them)
struct EdgeDistRec {
  double d;
  int idx;
  int pad;
  double pts[6];
};

__device__ __forceinline__ void store_edge_distance(long long e, double d, int idx, const double *pts, int lane, double *dist_out,
                                                    int32_t *index_out, double *points_out) {
  if (lane == 0) {
    dist_out[e] = d;
    if (index_out) index_out[e] = idx;
  }
  if (points_out) {
#pragma unroll
    for (int k = 0; k < 6; ++k)
      if (lane == k) points_out[6 * e + k] = pts[k];
  }
}

__global__ void __launch_bounds__(kThreads, kMinBlocksPerSm) distance_edges_kernel(EnvDev E, const double *starts,
                                                                                   const double *ends, long long m, double sample,
                                                                                   int rot_mode, double max_dist,
                                                                                   const uint8_t *free_in, const int32_t *first_hit,
                                                                                   double *dist_out, int32_t *index_out,
                                                                                   double *points_out, int split, EdgeDistRec *recs) {
  extern __shared__ __align__(16) unsigned char smem[];
  const CtaShared cs = stage_cta(E, smem, E.n_stage_max);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpScratch &ws = warp_scratch(E, smem, warp);
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  const double max2 = __dmul_ru(max_dist, max_dist);
  const long long units = m * split;
  while (true) {
    unsigned u = 0;
    if (lane == 0) u = atomicAdd(E.work_counter, 1u) - E.work_base;
    u = __shfl_sync(kFull, u, 0);
    if ((long long)u >= units) break;
    const unsigned eidx = u / (unsigned)split;
    const int part = (int)(u - eidx * (unsigned)split);
    double pts[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) pts[k] = nan;
    if (!__ldg(free_in + eidx)) {   // contact: 0 and the first colliding sample (split > 1: the finalize kernel writes it)
      if (split == 1) store_edge_distance(eidx, 0.0, __ldg(first_hit + eidx), pts, lane, dist_out, index_out, points_out);
      continue;
    }
    const EdgeSamples es = edge_samples(starts, ends, eidx, sample);
    // the range of check_edges_kernel's warp `part`
    const long long range_len = (es.S + split - 1) / split;
    const long long first_idx = 1 + (long long)part * range_len;
    const long long last_idx = first_idx + range_len - 1 < es.S ? first_idx + range_len - 1 : es.S;
    double rd = max_dist, seed2 = max2;   // the record's distance and the bound the next sample starts from
    int ri = 0;
    for (long long base = first_idx; base <= last_idx; base += 32) {
      const long long idx = base + lane;
      LanePose<kFmtEulerF64> lp;
      edge_sample_pose(es, idx, rot_mode, lp);
      float thi[3], tlo[3], R[9];
      lp.split(thi, tlo);
      const float tlo_mag = fabsf(tlo[0]) + fabsf(tlo[1]) + fabsf(tlo[2]);
      // lane-per-sample cap: a robot whose bounding sphere stays the record's distance away from the obstacle box cannot
      // lower it (re-checked against the record as it shrinks)
      const double lb = idx <= last_idx && E.n_obst > 0 ? (double)sphere_root_distance_lb(E, thi, tlo_mag) : CUDART_INF;
      const bool open = !(lb >= rd);
      if (open) lp.rot32(R);
      unsigned todo = __ballot_sync(kFull, open);
      while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        if (__shfl_sync(kFull, lb, src) >= rd) continue;
        PoseU P;
#pragma unroll
        for (int k = 0; k < 9; ++k) P.R[k] = __shfl_sync(kFull, R[k], src);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          P.Thi[k] = __shfl_sync(kFull, thi[k], src);
          P.Tlo[k] = __shfl_sync(kFull, tlo[k], src);
        }
        DistBest best;
        best.d2 = seed2;
        best.cull = cull_bound(seed2);
        warp_pose_distance<kFmtEulerF64>(E, ws, cs, P, lp, src, lane, best);
        if (best.d2 < seed2) {   // (warp-uniform)
          seed2 = best.d2;
          const double dd = __dsqrt_rn(best.d2);
          const double dr = dd > 0.0 ? dd : 4.9406564584124654e-324;   // what the pose query reports for this sample
          if (dd < max_dist && dr < rd) {
            rd = dr;
            ri = (int)(base + src);
#pragma unroll
            for (int k = 0; k < 6; ++k) pts[k] = best.pts[k];
          }
        }
      }
    }
    if (split == 1) {
      store_edge_distance(eidx, rd, ri, pts, lane, dist_out, index_out, points_out);
    } else {
      EdgeDistRec *r = recs + u;
      if (lane == 0) {
        r->d = rd;
        r->idx = ri;
      }
#pragma unroll
      for (int k = 0; k < 6; ++k)
        if (lane == k) r->pts[k] = pts[k];
    }
  }
}

// split > 1: the records of an edge's warps, in index order; the first one with the smallest distance holds the lowest
// index that reports it
__global__ void finalize_distance_edges_kernel(const EdgeDistRec *recs, int split, long long m, double max_dist,
                                               const uint8_t *free_in, const int32_t *first_hit, double *dist_out,
                                               int32_t *index_out, double *points_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  double d = 0.0;
  int idx = first_hit[i];
  const double *pts = nullptr;
  if (free_in[i]) {
    d = max_dist;
    idx = 0;
    for (int p = 0; p < split; ++p) {
      const EdgeDistRec &r = recs[i * split + p];
      if (r.d < d) {
        d = r.d;
        idx = r.idx;
        pts = r.pts;
      }
    }
  }
  dist_out[i] = d;
  if (index_out) index_out[i] = idx;
  if (points_out)
    for (int k = 0; k < 6; ++k) points_out[6 * i + k] = pts ? pts[k] : nan;
}

// ---------------------------------------------------------------------------------------------------------
// continuous edge check (sffg_sweep_edges): conservative advancement on the pose distance over the motion
// pose(tau) = start + tau (end - start), tau in [0, 1].  No robot point moves faster than mu per unit tau, so a pose at
// distance D >= margin certifies every pose up to tau + (D - margin / 2) / mu at distance >= margin / 2.  [0, 1] is cut into
// kSweepPieces fixed pieces, one lane each; a piece advances from its own start, so its outcome does not depend on which
// warp runs it.  A step's D is 0 on contact (check_32_poses, the verdict path), else min(d, C) with the cap
// C = mu (b - tau) + margin: the FP64 branch-and-bound minimum seeded at C^2, or C itself when the lane's bounding-sphere
// bound already proves d >= C.  Both ways D is C or the cap-independent minimum, so it is deterministic.
// ---------------------------------------------------------------------------------------------------------
constexpr int kSweepPieces = 32;

// one warp's lowest stopped piece of an edge (split > 1: finalize_sweep_edges_kernel reduces them), kSweepPieces for none
struct SweepRec {
  double t, d;
  int piece;
  int pad;
};

// the motion of one edge and mu, its motion bound rounded up: |f_xyz - s_xyz|, plus rho times the sum of the wrapped angle
// differences when the angles are interpolated (|omega| <= the sum of the Euler angle rates, |robot point| <= rho)
struct SweepEdge {
  double s[6], dir[3], adir[3];
  double mu;
};
__device__ __forceinline__ SweepEdge sweep_edge(const EnvDev &E, const double *starts, const double *ends, unsigned eidx,
                                                int rot_mode) {
  SweepEdge ed;
  double l2 = 0.0, turn = 0.0;
#pragma unroll
  for (int k = 0; k < 6; ++k) ed.s[k] = __ldg(starts + 6 * (size_t)eidx + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    ed.dir[k] = dsub(__ldg(ends + 6 * (size_t)eidx + k), ed.s[k]);
    ed.adir[k] = wrap_pi(dsub(__ldg(ends + 6 * (size_t)eidx + 3 + k), ed.s[3 + k]));
    l2 = __dadd_ru(l2, __dmul_ru(ed.dir[k], ed.dir[k]));
    turn = __dadd_ru(turn, fabs(ed.adir[k]));
  }
  ed.mu = __dsqrt_ru(l2);
  if (rot_mode == SFFG_ROT_INTERPOLATE) ed.mu = __dadd_ru(ed.mu, __dmul_ru((double)E.rob_radius, turn));
  return ed;
}
// pose(tau): each operation rounded to nearest, no FMA; reference mode keeps the identity rotation
__device__ __forceinline__ void sweep_pose(const SweepEdge &ed, double tau, int rot_mode, LanePose<kFmtEulerF64> &lp) {
  lp.clear();
  lp.identity = rot_mode != SFFG_ROT_INTERPOLATE;
#pragma unroll
  for (int k = 0; k < 3; ++k) lp.t[k] = dadd(ed.s[k], dmul(tau, ed.dir[k]));
  if (rot_mode == SFFG_ROT_INTERPOLATE) {
#pragma unroll
    for (int k = 0; k < 3; ++k) lp.a[k] = dadd(ed.s[3 + k], dmul(tau, ed.adir[k]));
  }
}

__device__ __forceinline__ void store_sweep(long long e, int piece, double t, double d, uint8_t *clear_out, double *t_out,
                                            double *dist_out) {
  clear_out[e] = piece == kSweepPieces ? 1 : 0;
  if (t_out) t_out[e] = t;
  if (dist_out) dist_out[e] = d;
}

// Units are (edge, part): warp `part` of an edge takes pieces part * (kSweepPieces / split) .. + kSweepPieces / split - 1,
// piece = first + lane.  Every round builds the current pose of each live piece, decides contact for all of them in one
// check_32_poses call, runs the branch and bound warp-cooperatively for the lanes the sphere bound leaves open, then
// advances each piece.  A piece above a known stop (this warp's, or with split > 1 another warp's, published in `stop`)
// cannot change the result and is dropped.
__global__ void __launch_bounds__(kThreads, kMinBlocksPerSm) sweep_edges_kernel(EnvDev E, const double *starts, const double *ends,
                                                                                long long m, int rot_mode, double margin,
                                                                                uint8_t *clear_out, double *t_out, double *dist_out,
                                                                                int split, int *stop, SweepRec *recs) {
  extern __shared__ __align__(16) unsigned char smem[];
  const CtaShared cs = stage_cta(E, smem, E.n_stage_max);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpScratch &ws = warp_scratch(E, smem, warp);
  const double half = 0.5 * margin;
  const int per = kSweepPieces / split;
  const long long units = m * split;
  Tally tally = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  while (true) {
    unsigned u = 0;
    if (lane == 0) u = atomicAdd(E.work_counter, 1u) - E.work_base;
    u = __shfl_sync(kFull, u, 0);
    if ((long long)u >= units) break;
    const unsigned eidx = u / (unsigned)split;
    const int part = (int)(u - eidx * (unsigned)split);
    const SweepEdge ed = sweep_edge(E, starts, ends, eidx, rot_mode);
    // a motionless edge is one pose (every piece would repeat piece 0); a non-finite one is never clear
    const bool finite = ed.mu <= DBL_MAX;
    const int npieces = ed.mu > 0.0 ? kSweepPieces : 1;
    const int piece = part * per + lane;
    bool live = finite && lane < per && piece < npieces;
    double tau = (double)piece * (1.0 / kSweepPieces);
    const double b = (double)(piece + 1) * (1.0 / kSweepPieces);
    int rp = finite ? kSweepPieces : 0;   // this warp's lowest stopped piece, its tau and its D
    double rt = finite ? 1.0 : 0.0, rd = finite ? margin : __longlong_as_double(0x7ff8000000000000ll);
    while (true) {
      int lowest = rp;
      if (split > 1) lowest = min(lowest, *reinterpret_cast<volatile int *>(stop + eidx));
      live = live && piece < lowest;
      if (!__any_sync(kFull, live)) break;
      LanePose<kFmtEulerF64> lp;
      sweep_pose(ed, tau, rot_mode, lp);
      float thi[3], tlo[3], R[9];
      lp.split(thi, tlo);
      const float tlo_mag = fabsf(tlo[0]) + fabsf(tlo[1]) + fabsf(tlo[2]);
      const double cap = __dadd_ru(__dmul_ru(ed.mu, __dsub_ru(b, tau)), margin);
      // the sphere bound proves d >= cap (so no contact either): D = cap without the walk
      const bool near = live && E.n_obst > 0 && !((double)sphere_root_distance_lb(E, thi, tlo_mag) >= cap);
      const bool hit = (check_32_poses<kFmtEulerF64, false>(E, ws, cs, near, lp, lane, false, tally) >> lane) & 1u;
      double D = hit ? 0.0 : cap;
      const bool open = near && !hit;
      if (open) lp.rot32(R);
      unsigned todo = __ballot_sync(kFull, open);
      while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        PoseU P;
#pragma unroll
        for (int k = 0; k < 9; ++k) P.R[k] = __shfl_sync(kFull, R[k], src);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          P.Thi[k] = __shfl_sync(kFull, thi[k], src);
          P.Tlo[k] = __shfl_sync(kFull, tlo[k], src);
        }
        const double c = __shfl_sync(kFull, cap, src), c2 = __dmul_ru(c, c);
        DistBest best;
        best.d2 = c2;
        best.cull = cull_bound(c2);
        warp_pose_distance<kFmtEulerF64>(E, ws, cs, P, lp, src, lane, best);
        if (lane == src && best.d2 < c2) {
          const double dd = __dsqrt_rn(best.d2);
          if (dd < c) D = dd > 0.0 ? dd : 4.9406564584124654e-324;   // what the pose query reports for this pose
        }
      }
      const bool stopped = live && D < margin;
      if (live && !stopped) {
        if (ed.mu == 0.0) {
          live = false;   // clear: the whole motion is this pose
        } else {
          // the step rounds down (mu is rounded up); when mu > 2^51 margin it can fall below one ulp of tau, and the piece
          // moves to the next double
          double next = __dadd_rd(tau, __ddiv_rd(__dsub_rd(D, half), ed.mu));
          if (next == tau) next = nextafter(tau, 2.0);
          tau = next;
          live = tau < b;
        }
      }
      const unsigned sm = __ballot_sync(kFull, stopped);
      if (sm) {
        const int l = __ffs(sm) - 1;   // lanes hold increasing pieces: the lowest stopped piece of this round
        const int p = __shfl_sync(kFull, piece, l);
        const double t = __shfl_sync(kFull, tau, l), d = __shfl_sync(kFull, D, l);
        if (p < rp) {
          rp = p;
          rt = t;
          rd = d;
          if (split > 1 && lane == 0) atomicMin(stop + eidx, p);
        }
      }
      live = live && !stopped;
    }
    if (split == 1) {
      if (lane == 0) store_sweep(eidx, rp, rt, rd, clear_out, t_out, dist_out);
    } else if (lane == 0) {
      recs[u].t = rt;
      recs[u].d = rd;
      recs[u].piece = rp;
    }
  }
}

// split > 1: the lowest stopped piece over an edge's warps decides; none stopped = clear
__global__ void finalize_sweep_edges_kernel(const SweepRec *recs, int split, long long m, double margin, uint8_t *clear_out,
                                            double *t_out, double *dist_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  int piece = kSweepPieces;
  double t = 1.0, d = margin;
  for (int p = 0; p < split; ++p) {
    const SweepRec &r = recs[i * split + p];
    if (r.piece < piece) {
      piece = r.piece;
      t = r.t;
      d = r.d;
    }
  }
  store_sweep(i, piece, t, d, clear_out, t_out, dist_out);
}


}  // namespace

// cudaFuncSetAttribute + occupancy are queried once per kernel instantiation (and per shared-memory size)
struct KernelCfg {
  size_t smem = ~size_t(0);
  int per_sm = 1;
  cudaError_t err = cudaSuccess;
};
template <auto Kernel>
static KernelCfg kernel_cfg(size_t smem) {
  static KernelCfg c;
  static std::mutex mu;   // environments of different host threads share the per-kernel cache
  std::lock_guard<std::mutex> lock(mu);
  if (c.smem != smem) {
    c.smem = smem;
    c.err = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 0;
    if (c.err == cudaSuccess &&
        (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, Kernel, kThreads, smem) != cudaSuccess || per_sm < 1))
      per_sm = 1;
    c.per_sm = per_sm < 1 ? 1 : per_sm;
  }
  return c;
}

size_t collide_smem_bytes(int n_robot, int n_stage_max) {
  return (size_t)n_robot * sizeof(RobotTri) + (size_t)2 * kTopSlots * sizeof(float4) +
         (size_t)n_stage_max * kWide * 2 * sizeof(float4) + (size_t)kWarpsPerBlock * sizeof(WarpScratch);
}


// launches `want` CTAs of kThreads, or as many as are resident at once if fewer (the kernels pull their work units from
// E.work_counter); the grid size goes to `*grid` for the work-counter bookkeeping
template <auto Kernel, class... Args>
static cudaError_t launch_resident(long long want, size_t smem, cudaStream_t stream, const LaunchCfg &cfg, int *grid, Args... args) {
  const KernelCfg kc = kernel_cfg<Kernel>(smem);
  if (kc.err != cudaSuccess) return kc.err;
  *grid = cfg.sm_count * kc.per_sm;
  if (want < *grid) *grid = (int)want;
  Kernel<<<*grid, kThreads, smem, stream>>>(args...);
  return cudaGetLastError();
}

template <int FMT>
static cudaError_t launch_poses_fmt(const EnvDev &env, const void *d_poses, int64_t n, const OutSet &d_verdict, const GatherSync &gs,
                                    cudaStream_t stream, const LaunchCfg &cfg, bool count, int chunk, int *grid) {
  const size_t smem = collide_smem_bytes(env.n_robot, env.n_stage_max);
  const long long chunks = (n + chunk - 1) / chunk;
  const long long want = (chunks + kWarpsPerBlock - 1) / kWarpsPerBlock;
  if (count)
    return launch_resident<collide_poses_kernel<FMT, true>>(want, smem, stream, cfg, grid, env, d_poses, (long long)n, d_verdict, gs, chunk);
  return launch_resident<collide_poses_kernel<FMT, false>>(want, smem, stream, cfg, grid, env, d_poses, (long long)n, d_verdict, gs, chunk);
}

// ---------------------------------------------------------------------------------------------------------
// cross-GPU completion barrier for the peer-store gather (one CTA of 32 threads, thread r talks to rank r)
// ---------------------------------------------------------------------------------------------------------
// signal == true : publish `epoch` to every rank (no wait)      -- what an empty shard owes its peers
// signal == false: wait until every rank has published >= epoch -- what a consumer of the gathered results enqueues
__global__ void peer_barrier_kernel(FlagSet f, unsigned epoch, bool signal, int *status) {
  if (signal) {
    const int r = threadIdx.x;
    if (r >= f.n) return;
    __threadfence_system();   // everything this stream did before is ordered before the signal
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f.p[r] + f.me), "r"(epoch) : "memory");
  } else if (threadIdx.x == 0) {
    wait_flags(f, epoch, status);
  }
}

cudaError_t launch_peer_barrier(const FlagSet &flags, unsigned epoch, bool signal, int *d_status, cudaStream_t stream) {
  peer_barrier_kernel<<<1, 32, 0, stream>>>(flags, epoch, signal, d_status);
  return cudaGetLastError();
}

// poses per work unit of the pose kernels: enough units for ~2 per resident warp (at 2 CTAs/SM), capped at a full warp
static int pose_chunk(int64_t n, const LaunchCfg &cfg) {
  int chunk = 32;
  const long long warps = (long long)cfg.sm_count * 2 * kWarpsPerBlock * 2;
  while (chunk > 1 && (n + chunk - 1) / chunk < warps) chunk >>= 1;
  return chunk;
}

// every warp of the grid leaves its loop through exactly one failing fetch, so a launch consumes
// (units + grid * warps) values of the shared counter; the host advances the base instead of resetting the counter
cudaError_t launch_collide_poses(const EnvDev &env_in, const void *d_poses, int pose_fmt, int64_t n, uint8_t *d_verdict,
                                 cudaStream_t stream, const LaunchCfg &cfg, bool count, unsigned *work_base_io) {
  OutSet one;
  one.n = 1;
  one.p[0] = d_verdict;
  GatherSync none{};
  return launch_collide_poses_gather(env_in, d_poses, pose_fmt, n, one, none, stream, cfg, count, work_base_io);
}

cudaError_t launch_collide_poses_gather(const EnvDev &env_in, const void *d_poses, int pose_fmt, int64_t n, const OutSet &d_verdict,
                                        const GatherSync &gs, cudaStream_t stream, const LaunchCfg &cfg, bool count,
                                        unsigned *work_base_io) {
  if (n <= 0) {
    // an empty shard still owes its peers the completion signal (after waiting like a real launch would)
    if (gs.flags.n > 0) {
      cudaError_t e = cudaSuccess;
      if (gs.wait_epoch != 0) e = launch_peer_barrier(gs.flags, gs.wait_epoch, false, env_in.status, stream);
      if (e == cudaSuccess) e = launch_peer_barrier(gs.flags, gs.signal_epoch, true, nullptr, stream);
      return e;
    }
    return cudaSuccess;
  }
  EnvDev env = env_in;
  env.work_base = *work_base_io;
  int grid = 0;
  const int chunk = pose_chunk(n, cfg);
  cudaError_t e = cudaErrorInvalidValue;
  switch (pose_fmt) {
    case 0: e = launch_poses_fmt<kFmtEulerF32>(env, d_poses, n, d_verdict, gs, stream, cfg, count, chunk, &grid); break;
    case 1: e = launch_poses_fmt<kFmtEulerF64>(env, d_poses, n, d_verdict, gs, stream, cfg, count, chunk, &grid); break;
    case 2: e = launch_poses_fmt<kFmtMatrixF64>(env, d_poses, n, d_verdict, gs, stream, cfg, count, chunk, &grid); break;
  }
  if (e == cudaSuccess) *work_base_io += (unsigned)((n + chunk - 1) / chunk) + (unsigned)grid * kWarpsPerBlock;
  return e;
}

cudaError_t launch_distance_poses(const EnvDev &env_in, const void *d_poses, int pose_fmt, int64_t n, double max_dist,
                                  double *d_dist, double *d_points, cudaStream_t stream, const LaunchCfg &cfg,
                                  unsigned *work_base_io) {
  if (n <= 0) return cudaSuccess;
  EnvDev env = env_in;
  env.work_base = *work_base_io;
  const int chunk = pose_chunk(n, cfg);
  const size_t smem = collide_smem_bytes(env.n_robot, env.n_stage_max);
  const long long chunks = (n + chunk - 1) / chunk;
  const long long want = (chunks + kWarpsPerBlock - 1) / kWarpsPerBlock;
  int grid = 0;
  cudaError_t e = cudaErrorInvalidValue;
  if (pose_fmt == kFmtEulerF32)
    e = launch_resident<distance_poses_kernel<kFmtEulerF32>>(want, smem, stream, cfg, &grid, env, d_poses, (long long)n, max_dist,
                                                             d_dist, d_points, chunk);
  else if (pose_fmt == kFmtEulerF64)
    e = launch_resident<distance_poses_kernel<kFmtEulerF64>>(want, smem, stream, cfg, &grid, env, d_poses, (long long)n, max_dist,
                                                             d_dist, d_points, chunk);
  if (e == cudaSuccess) *work_base_io += (unsigned)chunks + (unsigned)grid * kWarpsPerBlock;
  return e;
}

cudaError_t launch_check_edges(const EnvDev &env_in, const double *d_starts, const double *d_ends, int64_t m,
                               double sample_dist, int rot_mode, uint8_t *d_free, int32_t *d_first_hit, cudaStream_t stream,
                               const LaunchCfg &cfg, bool count, unsigned *work_base_io, int *d_fh_scratch) {
  if (m <= 0) return cudaSuccess;
  EnvDev env = env_in;
  env.work_base = *work_base_io;
  const size_t smem = collide_smem_bytes(env.n_robot, env.n_stage_max);
  // warps per edge: enough units for ~2 per resident warp, at most 32 (needs the scratch array)
  int split = 1;
  const long long warps = (long long)cfg.sm_count * kWarpsPerBlock * kEdgeUnitsPerWarp;
  if (d_fh_scratch)
    while (split < 32 && m * split < warps) split <<= 1;
  const long long units = m * split;
  const long long want = (units + kWarpsPerBlock - 1) / kWarpsPerBlock;
  cudaError_t e;
  if (split > 1 && (e = cudaMemsetAsync(d_fh_scratch, 0x7f, (size_t)m * sizeof(int), stream)) != cudaSuccess) return e;
  int grid = 0;
  if (count)
    e = launch_resident<check_edges_kernel<true>>(want, smem, stream, cfg, &grid, env, d_starts, d_ends, (long long)m, sample_dist,
                                                  rot_mode, d_free, d_first_hit, split, d_fh_scratch);
  else
    e = launch_resident<check_edges_kernel<false>>(want, smem, stream, cfg, &grid, env, d_starts, d_ends, (long long)m, sample_dist,
                                                   rot_mode, d_free, d_first_hit, split, d_fh_scratch);
  if (e != cudaSuccess) return e;
  *work_base_io += (unsigned)units + (unsigned)grid * kWarpsPerBlock;
  if (split > 1) {
    finalize_edges_kernel<<<(unsigned)((m + 255) / 256), 256, 0, stream>>>(d_fh_scratch, (long long)m, d_free, d_first_hit);
    e = cudaGetLastError();
  }
  return e;
}

// warps per edge of the edge distance kernel: the rule of launch_check_edges, several only with a record slot each
static int distance_edges_split(int64_t m, const LaunchCfg &cfg, bool have_recs) {
  int split = 1;
  const long long warps = (long long)cfg.sm_count * kWarpsPerBlock * kEdgeUnitsPerWarp;
  if (have_recs)
    while (split < 32 && m * split < warps) split <<= 1;
  return split;
}

size_t distance_edges_rec_bytes(int64_t m, const LaunchCfg &cfg) {
  const int split = distance_edges_split(m, cfg, true);
  return split > 1 ? (size_t)m * split * sizeof(EdgeDistRec) : 0;
}

cudaError_t launch_distance_edges(const EnvDev &env, const double *d_starts, const double *d_ends, int64_t m, double sample_dist,
                                  int rot_mode, double max_dist, double *d_dist, int32_t *d_index, double *d_points,
                                  cudaStream_t stream, const LaunchCfg &cfg, unsigned *work_base_io,
                                  const EdgeDistScratch &scr) {
  if (m <= 0) return cudaSuccess;
  cudaError_t e = launch_check_edges(env, d_starts, d_ends, m, sample_dist, rot_mode, scr.free, scr.first_hit, stream, cfg, false,
                                     work_base_io, scr.fh);
  if (e != cudaSuccess) return e;
  EnvDev v = env;
  v.work_base = *work_base_io;
  const int split = distance_edges_split(m, cfg, scr.recs != nullptr);
  const long long units = m * split;
  const long long want = (units + kWarpsPerBlock - 1) / kWarpsPerBlock;
  int grid = 0;
  e = launch_resident<distance_edges_kernel>(want, collide_smem_bytes(v.n_robot, v.n_stage_max), stream, cfg, &grid, v, d_starts,
                                             d_ends, (long long)m, sample_dist, rot_mode, max_dist, (const uint8_t *)scr.free,
                                             (const int32_t *)scr.first_hit, d_dist, d_index, d_points, split,
                                             (EdgeDistRec *)scr.recs);
  if (e != cudaSuccess) return e;
  *work_base_io += (unsigned)units + (unsigned)grid * kWarpsPerBlock;
  if (split > 1) {
    finalize_distance_edges_kernel<<<(unsigned)((m + 255) / 256), 256, 0, stream>>>(
        (const EdgeDistRec *)scr.recs, split, (long long)m, max_dist, scr.free, scr.first_hit, d_dist, d_index, d_points);
    e = cudaGetLastError();
  }
  return e;
}

size_t sweep_edges_rec_bytes(int64_t m, const LaunchCfg &cfg) {
  const int split = distance_edges_split(m, cfg, true);
  return split > 1 ? (size_t)m * split * sizeof(SweepRec) : 0;
}

cudaError_t launch_sweep_edges(const EnvDev &env_in, const double *d_starts, const double *d_ends, int64_t m, int rot_mode,
                               double margin, uint8_t *d_clear, double *d_t, double *d_dist, cudaStream_t stream,
                               const LaunchCfg &cfg, unsigned *work_base_io, const SweepScratch &scr) {
  if (m <= 0) return cudaSuccess;
  EnvDev env = env_in;
  env.work_base = *work_base_io;
  const int split = distance_edges_split(m, cfg, scr.stop != nullptr && scr.recs != nullptr);
  const long long units = m * split;
  const long long want = (units + kWarpsPerBlock - 1) / kWarpsPerBlock;
  cudaError_t e;
  if (split > 1 && (e = cudaMemsetAsync(scr.stop, 0x7f, (size_t)m * sizeof(int), stream)) != cudaSuccess) return e;
  int grid = 0;
  e = launch_resident<sweep_edges_kernel>(want, collide_smem_bytes(env.n_robot, env.n_stage_max), stream, cfg, &grid, env, d_starts,
                                          d_ends, (long long)m, rot_mode, margin, d_clear, d_t, d_dist, split, scr.stop,
                                          (SweepRec *)scr.recs);
  if (e != cudaSuccess) return e;
  *work_base_io += (unsigned)units + (unsigned)grid * kWarpsPerBlock;
  if (split > 1) {
    finalize_sweep_edges_kernel<<<(unsigned)((m + 255) / 256), 256, 0, stream>>>((const SweepRec *)scr.recs, split, (long long)m,
                                                                                  margin, d_clear, d_t, d_dist);
    e = cudaGetLastError();
  }
  return e;
}

cudaError_t launch_gen_poses(uint64_t seed, uint64_t first, int64_t n, const float range[6], float *d_out,
                             cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  const int threads = 256;
  const long long blocks = (n + threads - 1) / threads;
  gen_poses_kernel<<<(unsigned)blocks, threads, 0, stream>>>(seed, first, (long long)n, range[0], range[1], range[2],
                                                             range[3], range[4], range[5], d_out);
  return cudaGetLastError();
}

}  // namespace sffg
