// clearance_grid.cu -- the clearance grid: how it is sized, its build on the GPU and the owner of its device arrays.
//
// One warp per obstacle triangle marks the cells whose centre lies within `reach` of the triangle, and lowers, per cell,
// the bounds of the plane build and the keys of the witness build.  The pose and edge kernels read the result through
// GridDev (collide_kernels.cuh), where the cell arithmetic and the plane-record encoding live.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <utility>

#include "clearance_grid.cuh"

namespace sffg {
namespace {

__device__ __forceinline__ float point_tri_dist2(const float *p, const float *a, const float *b, const float *c) {
  // closest point on a triangle (Voronoi-region walk), squared distance
  const float ab[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, ac[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
  const float ap[3] = {p[0] - a[0], p[1] - a[1], p[2] - a[2]};
  const float d1 = ab[0] * ap[0] + ab[1] * ap[1] + ab[2] * ap[2], d2 = ac[0] * ap[0] + ac[1] * ap[1] + ac[2] * ap[2];
  float q[3];
  if (d1 <= 0.f && d2 <= 0.f) { q[0] = a[0]; q[1] = a[1]; q[2] = a[2]; }
  else {
    const float bp[3] = {p[0] - b[0], p[1] - b[1], p[2] - b[2]};
    const float d3 = ab[0] * bp[0] + ab[1] * bp[1] + ab[2] * bp[2], d4 = ac[0] * bp[0] + ac[1] * bp[1] + ac[2] * bp[2];
    if (d3 >= 0.f && d4 <= d3) { q[0] = b[0]; q[1] = b[1]; q[2] = b[2]; }
    else {
      const float vc = d1 * d4 - d3 * d2;
      if (vc <= 0.f && d1 >= 0.f && d3 <= 0.f) {
        const float v = d1 / (d1 - d3);
        q[0] = a[0] + v * ab[0]; q[1] = a[1] + v * ab[1]; q[2] = a[2] + v * ab[2];
      } else {
        const float cp[3] = {p[0] - c[0], p[1] - c[1], p[2] - c[2]};
        const float d5 = ab[0] * cp[0] + ab[1] * cp[1] + ab[2] * cp[2], d6 = ac[0] * cp[0] + ac[1] * cp[1] + ac[2] * cp[2];
        if (d6 >= 0.f && d5 <= d6) { q[0] = c[0]; q[1] = c[1]; q[2] = c[2]; }
        else {
          const float vb = d5 * d2 - d1 * d6;
          if (vb <= 0.f && d2 >= 0.f && d6 <= 0.f) {
            const float w = d2 / (d2 - d6);
            q[0] = a[0] + w * ac[0]; q[1] = a[1] + w * ac[1]; q[2] = a[2] + w * ac[2];
          } else {
            const float va = d3 * d6 - d5 * d4;
            if (va <= 0.f && (d4 - d3) >= 0.f && (d5 - d6) >= 0.f) {
              const float w = (d4 - d3) / ((d4 - d3) + (d5 - d6));
              q[0] = b[0] + w * (c[0] - b[0]); q[1] = b[1] + w * (c[1] - b[1]); q[2] = b[2] + w * (c[2] - b[2]);
            } else {
              const float den = 1.f / (va + vb + vc), v = vb * den, w = vc * den;
              q[0] = a[0] + ab[0] * v + ac[0] * w; q[1] = a[1] + ab[1] * v + ac[1] * w; q[2] = a[2] + ab[2] * v + ac[2] * w;
            }
          }
        }
      }
    }
  }
  const float dx = p[0] - q[0], dy = p[1] - q[1], dz = p[2] - q[2];
  return dx * dx + dy * dy + dz * dz;
}

// plane direction of pass slot j (the 26 directions skip d = 13)
__device__ __forceinline__ int pass_dir(int dir0, int j) {
  const int k = dir0 + j;
  return k < kNoPlaneDir ? k : k + 1;
}
// m.p rounded down: m has entries in {-1, 0, 1}, so the products are exact and only the two sums round
__device__ __forceinline__ float dot_dir_rd(const float *m, const float *p) {
  return __fadd_rd(__fadd_rd(m[0] * p[0], m[1] * p[1]), m[2] * p[2]);
}

// Marks (bits != null) the cells within `reach` of each triangle and lowers mins[j][cell] to the triangle's bound
// min over its vertices of m_d.p, d = pass_dir(dir0, j) for j < ndir: the float vertices, rounded down, minus
// |m|_1 times their representation error, so the bound holds for the FP64 triangle.
// With `keys` (witness passes, ndir = 0) it lowers keys[cell] to (distance^2 bits, triangle) of every triangle that marks
// the cell, except the cell's first witness `excl[cell].x` when `excl` is given.
constexpr int kClearanceThreads = 256;
__global__ void build_clearance_kernel(const float4 *__restrict__ tris, int n_tris, GridDev g, float reach, unsigned *bits, int *mins,
                                       int dir0, int ndir, unsigned long long *keys, const int2 *excl) {
  __shared__ int tri_min[kClearanceThreads / 32][32];
  const int lane = threadIdx.x & 31;
  const int t = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (t >= n_tris) return;
  const float4 v0 = __ldg(tris + 3 * (size_t)t), v1 = __ldg(tris + 3 * (size_t)t + 1), v2 = __ldg(tris + 3 * (size_t)t + 2);
  const float a[3] = {v0.x, v0.y, v0.z}, b[3] = {v1.x, v1.y, v1.z}, c[3] = {v2.x, v2.y, v2.z};
  int *tmin = tri_min[threadIdx.x >> 5];
  if (lane < ndir) {
    float m[3];
    plane_dir(pass_dir(dir0, lane), m);
    const float l1 = fabsf(m[0]) + fabsf(m[1]) + fabsf(m[2]);
    const float lo = fminf(dot_dir_rd(m, a), fminf(dot_dir_rd(m, b), dot_dir_rd(m, c)));
    tmin[lane] = float_to_ordered(__fsub_rd(lo, __fmul_ru(l1, v0.w)));
  }
  __syncwarp();
  const float inv = 1.0f / g.h;   // (not g.inv_h, which is rounded from double)
  int lo[3], hi[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float mn = fminf(a[k], fminf(b[k], c[k])) - reach, mx = fmaxf(a[k], fmaxf(b[k], c[k])) + reach;
    lo[k] = max(0, (int)floorf((mn - g.o[k]) * inv) - 1);
    hi[k] = min(g.n[k] - 1, (int)floorf((mx - g.o[k]) * inv) + 1);
  }
  const int sx = hi[0] - lo[0] + 1, sy = hi[1] - lo[1] + 1, sz = hi[2] - lo[2] + 1;
  if (sx <= 0 || sy <= 0 || sz <= 0) return;
  const long long total = (long long)sx * sy * sz;
  const float r2 = reach * reach;
  for (long long i = lane; i < total; i += 32) {
    const int ix = lo[0] + (int)(i % sx), iy = lo[1] + (int)((i / sx) % sy), iz = lo[2] + (int)(i / ((long long)sx * sy));
    float p[3];
    cell_centre(g, ix, iy, iz, p);
    const float d2 = point_tri_dist2(p, a, b, c);
    if (!(d2 > r2)) {   // NaN (degenerate triangle) marks the cell: never optimistic
      const unsigned cell = cell_index(g, ix, iy, iz);
      if (bits) atomicOr(bits + (cell >> 5), 1u << (cell & 31));
      const long long cells = cell_count(g);
      for (int j = 0; j < ndir; ++j) atomicMin(mins + j * cells + cell, tmin[j]);
      if (keys && !(excl && excl[cell].x == t))   // (d2 >= 0 or NaN: its bits order like the value, NaN last)
        atomicMin(keys + cell, ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)t);
    }
  }
}

// Each marked cell keeps, of the directions of this pass and the record it already holds (`first`: none), the one with the
// most room c - max_{x in cell} m.x per unit length of m -- what the robot's origin may use before it reaches the plane.
// A record with no room at all is the no-plane record.  Unmarked cells get the no-plane record on the first pass.
__global__ void choose_planes_kernel(GridDev g, const int *__restrict__ mins, int dir0, int ndir, bool first, unsigned *planes) {
  const long long cells = cell_count(g);
  const long long cell = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= cells) return;
  if (!((__ldg(g.bits + (cell >> 5)) >> (cell & 31)) & 1u)) {
    if (first) planes[cell] = kNoPlane;
    return;
  }
  float p[3];
  cell_centre(g, cell, p);
  const auto room = [&](int d, float c) {
    float m[3];
    plane_dir(d, m);
    const float l1 = fabsf(m[0]) + fabsf(m[1]) + fabsf(m[2]);
    return (c - (m[0] * p[0] + m[1] * p[1] + m[2] * p[2] + 0.5f * g.h * l1)) * rsqrtf(l1);
  };
  unsigned best = first ? kNoPlane : planes[cell];
  float best_room = (best & 31u) == kNoPlaneDir ? 0.f : room((int)(best & 31u), ordered_to_float((int)(best & ~31u)));
  for (int j = 0; j < ndir; ++j) {
    const int d = pass_dir(dir0, j);
    const int o = __ldg(mins + j * cells + cell);
    const float r = room(d, ordered_to_float(o));
    if (r > best_room) {
      best_room = r;
      best = ((unsigned)o & ~31u) | (unsigned)d;   // clearing low bits of an ordered int rounds the offset down
    }
  }
  planes[cell] = best;
}

// witness `slot` (0: .x, 1: .y) of every cell from the keys of its pass; a key left at ~0 (no triangle) gives -1
__global__ void take_witness_kernel(GridDev g, const unsigned long long *__restrict__ keys, int slot, int2 *witness) {
  const long long cell = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (cell >= cell_count(g)) return;
  const unsigned long long k = keys[cell];
  const int t = k == ~0ull ? -1 : (int)(unsigned)k;
  if (slot == 0) witness[cell] = make_int2(t, -1);
  else witness[cell].y = t;
}

#define CG_CUDA(expr)                 \
  do {                                \
    cudaError_t e_ = (expr);          \
    if (e_ != cudaSuccess) return e_; \
  } while (0)

// on unless the variable is set to a value that starts with '0'
bool switch_on(const char *name) {
  const char *v = std::getenv(name);
  return !(v && v[0] == '0');
}

// The grid's absolute slack, 1e-3 h + maxc * 3.9e-6, covers the float rounding of the vertices, of the cell lookup and of
// the distances for cells of edge h and coordinates within maxc of 0.  The clear bit's reach adds it to the bounding radius
// and the half cell diagonal.  The plane test must hold back every pose the reach does, so its pad carries it too, next to
// 2^-15 rho for the rotated robot: the argument is written next to plane_says_free (collide_kernels.cu).
struct Margins {
  float reach, plane_pad;
};
Margins clearance_margins(double rho, double h, double maxc) {
  const double slack = 1e-3 * h + maxc * 3.9e-6;
  return {(float)((rho + 0.8661 * h) * 1.002 + slack), round_up_f32((slack + rho * std::ldexp(1.0, -15)) * 1.001)};
}

}  // namespace

cudaError_t build_clearance_grid(const float4 *d_tris32, int64_t n_tris, const double root_lo[3], const double root_hi[3],
                                 double rho, cudaStream_t stream, ClearanceGrid *out) {
  if (n_tris <= 0 || !switch_on("SFFG_CLEARANCE_GRID")) return cudaSuccess;
  const bool witness = switch_on("SFFG_WITNESS");
  double h = rho / 4.0;
  double ext[3], maxc = 0;
  for (int k = 0; k < 3; ++k) {
    ext[k] = (root_hi[k] - root_lo[k]) + 2.0 * rho;
    maxc = std::max({maxc, std::fabs(root_lo[k]) + rho, std::fabs(root_hi[k]) + rho});
  }
  // cap the grid at 2^24 cells (2 MB of bits, L2-resident)
  while ((ext[0] / h + 1) * (ext[1] / h + 1) * (ext[2] / h + 1) > double(1 << 24)) h *= 1.25;
  ClearanceGrid g;
  GridDev &v = g.view;
  for (int k = 0; k < 3; ++k) {
    v.o[k] = (float)(root_lo[k] - rho);
    v.n[k] = std::max(1, (int)std::ceil(ext[k] / h));
  }
  v.h = (float)h;
  v.inv_h = (float)(1.0 / h);
  const Margins margins = clearance_margins(rho, h, maxc);
  v.plane_pad = margins.plane_pad;
  const size_t cells = (size_t)cell_count(v), words = (cells + 31) / 32;

  // One bit and one plane word per cell, and two contact witnesses (8 bytes) unless SFFG_WITNESS=0.  The build keeps the
  // per-direction plane bounds (one int per cell and direction) and then the witness keys (two ints per cell) in a
  // temporary block of at most 512 MB: one pass over the triangles for all 26 directions up to 5.1 M cells, more above.
  const size_t scratch_words = std::min<size_t>(26 * cells, std::max<size_t>(2 * cells, size_t(1) << 27));
  DevPtr<int> scratch;
  CG_CUDA(dev_alloc(g.bits, words * sizeof(unsigned)));
  CG_CUDA(cudaMemsetAsync(g.bits.get(), 0, words * sizeof(unsigned), stream));
  CG_CUDA(dev_alloc(g.planes, cells * sizeof(unsigned)));
  if (witness) CG_CUDA(dev_alloc(g.witness, cells * sizeof(int2)));
  CG_CUDA(dev_alloc(scratch, scratch_words * sizeof(int)));
  v.bits = g.bits.get();
  v.planes = g.planes.get();
  v.witness = g.witness.get();

  const int per_pass = (int)std::min<size_t>(26, scratch_words / cells);
  const long long blocks = ((long long)n_tris * 32 + kClearanceThreads - 1) / kClearanceThreads;
  const long long cell_blocks = ((long long)cells + 255) / 256;
  for (int dir0 = 0; dir0 < 26; dir0 += per_pass) {
    const int ndir = std::min(per_pass, 26 - dir0);
    CG_CUDA(cudaMemsetAsync(scratch.get(), 0x7f, (size_t)ndir * cells * sizeof(int), stream));
    build_clearance_kernel<<<(unsigned)blocks, kClearanceThreads, 0, stream>>>(d_tris32, (int)n_tris, v, margins.reach,
                                                                                dir0 == 0 ? g.bits.get() : nullptr, scratch.get(),
                                                                                dir0, ndir, nullptr, nullptr);
    choose_planes_kernel<<<(unsigned)cell_blocks, 256, 0, stream>>>(v, scratch.get(), dir0, ndir, dir0 == 0, g.planes.get());
    CG_CUDA(cudaGetLastError());
  }
  // contact witnesses: pass 0 takes each cell's nearest triangle, pass 1 the nearest of the others
  unsigned long long *keys = reinterpret_cast<unsigned long long *>(scratch.get());   // (cudaMalloc'd: 8-byte aligned)
  for (int slot = 0; witness && slot < 2; ++slot) {
    CG_CUDA(cudaMemsetAsync(keys, 0xff, cells * sizeof(unsigned long long), stream));
    build_clearance_kernel<<<(unsigned)blocks, kClearanceThreads, 0, stream>>>(d_tris32, (int)n_tris, v, margins.reach, nullptr,
                                                                                nullptr, 0, 0, keys, slot ? g.witness.get() : nullptr);
    take_witness_kernel<<<(unsigned)cell_blocks, 256, 0, stream>>>(v, keys, slot, g.witness.get());
    CG_CUDA(cudaGetLastError());
  }
  CG_CUDA(cudaStreamSynchronize(stream));

  g.bytes = words * sizeof(unsigned) + cells * sizeof(unsigned) + (witness ? cells * sizeof(int2) : 0);
  g.cells = (int64_t)cells;
  g.h = h;
  *out = std::move(g);
  return cudaSuccess;
}

}  // namespace sffg
