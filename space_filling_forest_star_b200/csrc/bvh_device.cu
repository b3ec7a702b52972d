// bvh_device.cu -- on-device construction of the obstacle hierarchy (SURVEY.md 8f row 4), sm_100a.
//
// The host builder (bvh_build.cpp, binned SAH) is the default for planner-sized maps; for large or changing obstacle sets
// (moving obstacles re-uploaded every frame) the same 8-wide AABB hierarchy is built on the GPU in a few milliseconds:
//
//   1. tri_prepare_kernel   per triangle: AABB in double -> outward-rounded floats, scene bounds by warp-reduced atomics
//   2. morton_kernel        63-bit Morton key (21 bits per axis) of the box centre, cub radix sort of (key, triangle)
//   3. split_level_kernel   top-down, one launch per level, one thread per open range of the sorted order: a range is cut at
//                           the first 3-bit Morton digit in which its keys differ (2..8 parts, an octree step with path
//                           compression); while fewer than 8 parts exist the largest one is cut further, so nodes are as
//                           full as the geometry allows.  Ranges of one triangle become leaf slots, the others are queued
//                           for the next level; node ids are contiguous per level.
//   4. fit_level_kernel     bottom-up, one launch per level, 8 lanes per node: a leaf slot takes its triangle's box, an inner
//                           slot the union of the child's 8 slot boxes; every operation rounds outward
//   5. gather_tris_kernel   FP64 and FP32 (+ representation error bound) triangle arrays in leaf (= Morton) order
//
// Any conservative hierarchy gives the same verdicts (SURVEY A.5), and every box here is rounded outward from the double
// vertices, so parity with the oracle does not depend on which builder ran (tests/test_gpu_bvh_device.py).
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <vector>

#include "bvh_device.cuh"

namespace sffg {
namespace {

// tbox: 6 floats per triangle (lo.xyz rounded down, hi.xyz rounded up); bounds: 3 x min, 3 x max as ordered ints
__global__ void tri_prepare_kernel(const double *__restrict__ soup, int n, float *__restrict__ tbox, int *bounds) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
  if (t < n) {
    const double *p = soup + 9 * (size_t)t;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double a = p[k], b = p[3 + k], c = p[6 + k];
      lo[k] = __double2float_rd(fmin(a, fmin(b, c)));
      hi[k] = __double2float_ru(fmax(a, fmax(b, c)));
      tbox[6 * (size_t)t + k] = lo[k];
      tbox[6 * (size_t)t + 3 + k] = hi[k];
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    int l = float_to_ordered(lo[k]), h = float_to_ordered(hi[k]);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
      l = min(l, __shfl_xor_sync(0xffffffffu, l, s));
      h = max(h, __shfl_xor_sync(0xffffffffu, h, s));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(bounds + k, l);
      atomicMax(bounds + 3 + k, h);
    }
  }
}

__device__ __forceinline__ unsigned long long spread21(unsigned v) {   // 21 bits -> every third bit of 63
  unsigned long long x = v & 0x1fffffull;
  x = (x | x << 32) & 0x1f00000000ffffull;
  x = (x | x << 16) & 0x1f0000ff0000ffull;
  x = (x | x << 8) & 0x100f00f00f00f00full;
  x = (x | x << 4) & 0x10c30c30c30c30c3ull;
  x = (x | x << 2) & 0x1249249249249249ull;
  return x;
}

__global__ void morton_kernel(const float *__restrict__ tbox, int n, const int *__restrict__ bounds, unsigned long long *keys,
                              int *vals) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  unsigned q[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float lo = ordered_to_float(bounds[k]), hi = ordered_to_float(bounds[3 + k]);
    const float c = 0.5f * tbox[6 * (size_t)t + k] + 0.5f * tbox[6 * (size_t)t + 3 + k];
    const float ext = hi - lo;
    float u = ext > 0.f ? (c - lo) / ext : 0.f;
    u = fminf(fmaxf(u, 0.f), 0.99999994f);
    q[k] = (unsigned)(u * 2097152.f);
  }
  keys[t] = spread21(q[0]) | spread21(q[1]) << 1 | spread21(q[2]) << 2;
  vals[t] = t;
}

struct Range {
  int first, count;
};

// cuts [first, first+count) at the most significant 3-bit digit in which its (sorted) keys differ; returns the number of parts
__device__ int split_range(const unsigned long long *__restrict__ keys, Range r, Range *parts) {
  const unsigned long long lo = keys[r.first], hi = keys[r.first + r.count - 1];
  if (lo == hi) {   // identical keys: cut by position
    const int np = min(8, r.count);
    int at = r.first;
    for (int i = 0; i < np; ++i) {
      const int c = r.count / np + (i < r.count % np ? 1 : 0);
      parts[i] = {at, c};
      at += c;
    }
    return np;
  }
  const int p = 63 - __clzll((long long)(lo ^ hi));   // highest differing bit
  const int shift = (p / 3) * 3;
  int np = 0, at = r.first;
  const int end = r.first + r.count;
  while (at < end) {
    const unsigned digit = (unsigned)(keys[at] >> shift) & 7u;
    // first position in [at, end) whose digit is larger (digits are non-decreasing inside the range)
    int a = at + 1, b = end;
    while (a < b) {
      const int m = (a + b) >> 1;
      if (((unsigned)(keys[m] >> shift) & 7u) > digit) b = m;
      else a = m + 1;
    }
    parts[np++] = {at, a - at};
    at = a;
  }
  return np;
}

// child word of a slot while the tree is being laid out: >= 0 inner node id, < 0 ~leaf position, kEmptyChild unused
__global__ void split_level_kernel(const unsigned long long *__restrict__ keys, const Range *__restrict__ cur, int n_cur, int node_base,
                                   int next_base, Range *next, int *next_count, ChildSlot *slots) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_cur) return;
  Range list[8], parts[8];
  bool fixed[8];
  int len = split_range(keys, cur[t], list);
  for (int i = 0; i < 8; ++i) fixed[i] = false;
  while (len < 8) {
    int pick = -1, best = 1;
    for (int i = 0; i < len; ++i)
      if (!fixed[i] && list[i].count > best) {
        best = list[i].count;
        pick = i;
      }
    if (pick < 0) break;
    const int np = split_range(keys, list[pick], parts);
    if (len - 1 + np > 8) {
      fixed[pick] = true;
      continue;
    }
    list[pick] = parts[0];
    for (int i = 1; i < np; ++i) {
      list[len] = parts[i];
      fixed[len] = false;
      ++len;
    }
  }
  // keep spatially adjacent children adjacent: order by first position (insertion sort, <= 8 entries)
  for (int i = 1; i < len; ++i) {
    const Range x = list[i];
    int j = i - 1;
    while (j >= 0 && list[j].first > x.first) {
      list[j + 1] = list[j];
      --j;
    }
    list[j + 1] = x;
  }
  ChildSlot *node = slots + (size_t)(node_base + t) * kWide;
  for (int i = 0; i < kWide; ++i) {
    ChildSlot s;
    s.cx = s.cy = s.cz = 3.0e38f;
    s.hx = s.hy = s.hz = -1.0f;
    s.pad = 0.f;
    s.child = kEmptyChild;
    if (i < len) {
      if (list[i].count == 1) {
        s.child = ~list[i].first;
      } else {
        const int pos = atomicAdd(next_count, 1);
        next[pos] = list[i];
        s.child = next_base + pos;
      }
    }
    node[i] = s;
  }
}

// 8 lanes per node; boxes of deeper levels are final when a level runs
__global__ void fit_level_kernel(ChildSlot *slots, int node_base, int n_nodes, const float *__restrict__ tbox,
                                 const int *__restrict__ order) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  const int node = g >> 3, i = g & 7;
  if (node >= n_nodes) return;
  ChildSlot *s = slots + (size_t)(node_base + node) * kWide + i;
  const int child = s->child;
  if (child == kEmptyChild) return;
  float lo[3], hi[3];
  if (child < 0) {
    const float *b = tbox + 6 * (size_t)order[~child];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      lo[k] = b[k];
      hi[k] = b[3 + k];
    }
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      lo[k] = 3.0e38f;
      hi[k] = -3.0e38f;
    }
    const ChildSlot *c = slots + (size_t)child * kWide;
    for (int j = 0; j < kWide; ++j) {
      if (c[j].child == kEmptyChild) continue;
      const float cc[3] = {c[j].cx, c[j].cy, c[j].cz}, ch[3] = {c[j].hx, c[j].hy, c[j].hz};
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        lo[k] = fminf(lo[k], __fsub_rd(cc[k], ch[k]));
        hi[k] = fmaxf(hi[k], __fadd_ru(cc[k], ch[k]));
      }
    }
  }
  float c3[3], h3[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    c3[k] = 0.5f * lo[k] + 0.5f * hi[k];
    h3[k] = fmaxf(__fsub_ru(hi[k], c3[k]), __fsub_ru(c3[k], lo[k]));
  }
  s->cx = c3[0];
  s->cy = c3[1];
  s->cz = c3[2];
  s->hx = h3[0];
  s->hy = h3[1];
  s->hz = h3[2];
}

__global__ void gather_tris_kernel(const double *__restrict__ soup, const int *__restrict__ order, int n, double *__restrict__ t64,
                                   float4 *__restrict__ t32) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double *src = soup + 9 * (size_t)order[i];
  double v[9];
  double err = 0.0;
  float f[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    v[k] = src[k];
    t64[9 * (size_t)i + k] = v[k];
    f[k] = __double2float_rn(v[k]);
    err = fmax(err, fabs(v[k] - (double)f[k]));
  }
  t32[3 * (size_t)i + 0] = make_float4(f[0], f[1], f[2], __double2float_ru(err * 1.0000001));
  t32[3 * (size_t)i + 1] = make_float4(f[3], f[4], f[5], 0.f);
  t32[3 * (size_t)i + 2] = make_float4(f[6], f[7], f[8], 0.f);
}

__global__ void init_bounds_kernel(int *bounds) {
  if (threadIdx.x < 3) bounds[threadIdx.x] = 0x7fffffff;
  else if (threadIdx.x < 6) bounds[threadIdx.x] = (int)0x80000000;
}

struct Scratch {
  std::vector<void *> ptrs;
  ~Scratch() {
    for (void *p : ptrs) cudaFree(p);
  }
  template <class T>
  cudaError_t get(T **p, size_t count) {
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, std::max<size_t>(count * sizeof(T), 16));
    if (e == cudaSuccess) ptrs.push_back(q);
    *p = (T *)q;
    return e;
  }
};

#define BD_CUDA(expr)                 \
  do {                                \
    cudaError_t e_ = (expr);          \
    if (e_ != cudaSuccess) return e_; \
  } while (0)

// waits for the stream and reads the scene bounds tri_prepare_kernel left in `bounds` as the root box
cudaError_t read_root_bounds(const int *bounds, cudaStream_t st, double root_lo[3], double root_hi[3]) {
  int hb[6];
  BD_CUDA(cudaMemcpyAsync(hb, bounds, sizeof hb, cudaMemcpyDeviceToHost, st));
  BD_CUDA(cudaStreamSynchronize(st));
  BD_CUDA(cudaGetLastError());
  for (int k = 0; k < 3; ++k) {
    root_lo[k] = ordered_to_float(hb[k]);
    root_hi[k] = ordered_to_float(hb[3 + k]);
  }
  return cudaSuccess;
}

}  // namespace

cudaError_t build_bvh_device(const double *d_soup, int n, cudaStream_t st, DeviceBvh *out) {
  *out = DeviceBvh{};
  if (n <= 0) return cudaSuccess;
  Scratch tmp;
  float *tbox;
  int *bounds, *vals_in, *vals_out, *next_count;
  unsigned long long *keys_in, *keys_out;
  Range *q[2];
  ChildSlot *slots_big;
  BD_CUDA(tmp.get(&tbox, 6 * (size_t)n));
  BD_CUDA(tmp.get(&bounds, 8));
  BD_CUDA(tmp.get(&keys_in, (size_t)n));
  BD_CUDA(tmp.get(&keys_out, (size_t)n));
  BD_CUDA(tmp.get(&vals_in, (size_t)n));
  BD_CUDA(tmp.get(&next_count, 4));
  BD_CUDA(tmp.get(&q[0], (size_t)n));
  BD_CUDA(tmp.get(&q[1], (size_t)n));
  // every inner node has >= 2 children, so there are at most n - 1 of them (a single triangle still gets a root)
  const size_t max_nodes = (size_t)std::max(n - 1, 1);
  BD_CUDA(tmp.get(&slots_big, max_nodes * kWide));
  BD_CUDA(cudaMalloc((void **)&vals_out, (size_t)n * sizeof(int)));   // becomes out->d_order
  auto fail_free = [&](cudaError_t e) {
    cudaFree(vals_out);
    return e;
  };
  const int T = 256, G = (n + T - 1) / T;
  init_bounds_kernel<<<1, 32, 0, st>>>(bounds);
  tri_prepare_kernel<<<G, T, 0, st>>>(d_soup, n, tbox, bounds);
  morton_kernel<<<G, T, 0, st>>>(tbox, n, bounds, keys_in, vals_in);
  size_t sort_bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, keys_in, keys_out, vals_in, vals_out, n, 0, 63, st);
  if (e != cudaSuccess) return fail_free(e);
  unsigned char *sort_tmp;
  if ((e = tmp.get(&sort_tmp, sort_bytes)) != cudaSuccess) return fail_free(e);
  e = cub::DeviceRadixSort::SortPairs(sort_tmp, sort_bytes, keys_in, keys_out, vals_in, vals_out, n, 0, 63, st);
  if (e != cudaSuccess) return fail_free(e);

  // ---- top-down layout, level by level
  std::vector<int> level_base, level_count;
  int cur = 0, n_cur = 1, node_base = 0;
  if (n == 1) {
    // a single triangle: the root holds one leaf slot
    std::vector<ChildSlot> root(kWide);
    for (int i = 0; i < kWide; ++i) {
      root[i].cx = root[i].cy = root[i].cz = 3.0e38f;
      root[i].hx = root[i].hy = root[i].hz = -1.0f;
      root[i].pad = 0.f;
      root[i].child = i == 0 ? ~0 : kEmptyChild;
    }
    if ((e = cudaMemcpyAsync(slots_big, root.data(), kWide * sizeof(ChildSlot), cudaMemcpyHostToDevice, st)) != cudaSuccess) return fail_free(e);
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return fail_free(e);
    level_base.push_back(0);
    level_count.push_back(1);
    node_base = 1;
  } else {
    const Range whole{0, n};
    if ((e = cudaMemcpyAsync(q[0], &whole, sizeof whole, cudaMemcpyHostToDevice, st)) != cudaSuccess) return fail_free(e);
    while (n_cur > 0) {
      if ((e = cudaMemsetAsync(next_count, 0, sizeof(int), st)) != cudaSuccess) return fail_free(e);
      const int next_base = node_base + n_cur;
      split_level_kernel<<<(n_cur + 127) / 128, 128, 0, st>>>(keys_out, q[cur], n_cur, node_base, next_base, q[cur ^ 1], next_count,
                                                             slots_big);
      level_base.push_back(node_base);
      level_count.push_back(n_cur);
      int n_next = 0;
      if ((e = cudaMemcpyAsync(&n_next, next_count, sizeof(int), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return fail_free(e);
      if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return fail_free(e);
      node_base = next_base;
      n_cur = n_next;
      cur ^= 1;
      if (level_base.size() > 96) return fail_free(cudaErrorUnknown);   // 21 digits + position cuts: cannot happen
    }
  }
  const int n_nodes = node_base;
  // ---- bottom-up boxes
  for (int l = (int)level_base.size() - 1; l >= 0; --l) {
    const int threads = level_count[l] * 8;
    fit_level_kernel<<<(threads + 255) / 256, 256, 0, st>>>(slots_big, level_base[l], level_count[l], tbox, vals_out);
  }
  // ---- outputs
  ChildSlot *slots;
  double *t64;
  float4 *t32;
  if ((e = cudaMalloc((void **)&slots, (size_t)n_nodes * kWide * sizeof(ChildSlot))) != cudaSuccess) return fail_free(e);
  if ((e = cudaMalloc((void **)&t64, 9 * (size_t)n * sizeof(double))) != cudaSuccess) {
    cudaFree(slots);
    return fail_free(e);
  }
  if ((e = cudaMalloc((void **)&t32, 3 * (size_t)n * sizeof(float4))) != cudaSuccess) {
    cudaFree(slots);
    cudaFree(t64);
    return fail_free(e);
  }
  cudaMemcpyAsync(slots, slots_big, (size_t)n_nodes * kWide * sizeof(ChildSlot), cudaMemcpyDeviceToDevice, st);
  gather_tris_kernel<<<G, T, 0, st>>>(d_soup, vals_out, n, t64, t32);
  if ((e = read_root_bounds(bounds, st, out->root_lo, out->root_hi)) != cudaSuccess) {
    cudaFree(slots);
    cudaFree(t64);
    cudaFree(t32);
    return fail_free(e);
  }
  out->d_slots = slots;
  out->d_tris64 = t64;
  out->d_tris32 = t32;
  out->d_order = vals_out;
  out->n_nodes = n_nodes;
  out->depth = (int)level_base.size();
  out->level_base = level_base;
  out->level_count = level_count;
  return cudaSuccess;
}

cudaError_t refit_bvh_device(const double *d_soup, int n, ChildSlot *d_slots, double *d_tris64, float4 *d_tris32, const int *d_order,
                             const std::vector<int> &level_base, const std::vector<int> &level_count, cudaStream_t st,
                             double root_lo[3], double root_hi[3]) {
  if (n <= 0) return cudaSuccess;
  Scratch tmp;
  float *tbox;
  int *bounds;
  BD_CUDA(tmp.get(&tbox, 6 * (size_t)n));
  BD_CUDA(tmp.get(&bounds, 8));
  const int T = 256, G = (n + T - 1) / T;
  init_bounds_kernel<<<1, 32, 0, st>>>(bounds);
  tri_prepare_kernel<<<G, T, 0, st>>>(d_soup, n, tbox, bounds);
  gather_tris_kernel<<<G, T, 0, st>>>(d_soup, d_order, n, d_tris64, d_tris32);
  for (int l = (int)level_base.size() - 1; l >= 0; --l) {
    const int threads = level_count[l] * 8;
    fit_level_kernel<<<(threads + 255) / 256, 256, 0, st>>>(d_slots, level_base[l], level_count[l], tbox, d_order);
  }
  return read_root_bounds(bounds, st, root_lo, root_hi);
}

}  // namespace sffg
