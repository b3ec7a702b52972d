// sffg_api.cu -- the C ABI of libsffg.so (declared in include/sffg.h).  Host-side glue only: handle lifetime,
// HBM layout, chunked H2D / kernel / D2H pipelining on two streams.  No compute happens on the CPU and there is no
// fallback: without a usable sm_100 device every compute entry point returns SFFG_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <vector>

#include "bvh_device.cuh"
#include "clearance_grid.cuh"
#include "collide_kernels.cuh"
#include "common.h"
#include "cuda_handles.h"
#include "knn_kernels.cuh"
#include "knn_pruned.cuh"

namespace sffg {

static thread_local std::string g_error;
void set_error(const std::string &msg) { g_error = msg; }
int fail(int code, const std::string &msg) {
  g_error = msg;
  return code;
}

namespace {

constexpr size_t kSmallBytes = 1 << 20;   // pinned, device-mapped staging area of each object for planner-sized calls

// The environment's staging area: inputs in the first 3/4, outputs in the last 1/4.  The outputs of a pose call are its
// verdicts; those of a distance call are the distances [n] then (if asked for) the points [n][6]; those of an edge call
// are first hits [m] then free flags [m]; those of a move call are free flags [m] then pose hits [m]; those of an edge
// distance call are the distances [m], the points [m][6], then the sample indices [m]; those of a sweep call are the
// stop parameters [m], the distances [m], then the clear flags [m].
struct EnvStaging {
  static constexpr size_t kInBytes = 768 << 10;
  static constexpr size_t kOutBytes = kSmallBytes - kInBytes;
  unsigned char *base;
  unsigned char *in() const { return base; }
  uint8_t *out() const { return base + kInBytes; }
  int32_t *edge_first_hit() const { return reinterpret_cast<int32_t *>(out()); }
  uint8_t *edge_free(int64_t m) const { return out() + (size_t)m * 4; }
  uint8_t *move_free() const { return out(); }
  uint8_t *move_hit(int64_t m) const { return out() + (size_t)m; }
  double *edge_dist() const { return reinterpret_cast<double *>(out()); }
  double *edge_points(int64_t m) const { return reinterpret_cast<double *>(out() + (size_t)m * 8); }
  int32_t *edge_index(int64_t m) const { return reinterpret_cast<int32_t *>(out() + (size_t)m * 56); }
  double *sweep_t() const { return reinterpret_cast<double *>(out()); }
  double *sweep_dist(int64_t m) const { return reinterpret_cast<double *>(out() + (size_t)m * 8); }
  uint8_t *sweep_clear(int64_t m) const { return out() + (size_t)m * 16; }
};

// The index's staging area.  The first 64 KiB hold the queries; the one-kernel radius search keeps its fallback flag in
// their last 16 bytes.  After them:
//   k-NN:    ids [nq * k], then d2 [nq * k]
//   radius:  counts [nq] (64 KiB), then from 128 KiB the rows part: a head, ids [cap], d2 [cap].  The head is the row
//            offsets [nq] (one-kernel form) or the total (one-sync form); the two-sync form has no head and stages the
//            row offsets in the query part instead.
// sffg_index_add_multi_begin uses the whole area for the rows to append.
struct IndexStaging {
  static constexpr size_t kQueryBytes = 64 << 10;
  static constexpr size_t kCountBytes = 64 << 10;
  static constexpr size_t kRowsAt = 128 << 10;
  static constexpr size_t kRowsBytes = kSmallBytes - kRowsAt;
  static constexpr size_t kKnnOutBytes = kSmallBytes - kQueryBytes;
  static constexpr size_t kFlagAt = kQueryBytes - 16;
  // entries of ids and of d2 that fit behind a head of `head_bytes`
  static int64_t rows_cap(size_t head_bytes) { return (int64_t)((kRowsBytes - head_bytes) / 8); }
  unsigned char *base;
  unsigned char *queries() const { return base; }
  int *fused_flag() const { return reinterpret_cast<int *>(base + kFlagAt); }
  int32_t *knn_ids() const { return reinterpret_cast<int32_t *>(base + kQueryBytes); }
  float *knn_d2(size_t obytes) const { return reinterpret_cast<float *>(base + kQueryBytes + obytes); }
  int32_t *counts() const { return reinterpret_cast<int32_t *>(base + kQueryBytes); }
  int64_t *rows_head() const { return reinterpret_cast<int64_t *>(base + kRowsAt); }
  int32_t *rows_ids(size_t head_bytes) const { return reinterpret_cast<int32_t *>(base + kRowsAt + head_bytes); }
  float *rows_d2(size_t head_bytes, int64_t cap) const {
    return reinterpret_cast<float *>(base + kRowsAt + head_bytes + (size_t)cap * 4);
  }
};

// enqueues an upload of host data on `st`, through `staging` (pinned) unless it is null
cudaError_t upload_async(void *dst, const void *src, size_t bytes, unsigned char *staging, cudaStream_t st) {
  if (staging) src = std::memcpy(staging, src, bytes);
  return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
}

// a device copy of `n` bytes of host data (at least 16 bytes allocated); adds `n` to *counted
template <class T> cudaError_t upload(DevPtr<T> &dst, const void *src, size_t n, size_t *counted) {
  cudaError_t e = dev_alloc(dst, std::max<size_t>(n, 16));
  if (e != cudaSuccess) return e;
  *counted += n;
  return n ? cudaMemcpy(dst.get(), src, n, cudaMemcpyHostToDevice) : cudaSuccess;
}

struct Runtime {
  bool ready = false;
  int device = -1;
  int sm_count = 0;
  int smem_optin = 0;   // largest dynamic shared memory a CTA may ask for
};
Runtime g_rt;

#define SFFG_CUDA(expr)                                                                          \
  do {                                                                                           \
    cudaError_t e_ = (expr);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return fail(SFFG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));            \
  } while (0)

int ensure_runtime() {
  if (g_rt.ready) return SFFG_OK;
  return sffg_init(-1);
}

// grow-only device buffer
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { release(); }
  int reserve(size_t bytes) {
    if (bytes <= cap) return SFFG_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    SFFG_CUDA(cudaMalloc(&p, want));
    cap = want;
    return SFFG_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

}  // namespace
}  // namespace sffg

using namespace sffg;

// ---------------------------------------------------------------------------------------------------------------
struct sffg_env {
  EnvDev dev{};
  DevPtr<ChildSlot> d_slots, d_top;
  ClearanceGrid grid;
  DevPtr<float4> d_rob_verts;
  DevPtr<float4> d_tris32;
  DevPtr<double> d_tris64, d_robot64;
  DevPtr<RobotTri> d_robot;
  DevPtr<int> d_order;                           // leaf position -> caller's triangle index (refit)
  std::vector<int> level_base, level_count;      // breadth-first level table of the hierarchy (refit)
  int64_t obst_bytes = 0;
  double obst_max_abs = 0;                       // max |obstacle coordinate| (root box), 0 without obstacles
  DevPtr<unsigned long long> d_counters;
  PinnedPtr<int> h_status;      // the kernels raise it, the host reads it without a copy
  DevPtr<unsigned> d_work;      // ring of 8 work counters (never reset; see launch_collide_poses)
  unsigned work_base[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int work_next = 0;
  PinnedPtr<unsigned char> h_small;   // staging for small calls (planner-sized batches), see EnvStaging
  EnvStaging staging() const { return {h_small.get()}; }
  Stream streams[2];
  // launches of one environment share state (the ring of work counters, the first-hit scratch `fh`), so they are kept in
  // order across whatever streams the caller uses: every *_device launch records order_ev, and a launch on another
  // stream (or an internal stream of the host-pointer calls) first waits for it
  Event order_ev;
  cudaStream_t last_stream = nullptr;
  bool order_pending = false;
  DevBuf in[2], out[2], aux[2], fh;   // fh: per-edge first-hit scratch of small edge batches
  DevBuf edge_scr, edge_rec;          // edge distance calls: the verdict launch's results, the per-warp records
  bool count = false;
  int64_t robot_bytes = 0;
  sffg_env_info_t info{};
  LaunchCfg cfg{};
  // asynchronous form (sffg_check_edges_begin / sffg_check_moves_begin + sffg_env_end): what the end still has to do
  struct Pending {
    int kind = 0;   // 0 none, 1 edges, 2 moves
    int64_t m = 0;
    uint8_t *out = nullptr;
    int32_t *first_out = nullptr;
  } pend;
};
static int env_busy(const sffg_env *env, const char *who) {
  if (env->pend.kind != 0) return fail(SFFG_ERR_ARG, std::string(who) + ": an asynchronous call on this environment is pending (sffg_env_end first)");
  return SFFG_OK;
}

struct sffg_index {
  int dim = 0;
  DevPtr<float> d_coords;
  DevPtr<unsigned> d_amax;   // float bits of the largest |angle| stored (dim 6): selects the kernels' exact wide wrap
  int64_t cap = 0, n = 0;
  Stream stream;
  Event ev;   // fork / join of multi-index calls
  DevBuf q, ids, d2, scratch, counts, offsets, cursor, keys, stage;
  PinnedPtr<unsigned char> h_small;   // staging for planner-sized queries, see IndexStaging
  IndexStaging staging() const { return {h_small.get()}; }
  // spatially sorted view (knn_pruned.cu): covers nodes [0, n_sorted); rebuilt when the unsorted tail grows too long
  DevBuf s_coords, s_ids, s_bb, s_keys, s_vals, s_temp, s_bounds;
  int64_t n_sorted = 0, s_cap = 0, s_nblk_cap = 0;
  bool pruning = true;
  // asynchronous form (sffg_*_begin / sffg_index_end): what the matching end still has to do.  One pending call per index.
  struct HostCopy { void *dst; const void *src; size_t bytes; };
  struct Pending {
    int kind = 0;   // 0 none, 1 knn_multi, 2 radius, 3 add_multi
    HostCopy copy[3];
    int n_copy = 0;
    // radius
    int64_t nq = 0, capacity = 0, cap1 = 0;
    float r2 = 0;
    int32_t *counts_out = nullptr, *ids_out = nullptr;
    float *d2_out = nullptr;
    int64_t *total_out = nullptr;
    bool small = false, one_sync = false, pruned = false, fused = false;
    const float *queries = nullptr;
  } pend;
  Event add_ev;   // appends enqueued by sffg_index_add_multi_begin have run
  DevPtr<unsigned long long> d_total;   // row allocator of the one-kernel radius search
};
static int index_busy(const sffg_index *idx, const char *who) {
  if (idx->pend.kind != 0) return fail(SFFG_ERR_ARG, std::string(who) + ": an asynchronous call on this index is pending (sffg_index_end first)");
  return SFFG_OK;
}

extern "C" {

int sffg_version(void) { return 100; }
const char *sffg_last_error(void) { return g_error.c_str(); }

int sffg_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int sffg_init(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(SFFG_ERR_NO_DEVICE, "no CUDA device visible: the sffg engine has no CPU path and refuses to run");
  }
  if (device < 0) {
    if (cudaGetDevice(&device) != cudaSuccess) device = 0;
  }
  if (device >= n) return fail(SFFG_ERR_ARG, "device ordinal out of range");
  SFFG_CUDA(cudaSetDevice(device));
  // (attributes, not cudaGetDeviceProperties: the full property query costs tens of milliseconds of every process start)
  int major = 0, minor = 0, sms = 0, optin = 0;
  SFFG_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  SFFG_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
  SFFG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  SFFG_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  if (major != 10)
    return fail(SFFG_ERR_NO_DEVICE, "device " + std::to_string(device) + " is sm_" + std::to_string(major) + std::to_string(minor) +
                                        "; libsffg.so carries sm_100a code only");
  g_rt.device = device;
  g_rt.sm_count = sms;
  g_rt.smem_optin = optin;
  g_rt.ready = true;
  return SFFG_OK;
}

// ---- meshes -----------------------------------------------------------------------------------------------
int sffg_mesh_load(const char *path, int is_obj, const double position[3], double scale, double **tris_out,
                   int64_t *n_tris_out, double bbox_out[6]) {
  if (!path || !tris_out || !n_tris_out) return fail(SFFG_ERR_ARG, "sffg_mesh_load: null argument");
  const double zero[3] = {0, 0, 0};
  std::vector<double> tris;
  double bbox[6];
  int rc = load_mesh(path, is_obj, position ? position : zero, scale, &tris, bbox);
  if (rc != SFFG_OK) return rc;
  double *out = (double *)std::malloc(std::max<size_t>(tris.size(), 1) * sizeof(double));
  if (!out) return fail(SFFG_ERR_ARG, "out of host memory");
  std::memcpy(out, tris.data(), tris.size() * sizeof(double));
  *tris_out = out;
  *n_tris_out = (int64_t)(tris.size() / 9);
  if (bbox_out) std::memcpy(bbox_out, bbox, sizeof bbox);
  return SFFG_OK;
}
void sffg_free(void *p) { std::free(p); }

// ---- environment ------------------------------------------------------------------------------------------
static void cross3(const double *a, const double *b, double *r) {
  r[0] = a[1] * b[2] - a[2] * b[1];
  r[1] = a[2] * b[0] - a[0] * b[2];
  r[2] = a[0] * b[1] - a[1] * b[0];
}

static void make_robot_tri(const double *t, RobotTri *o) {
  const double *q[3] = {t, t + 3, t + 6};
  double f[3][3], m[3], h[3][3];
  for (int k = 0; k < 3; ++k) {
    f[0][k] = q[1][k] - q[0][k];
    f[1][k] = q[2][k] - q[1][k];
    f[2][k] = q[0][k] - q[2][k];
  }
  cross3(f[0], f[1], m);
  for (int j = 0; j < 3; ++j) cross3(f[j], m, h[j]);
  double qmax = 0;
  for (int v = 0; v < 3; ++v)
    for (int k = 0; k < 3; ++k) {
      o->q[v][k] = (float)q[v][k];
      o->f[v][k] = (float)f[v][k];
      o->h[v][k] = (float)h[v][k];
      qmax = std::max(qmax, std::fabs(q[v][k]));
    }
  for (int k = 0; k < 3; ++k) o->m[k] = (float)m[k];
  // projection intervals of the TRUE triangle on the float axes, widened and rounded outward
  auto interval = [&](const float *axis, float *lo, float *hi) {
    double mn = std::numeric_limits<double>::max(), mx = -mn, mag = 0;
    for (int v = 0; v < 3; ++v) {
      double p = (double)axis[0] * q[v][0] + (double)axis[1] * q[v][1] + (double)axis[2] * q[v][2];
      mag = std::max(mag, std::fabs((double)axis[0] * q[v][0]) + std::fabs((double)axis[1] * q[v][1]) +
                              std::fabs((double)axis[2] * q[v][2]));
      mn = std::min(mn, p);
      mx = std::max(mx, p);
    }
    const double slack = mag * 1e-14;
    *lo = round_down_f32(mn - slack);
    *hi = round_up_f32(mx + slack);
  };
  interval(o->m, &o->m_lo, &o->m_hi);
  for (int j = 0; j < 3; ++j) interval(o->h[j], &o->h_lo[j], &o->h_hi[j]);
  for (int k = 0; k < 3; ++k) {
    o->lo[k] = round_down_f32(std::min({q[0][k], q[1][k], q[2][k]}));
    o->hi[k] = round_up_f32(std::max({q[0][k], q[1][k], q[2][k]}));
  }
  o->qmax = round_up_f32(qmax);
  o->pad[0] = o->pad[1] = o->pad[2] = 0.f;
}

int sffg_env_destroy(sffg_env *env) {
  if (!env) return SFFG_OK;
  for (const Stream &s : env->streams)
    if (s) cudaStreamSynchronize(s.get());
  delete env;
  return SFFG_OK;
}

// (re)builds everything that depends on the obstacle soup: hierarchy, triangle arrays, root box, clearance grid.
// The robot side of `env` must already be in place (the grid is dilated by the robot's bounding radius).
constexpr int64_t kDeviceBuildMin = 1 << 18;   // SFFG_BUILD_AUTO: triangle count from which the hierarchy is built on the GPU

// everything that hangs off a finished hierarchy: top cut, root box, clearance grid, device view, info
static int finish_obstacles(sffg_env *env, const std::vector<ChildSlot> &top, const double root_lo[3], const double root_hi[3],
                            int64_t n_obst, int64_t n_nodes, int depth, bool on_device, size_t bytes) {
  EnvDev &d = env->dev;
  env->d_top.reset();
  SFFG_CUDA(upload(env->d_top, top.data(), top.size() * sizeof(ChildSlot), &bytes));
  d.n_obst = (int)n_obst;
  env->obst_max_abs = 0;
  for (int k = 0; k < 3; ++k) {
    // rounded up to float: the device builder's root box is outward rounded to float, the host builder's is exact
    if (n_obst) env->obst_max_abs = std::max({env->obst_max_abs, (double)round_up_f32(std::fabs(root_lo[k])),
                                              (double)round_up_f32(std::fabs(root_hi[k]))});
    const double oc = 0.5 * (root_lo[k] + root_hi[k]);
    d.root_c[k] = (float)oc;
    d.root_h[k] = n_obst ? round_up_f32(std::max(root_hi[k] - (double)d.root_c[k], (double)d.root_c[k] - root_lo[k]) * 1.0000001) : 0.f;
  }
  // the old grid goes before the new one is built, so that a set or refit never holds two
  env->grid = ClearanceGrid();
  const cudaError_t grid_err = build_clearance_grid(env->d_tris32.get(), n_obst, root_lo, root_hi, d.rob_radius, env->streams[0].get(),
                                                    &env->grid);
  d.grid = env->grid.view;   // no grid unless the build succeeded
  env->info.grid_cells = env->grid.cells;
  env->info.grid_cell_size = env->grid.h;
  if (grid_err != cudaSuccess) return fail(SFFG_ERR_CUDA, std::string("clearance grid build: ") + cudaGetErrorString(grid_err));
  bytes += env->grid.bytes;
  d.slots = reinterpret_cast<const float4 *>(env->d_slots.get());
  d.top = reinterpret_cast<const float4 *>(env->d_top.get());
  d.n_top = (int)top.size();
  {
    // leading (breadth-first) nodes a CTA stages in shared memory: what fits next to the robot and the warp scratch
    const int64_t room = ((int64_t)g_rt.smem_optin - 1024 - (int64_t)collide_smem_bytes(d.n_robot, 0)) / (int64_t)(kWide * sizeof(ChildSlot));
    d.n_stage_max = (int)std::max<int64_t>(0, std::min<int64_t>({n_nodes, (int64_t)kStageNodesCap, room}));
  }
  d.tris32 = env->d_tris32.get();
  d.tris64 = env->d_tris64.get();
  env->info.n_obst_tris = n_obst;
  env->info.n_nodes = n_nodes;
  env->info.depth = depth;
  env->info.device_bytes = env->robot_bytes + (int64_t)bytes;
  env->info.built_on_device = on_device ? 1 : 0;
  return SFFG_OK;
}

// the caller's soup (9 doubles per triangle) in a temporary device block, copied on the environment's first stream
static cudaError_t upload_soup(sffg_env *env, DevPtr<double> &d_soup, const double *tris, int64_t n) {
  const size_t bytes = 9 * (size_t)n * sizeof(double);
  const cudaError_t e = dev_alloc(d_soup, bytes);
  return e == cudaSuccess ? cudaMemcpyAsync(d_soup.get(), tris, bytes, cudaMemcpyHostToDevice, env->streams[0].get()) : e;
}

// the cut through the top of the device-resident hierarchy, chosen on the host from its first levels (nodes are stored
// level by level)
static int read_top_cut(const sffg_env *env, int64_t n_nodes, std::vector<ChildSlot> *top) {
  HostBvh head;
  head.slots.resize((size_t)std::min<int64_t>(n_nodes, 1 + 8 + 64) * kWide);
  SFFG_CUDA(cudaMemcpy(head.slots.data(), env->d_slots.get(), head.slots.size() * sizeof(ChildSlot), cudaMemcpyDeviceToHost));
  top_cut(head, top);
  return SFFG_OK;
}

static int set_obstacles(sffg_env *env, const double *obst_tris, int64_t n_obst, int build_mode) {
  const bool on_device = n_obst > 0 && (build_mode == SFFG_BUILD_DEVICE || (build_mode == SFFG_BUILD_AUTO && n_obst >= kDeviceBuildMin));
  env->level_base.clear();
  env->level_count.clear();
  env->d_slots.reset();
  env->d_tris32.reset();
  env->d_tris64.reset();
  env->d_order.reset();
  size_t bytes = 0;
  double root_lo[3] = {0, 0, 0}, root_hi[3] = {0, 0, 0};
  std::vector<ChildSlot> top;
  int64_t n_nodes = 0;
  int depth = 0;
  if (!on_device) {
    // ---- host: binned-SAH hierarchy + FP32 / FP64 triangle arrays in leaf order
    HostBvh bvh;
    build_wide_bvh(obst_tris, n_obst, &bvh);
    std::vector<TriF32> t32((size_t)n_obst);
    std::vector<double> t64(9 * (size_t)n_obst);
    for (int64_t i = 0; i < n_obst; ++i) {
      const double *src = obst_tris + 9 * (size_t)bvh.tri_order[(size_t)i];
      std::memcpy(&t64[9 * (size_t)i], src, 9 * sizeof(double));
      double err = 0;
      for (int v = 0; v < 3; ++v) {
        for (int k = 0; k < 3; ++k) {
          float f = (float)src[3 * v + k];
          t32[(size_t)i].p[v][k] = f;
          err = std::max(err, std::fabs(src[3 * v + k] - (double)f));
        }
        t32[(size_t)i].p[v][3] = 0.f;
      }
      t32[(size_t)i].p[0][3] = round_up_f32(err * 1.0000001);
    }
    SFFG_CUDA(upload(env->d_slots, bvh.slots.data(), bvh.slots.size() * sizeof(ChildSlot), &bytes));
    SFFG_CUDA(upload(env->d_tris32, t32.data(), t32.size() * sizeof(TriF32), &bytes));
    SFFG_CUDA(upload(env->d_tris64, t64.data(), t64.size() * sizeof(double), &bytes));
    SFFG_CUDA(upload(env->d_order, bvh.tri_order.data(), bvh.tri_order.size() * sizeof(int32_t), &bytes));
    env->level_base = bvh.level_base;
    env->level_count = bvh.level_count;
    top_cut(bvh, &top);
    n_nodes = (int64_t)(bvh.slots.size() / kWide);
    depth = bvh.depth;
    for (int k = 0; k < 3; ++k) {
      root_lo[k] = bvh.root_lo[k];
      root_hi[k] = bvh.root_hi[k];
    }
  } else {
    // ---- device: Morton-ordered 8-wide hierarchy built by bvh_device.cu from the uploaded soup
    DevPtr<double> d_soup;
    cudaError_t e = upload_soup(env, d_soup, obst_tris, n_obst);
    DeviceBvh db;
    if (e == cudaSuccess) e = build_bvh_device(d_soup.get(), (int)n_obst, env->streams[0].get(), &db);
    d_soup.reset();
    env->d_slots.reset(db.d_slots);
    env->d_tris32.reset(db.d_tris32);
    env->d_tris64.reset(db.d_tris64);
    env->d_order.reset(db.d_order);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(SFFG_ERR_CUDA, std::string("device BVH build: ") + cudaGetErrorString(e));
    }
    env->level_base = db.level_base;
    env->level_count = db.level_count;
    bytes += (size_t)db.n_nodes * kWide * sizeof(ChildSlot) + (size_t)n_obst * (sizeof(TriF32) + 9 * sizeof(double));
    const int rc = read_top_cut(env, db.n_nodes, &top);
    if (rc != SFFG_OK) return rc;
    n_nodes = db.n_nodes;
    depth = db.depth;
    for (int k = 0; k < 3; ++k) {
      root_lo[k] = db.root_lo[k];
      root_hi[k] = db.root_hi[k];
    }
  }
  env->obst_bytes = (int64_t)bytes;
  return finish_obstacles(env, top, root_lo, root_hi, n_obst, n_nodes, depth, on_device, bytes);
}

int sffg_env_create_ex(const double *obst_tris, int64_t n_obst, const double *robot_tris, int64_t n_robot, int build_mode,
                       sffg_env **out) {
  if (!out || n_obst < 0 || n_robot <= 0 || !robot_tris || (n_obst > 0 && !obst_tris) || build_mode < 0 || build_mode > 2)
    return fail(SFFG_ERR_ARG, "sffg_env_create: bad arguments");
  if (n_obst > 0x3fffffff || n_robot > 4096) return fail(SFFG_ERR_ARG, "sffg_env_create: mesh too large");
  int rc = ensure_runtime();
  if (rc != SFFG_OK) return rc;
  // the kernels keep the whole robot in shared memory next to the per-warp scratch: refuse what cannot fit instead of
  // building an environment whose every call would fail to launch
  if (collide_smem_bytes((int)n_robot, 0) + 1024 > (size_t)g_rt.smem_optin) {
    const size_t room = (size_t)g_rt.smem_optin - 1024 - collide_smem_bytes(0, 0);
    return fail(SFFG_ERR_ARG, "sffg_env_create: robot mesh of " + std::to_string(n_robot) + " triangles does not fit the kernels' "
                              "shared-memory staging (at most " + std::to_string(room / sizeof(RobotTri)) + " on this device)");
  }
  const auto t0 = std::chrono::steady_clock::now();

  std::unique_ptr<sffg_env, int (*)(sffg_env *)> env(new sffg_env(), sffg_env_destroy);   // released on every error return

  // ---- robot
  std::vector<RobotTri> rob((size_t)n_robot);
  double rlo[3] = {1e300, 1e300, 1e300}, rhi[3] = {-1e300, -1e300, -1e300}, rad2 = 0;
  for (int64_t r = 0; r < n_robot; ++r) {
    make_robot_tri(robot_tris + 9 * r, &rob[(size_t)r]);
    for (int v = 0; v < 3; ++v) {
      const double *p = robot_tris + 9 * r + 3 * v;
      rad2 = std::max(rad2, p[0] * p[0] + p[1] * p[1] + p[2] * p[2]);
      for (int k = 0; k < 3; ++k) {
        rlo[k] = std::min(rlo[k], p[k]);
        rhi[k] = std::max(rhi[k], p[k]);
      }
    }
  }
  EnvDev &d = env->dev;
  d.n_robot = (int)n_robot;
  d.n_obst = (int)n_obst;
  for (int k = 0; k < 3; ++k) {
    const double c = 0.5 * (rlo[k] + rhi[k]);
    d.rob_c[k] = (float)c;
    d.rob_h[k] = round_up_f32(std::max(rhi[k] - (double)d.rob_c[k], (double)d.rob_c[k] - rlo[k]) * 1.0000001);
  }
  d.rob_radius = round_up_f32(std::sqrt(rad2) * 1.000001);
  // distinct robot vertices for the plane test of the clearance grid (nearest floats; the test's margin covers the rounding)
  std::vector<float4> verts;
  {
    std::vector<std::array<double, 3>> dv;
    for (int64_t i = 0; i < 3 * n_robot; ++i) dv.push_back({robot_tris[3 * i], robot_tris[3 * i + 1], robot_tris[3 * i + 2]});
    std::sort(dv.begin(), dv.end());
    dv.erase(std::unique(dv.begin(), dv.end()), dv.end());
    if (dv.size() <= (size_t)kPlaneVertCap)
      for (const auto &v : dv) verts.push_back(make_float4((float)v[0], (float)v[1], (float)v[2], 0.f));
  }

  size_t bytes = 0;
  SFFG_CUDA(upload(env->d_robot, rob.data(), rob.size() * sizeof(RobotTri), &bytes));
  if (!verts.empty()) SFFG_CUDA(upload(env->d_rob_verts, verts.data(), verts.size() * sizeof(float4), &bytes));
  SFFG_CUDA(upload(env->d_robot64, robot_tris, 9 * (size_t)n_robot * sizeof(double), &bytes));
  SFFG_CUDA(dev_alloc(env->d_counters, 10 * sizeof(unsigned long long)));
  SFFG_CUDA(cudaMemset(env->d_counters.get(), 0, 10 * sizeof(unsigned long long)));
  SFFG_CUDA(host_alloc(env->h_status, sizeof(int)));
  *env->h_status = 0;
  SFFG_CUDA(host_alloc(env->h_small, kSmallBytes));
  SFFG_CUDA(dev_alloc(env->d_work, 8 * sizeof(unsigned)));
  SFFG_CUDA(cudaMemset(env->d_work.get(), 0, 8 * sizeof(unsigned)));
  for (Stream &s : env->streams) SFFG_CUDA(make_stream(s));
  SFFG_CUDA(make_event(env->order_ev));
  d.robot = env->d_robot.get();
  d.robot64 = env->d_robot64.get();
  d.rob_verts = verts.empty() ? nullptr : env->d_rob_verts.get();
  d.n_rob_verts = (int)verts.size();
  d.counters = nullptr;
  d.status = env->h_status.get();   // unified addressing: the mapped host pointer is valid on the device
  d.work_counter = env->d_work.get();
  env->cfg.sm_count = g_rt.sm_count;
  env->cfg.blocks_per_sm = 0;

  env->info.n_robot_tris = n_robot;
  env->robot_bytes = (int64_t)bytes;
  rc = set_obstacles(env.get(), obst_tris, n_obst, build_mode);
  if (rc != SFFG_OK) return rc;
  env->info.build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  *out = env.release();
  return SFFG_OK;
}

int sffg_env_create(const double *obst_tris, int64_t n_obst, const double *robot_tris, int64_t n_robot, sffg_env **out) {
  return sffg_env_create_ex(obst_tris, n_obst, robot_tris, n_robot, SFFG_BUILD_AUTO, out);
}

int sffg_env_set_obstacles(sffg_env *env, const double *obst_tris, int64_t n_obst, int build_mode) {
  if (!env || n_obst < 0 || (n_obst > 0 && !obst_tris) || n_obst > 0x3fffffff || build_mode < 0 || build_mode > 2)
    return fail(SFFG_ERR_ARG, "sffg_env_set_obstacles: bad arguments");
  int rc = env_busy(env, "sffg_env_set_obstacles");
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(cudaDeviceSynchronize());   // nothing may still be traversing the old hierarchy
  const auto t0 = std::chrono::steady_clock::now();
  env->dev.n_obst = 0;
  *env->h_status = 4;                   // until the new set is complete every verdict call reports an error, never "free"
  rc = set_obstacles(env, obst_tris, n_obst, build_mode);
  if (rc == SFFG_OK) *env->h_status = 0;
  env->info.build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

int sffg_env_refit_obstacles(sffg_env *env, const double *obst_tris, int64_t n_obst) {
  if (!env || !obst_tris || n_obst <= 0) return fail(SFFG_ERR_ARG, "sffg_env_refit_obstacles: bad arguments");
  int rc = env_busy(env, "sffg_env_refit_obstacles");
  if (rc != SFFG_OK) return rc;
  if (n_obst != env->info.n_obst_tris || !env->d_order || env->level_base.empty())
    return fail(SFFG_ERR_ARG, "sffg_env_refit_obstacles: the soup must have the " + std::to_string(env->info.n_obst_tris) +
                                  " triangles of the current obstacle set, in the same order (use sffg_env_set_obstacles otherwise)");
  SFFG_CUDA(cudaDeviceSynchronize());   // nothing may still be traversing the boxes that are about to move
  const auto t0 = std::chrono::steady_clock::now();
  *env->h_status = 4;                   // until the refit is complete every verdict call reports an error, never "free"
  DevPtr<double> d_soup;
  cudaError_t e = upload_soup(env, d_soup, obst_tris, n_obst);
  double root_lo[3], root_hi[3];
  if (e == cudaSuccess)
    e = refit_bvh_device(d_soup.get(), (int)n_obst, env->d_slots.get(), env->d_tris64.get(), env->d_tris32.get(), env->d_order.get(),
                         env->level_base, env->level_count, env->streams[0].get(), root_lo, root_hi);
  d_soup.reset();
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(SFFG_ERR_CUDA, std::string("refit: ") + cudaGetErrorString(e));
  }
  // the top cut is re-chosen from the refitted head (its boxes changed)
  std::vector<ChildSlot> top;
  rc = read_top_cut(env, env->info.n_nodes, &top);
  if (rc != SFFG_OK) return rc;
  rc = finish_obstacles(env, top, root_lo, root_hi, n_obst, env->info.n_nodes, env->info.depth, env->info.built_on_device != 0,
                        (size_t)env->obst_bytes);
  if (rc == SFFG_OK) *env->h_status = 0;
  env->info.build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return rc;
}

int sffg_env_info(const sffg_env *env, sffg_env_info_t *out) {
  if (!env || !out) return fail(SFFG_ERR_ARG, "sffg_env_info: null argument");
  *out = env->info;
  return SFFG_OK;
}

int sffg_env_enable_counters(sffg_env *env, int on) {
  if (!env) return fail(SFFG_ERR_ARG, "null env");
  env->count = on != 0;
  SFFG_CUDA(cudaMemset(env->d_counters.get(), 0, 10 * sizeof(unsigned long long)));
  return SFFG_OK;
}

int sffg_env_read_counters(sffg_env *env, sffg_counters_t *out) {
  if (!env || !out) return fail(SFFG_ERR_ARG, "null argument");
  unsigned long long h[10];
  SFFG_CUDA(cudaDeviceSynchronize());
  SFFG_CUDA(cudaMemcpy(h, env->d_counters.get(), sizeof h, cudaMemcpyDeviceToHost));
  out->poses = (int64_t)h[0];
  out->poses_past_root = (int64_t)h[1];
  out->box_tests = (int64_t)h[2];
  out->pair_tests = (int64_t)h[3];
  out->exact_tests = (int64_t)h[4];
  out->traversal_steps = (int64_t)h[5];
  out->triangle_passes = (int64_t)h[6];
  out->triangles_transformed = (int64_t)h[7];
  out->exact_run = (int64_t)h[8];
  out->poses_past_grid = (int64_t)h[9];
  return SFFG_OK;
}

// picks the next work counter of the ring; *base_io points at the host-side base that the launch advances
static EnvDev env_view(sffg_env *env, unsigned **base_io) {
  EnvDev v = env->dev;
  const int slot = env->work_next++ & 7;
  v.counters = env->count ? env->d_counters.get() : nullptr;
  v.work_counter = env->d_work.get() + slot;
  *base_io = &env->work_base[slot];
  return v;
}

// stream ordering of the launches of one environment (see sffg_env::order_ev)
static int env_enter(sffg_env *env, cudaStream_t st) {
  if (env->order_pending && env->last_stream != st) SFFG_CUDA(cudaStreamWaitEvent(st, env->order_ev.get(), 0));
  return SFFG_OK;
}
static int env_leave(sffg_env *env, cudaStream_t st) {
  SFFG_CUDA(cudaEventRecord(env->order_ev.get(), st));
  env->last_stream = st;
  env->order_pending = true;
  return SFFG_OK;
}
// host-pointer calls run on the environment's own two streams and synchronise before they return
static int env_enter_host(sffg_env *env) {
  {
    const int rc = env_busy(env, "sffg (host-pointer call)");
    if (rc != SFFG_OK) return rc;
  }
  if (env->order_pending) {
    for (const Stream &s : env->streams) SFFG_CUDA(cudaStreamWaitEvent(s.get(), env->order_ev.get(), 0));
    env->order_pending = false;   // everything recorded so far is complete once this call has synchronised
  }
  return SFFG_OK;
}

// call after the streams were synchronised
static int check_status(sffg_env *env) {
  const int st = *reinterpret_cast<volatile int *>(env->h_status.get());
  if (st != 0) {
    if (st == 4)   // sticky: stays until sffg_env_set_obstacles or sffg_env_refit_obstacles succeeds
      return fail(SFFG_ERR_INTERNAL,
                  "the environment has no valid obstacle set: the last sffg_env_set_obstacles or sffg_env_refit_obstacles failed");
    *env->h_status = 0;
    if (st == 3) return fail(SFFG_ERR_INTERNAL, "peer barrier timed out: a rank of the gather group never signalled");
    return fail(SFFG_ERR_INTERNAL, "BVH traversal stack overflow: results of this call are invalid");
  }
  return SFFG_OK;
}

int sffg_env_sync_check(sffg_env *env) {
  if (!env) return fail(SFFG_ERR_ARG, "null env");
  SFFG_CUDA(cudaDeviceSynchronize());
  return check_status(env);
}

int sffg_collide_poses_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n, uint8_t *d_verdict_out,
                              void *stream) {
  if (!env || n < 0 || (n > 0 && (!d_poses || !d_verdict_out))) return fail(SFFG_ERR_ARG, "sffg_collide_poses_device: bad arguments");
  unsigned *base;
  int rc = env_enter(env, (cudaStream_t)stream);
  if (rc != SFFG_OK) return rc;
  EnvDev v = env_view(env, &base);
  SFFG_CUDA(launch_collide_poses(v, d_poses, poses_are_f64 ? 1 : 0, n, d_verdict_out, (cudaStream_t)stream, env->cfg,
                                 env->count, base));
  return env_leave(env, (cudaStream_t)stream);
}

// ---- multi-GPU: verdict all-gather fused into the kernel's stores (SURVEY 8e) -----------------------------------------
int sffg_peer_buffer_create(int64_t bytes, void **d_ptr_out, uint8_t handle_out[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (bytes <= 0 || !d_ptr_out || !handle_out) return fail(SFFG_ERR_ARG, "sffg_peer_buffer_create: bad arguments");
  void *p = nullptr;
  SFFG_CUDA(cudaMalloc(&p, (size_t)bytes));
  SFFG_CUDA(cudaMemset(p, 0, (size_t)bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    cudaGetLastError();
    return fail(SFFG_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
  }
  std::memcpy(handle_out, &h, 64);
  *d_ptr_out = p;
  return SFFG_OK;
}
int sffg_peer_buffer_open(const uint8_t handle[64], void **d_ptr_out) {
  if (!handle || !d_ptr_out) return fail(SFFG_ERR_ARG, "sffg_peer_buffer_open: bad arguments");
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, 64);
  SFFG_CUDA(cudaIpcOpenMemHandle(d_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
  return SFFG_OK;
}
int sffg_peer_buffer_close(void *d_ptr) {
  if (d_ptr) SFFG_CUDA(cudaIpcCloseMemHandle(d_ptr));
  return SFFG_OK;
}
int sffg_peer_buffer_destroy(void *d_ptr) {
  if (d_ptr) SFFG_CUDA(cudaFree(d_ptr));
  return SFFG_OK;
}

static int fill_flags(FlagSet *f, uint32_t *const *d_flags, int n_ranks, int my_rank, const char *who) {
  if (!d_flags || n_ranks < 1 || n_ranks > kMaxPeers || my_rank < 0 || my_rank >= n_ranks)
    return fail(SFFG_ERR_ARG, std::string(who) + ": bad rank arguments");
  f->n = n_ranks;
  f->me = my_rank;
  for (int r = 0; r < n_ranks; ++r) {
    if (!d_flags[r]) return fail(SFFG_ERR_ARG, std::string(who) + ": null flag array");
    f->p[r] = d_flags[r];
  }
  return SFFG_OK;
}

static int fill_outs(OutSet *outs, uint8_t *const *d_outs, int n_outs, const char *who) {
  if (!d_outs || n_outs < 1 || n_outs > kMaxPeers) return fail(SFFG_ERR_ARG, std::string(who) + ": bad destination list");
  outs->n = n_outs;
  for (int r = 0; r < n_outs; ++r) {
    if (!d_outs[r] || (reinterpret_cast<uintptr_t>(d_outs[r]) & 3u))
      return fail(SFFG_ERR_ARG, std::string(who) + ": every destination must be non-null and 4-byte aligned");
    outs->p[r] = d_outs[r];
  }
  return SFFG_OK;
}

int sffg_collide_poses_gather_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n, uint8_t *const *d_outs,
                                     int n_outs, void *stream) {
  if (!env || n < 0 || (n > 0 && !d_poses)) return fail(SFFG_ERR_ARG, "sffg_collide_poses_gather_device: bad arguments");
  OutSet outs;
  int rc = fill_outs(&outs, d_outs, n_outs, "sffg_collide_poses_gather_device");
  if (rc != SFFG_OK) return rc;
  GatherSync none{};
  unsigned *base;
  rc = env_enter(env, (cudaStream_t)stream);
  if (rc != SFFG_OK) return rc;
  EnvDev v = env_view(env, &base);
  SFFG_CUDA(launch_collide_poses_gather(v, d_poses, poses_are_f64 ? 1 : 0, n, outs, none, (cudaStream_t)stream, env->cfg, env->count, base));
  return env_leave(env, (cudaStream_t)stream);
}

int sffg_collide_poses_gather_sync_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n, uint8_t *const *d_outs,
                                          uint32_t *const *d_flags, int n_ranks, int my_rank, uint32_t signal_epoch,
                                          uint32_t wait_epoch, uint32_t *d_done_counter, void *stream) {
  if (!env || n < 0 || (n > 0 && !d_poses) || !d_done_counter || signal_epoch == 0)
    return fail(SFFG_ERR_ARG, "sffg_collide_poses_gather_sync_device: bad arguments");
  OutSet outs;
  GatherSync gs{};
  int rc = fill_outs(&outs, d_outs, n_ranks, "sffg_collide_poses_gather_sync_device");
  if (rc == SFFG_OK) rc = fill_flags(&gs.flags, d_flags, n_ranks, my_rank, "sffg_collide_poses_gather_sync_device");
  if (rc != SFFG_OK) return rc;
  gs.signal_epoch = signal_epoch;
  gs.wait_epoch = wait_epoch;
  gs.done_counter = d_done_counter;
  unsigned *base;
  rc = env_enter(env, (cudaStream_t)stream);
  if (rc != SFFG_OK) return rc;
  EnvDev v = env_view(env, &base);
  SFFG_CUDA(launch_collide_poses_gather(v, d_poses, poses_are_f64 ? 1 : 0, n, outs, gs, (cudaStream_t)stream, env->cfg, env->count, base));
  return env_leave(env, (cudaStream_t)stream);
}

int sffg_peer_wait_device(sffg_env *env, uint32_t *const *d_flags, int n_ranks, int my_rank, uint32_t epoch, void *stream) {
  FlagSet f;
  int rc = fill_flags(&f, d_flags, n_ranks, my_rank, "sffg_peer_wait_device");
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(launch_peer_barrier(f, epoch, false, env ? env->h_status.get() : nullptr, (cudaStream_t)stream));
  return SFFG_OK;
}

int sffg_peer_barrier_device(sffg_env *env, uint32_t *const *d_flags, int n_ranks, int my_rank, uint32_t epoch, void *stream) {
  FlagSet f;
  int rc = fill_flags(&f, d_flags, n_ranks, my_rank, "sffg_peer_barrier_device");
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(launch_peer_barrier(f, epoch, true, nullptr, (cudaStream_t)stream));
  SFFG_CUDA(launch_peer_barrier(f, epoch, false, env ? env->h_status.get() : nullptr, (cudaStream_t)stream));
  return SFFG_OK;
}

// Host-pointer pose calls (verdicts, distances) stage through one path: planner-sized batches through the pinned mapped
// area (one kernel reading and writing it, one synchronisation, no DMA copies), larger ones in chunks of 2^20 poses on the
// environment's two streams.  Pose i takes psz input bytes; output k (k < 2, null = not requested) takes osz[k] bytes per
// pose.  launch(env view, d_in, cnt, d_out, stream, work base) enqueues the kernel for cnt poses.
extern "C++" {   // (a template cannot have C linkage)
template <class Launch>
static int pose_call_host(sffg_env *env, const void *poses, size_t psz, int64_t n, void *const out[2], const size_t osz[2],
                          const Launch &launch) {
  const size_t ob[2] = {out[0] ? osz[0] : 0, out[1] ? osz[1] : 0};
  unsigned *base;
  {
    const int rc0 = env_enter_host(env);
    if (rc0 != SFFG_OK) return rc0;
  }
  if ((size_t)n * psz <= EnvStaging::kInBytes && (size_t)n * (ob[0] + ob[1]) <= EnvStaging::kOutBytes) {
    cudaStream_t st = env->streams[0].get();
    const EnvStaging h = env->staging();
    void *const d_out[2] = {out[0] ? h.out() : nullptr, out[1] ? h.out() + (size_t)n * ob[0] : nullptr};
    std::memcpy(h.in(), poses, (size_t)n * psz);
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch(v, h.in(), n, d_out, st, base));
    SFFG_CUDA(cudaStreamSynchronize(st));
    for (int k = 0; k < 2; ++k)
      if (out[k]) std::memcpy(out[k], d_out[k], (size_t)n * ob[k]);
    return check_status(env);
  }
  const int64_t chunk = 1 << 20;
  int s = 0;
  for (int64_t off = 0; off < n; off += chunk, s ^= 1) {
    const int64_t cnt = std::min(chunk, n - off);
    cudaStream_t st = env->streams[s].get();
    SFFG_CUDA(cudaStreamSynchronize(st));   // buffers of this stream are free again
    DevBuf *const bufs[2] = {&env->out[s], &env->aux[s]};
    int rc = env->in[s].reserve((size_t)cnt * psz);
    for (int k = 0; k < 2 && rc == SFFG_OK; ++k)
      if (out[k]) rc = bufs[k]->reserve((size_t)cnt * ob[k]);
    if (rc != SFFG_OK) return rc;
    void *const d_out[2] = {out[0] ? bufs[0]->p : nullptr, out[1] ? bufs[1]->p : nullptr};
    SFFG_CUDA(cudaMemcpyAsync(env->in[s].p, (const char *)poses + (size_t)off * psz, (size_t)cnt * psz, cudaMemcpyHostToDevice, st));
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch(v, env->in[s].p, cnt, d_out, st, base));
    for (int k = 0; k < 2; ++k)
      if (out[k])
        SFFG_CUDA(cudaMemcpyAsync((char *)out[k] + (size_t)off * ob[k], d_out[k], (size_t)cnt * ob[k], cudaMemcpyDeviceToHost, st));
  }
  for (const Stream &st : env->streams) SFFG_CUDA(cudaStreamSynchronize(st.get()));
  return check_status(env);
}
}  // extern "C++"

static int collide_poses_host(sffg_env *env, const void *poses, int fmt, int64_t n, uint8_t *verdict_out) {
  if (!env || n < 0 || (n > 0 && (!poses || !verdict_out))) return fail(SFFG_ERR_ARG, "sffg_collide_poses: bad arguments");
  if (n == 0) return SFFG_OK;
  const size_t psz = fmt == 0 ? 24 : (fmt == 1 ? 48 : 96);
  void *const out[2] = {verdict_out, nullptr};
  const size_t osz[2] = {1, 0};
  return pose_call_host(env, poses, psz, n, out, osz,
                        [&](const EnvDev &v, const void *d_in, int64_t cnt, void *const *d_out, cudaStream_t st, unsigned *base) {
                          return launch_collide_poses(v, d_in, fmt, cnt, (uint8_t *)d_out[0], st, env->cfg, env->count, base);
                        });
}

// ---- separation distance per pose ------------------------------------------------------------------------------------
static int distance_args(const sffg_env *env, const void *poses, int64_t n, double max_dist, const double *dist_out,
                         const char *who) {
  if (!env || n < 0 || (n > 0 && (!poses || !dist_out)) || !(max_dist > 0))
    return fail(SFFG_ERR_ARG, std::string(who) + ": bad arguments (max_dist must be > 0)");
  return SFFG_OK;
}

int sffg_distance_poses(sffg_env *env, const void *poses, int poses_are_f64, int64_t n, double max_dist, double *dist_out,
                        double *points_out) {
  const int rc = distance_args(env, poses, n, max_dist, dist_out, "sffg_distance_poses");
  if (rc != SFFG_OK || n == 0) return rc;
  const int fmt = poses_are_f64 ? 1 : 0;
  void *const out[2] = {dist_out, points_out};
  const size_t osz[2] = {8, 48};
  return pose_call_host(env, poses, fmt ? 48 : 24, n, out, osz,
                        [&](const EnvDev &v, const void *d_in, int64_t cnt, void *const *d_out, cudaStream_t st, unsigned *base) {
                          return launch_distance_poses(v, d_in, fmt, cnt, max_dist, (double *)d_out[0], (double *)d_out[1], st,
                                                       env->cfg, base);
                        });
}

int sffg_distance_poses_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n, double max_dist,
                               double *d_dist_out, double *d_points_out, void *stream) {
  int rc = distance_args(env, d_poses, n, max_dist, d_dist_out, "sffg_distance_poses_device");
  if (rc != SFFG_OK) return rc;
  unsigned *base;
  rc = env_enter(env, (cudaStream_t)stream);
  if (rc != SFFG_OK) return rc;
  EnvDev v = env_view(env, &base);
  SFFG_CUDA(launch_distance_poses(v, d_poses, poses_are_f64 ? 1 : 0, n, max_dist, d_dist_out, d_points_out,
                                  (cudaStream_t)stream, env->cfg, base));
  return env_leave(env, (cudaStream_t)stream);
}

int sffg_collide_poses_f32(sffg_env *env, const float *poses, int64_t n, uint8_t *verdict_out) {
  return collide_poses_host(env, poses, 0, n, verdict_out);
}
int sffg_collide_poses_f64(sffg_env *env, const double *poses, int64_t n, uint8_t *verdict_out) {
  return collide_poses_host(env, poses, 1, n, verdict_out);
}
int sffg_collide_transforms_f64(sffg_env *env, const double *rt, int64_t n, uint8_t *verdict_out) {
  return collide_poses_host(env, rt, 2, n, verdict_out);
}

// arguments of the edge and move calls; the sweep call has no sample spacing and passes check_sample = false
static int check_segment_args(const sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist,
                              int rot_mode, const void *out, const char *who, bool check_sample = true) {
  if (!env || m < 0 || (m > 0 && (!starts || !ends || !out)) || (check_sample && !(sample_dist > 0)) ||
      (rot_mode != SFFG_ROT_REFERENCE && rot_mode != SFFG_ROT_INTERPOLATE))
    return fail(SFFG_ERR_ARG, std::string(who) + ": bad arguments");
  return SFFG_OK;
}

int sffg_check_edges_device(sffg_env *env, const double *d_starts, const double *d_ends, int64_t m, double sample_dist,
                            int rot_mode, uint8_t *d_free_out, int32_t *d_first_hit_out, void *stream) {
  int rc = check_segment_args(env, d_starts, d_ends, m, sample_dist, rot_mode, d_free_out, "sffg_check_edges_device");
  if (rc != SFFG_OK) return rc;
  unsigned *base;
  rc = env_enter(env, (cudaStream_t)stream);
  if (rc != SFFG_OK) return rc;
  EnvDev v = env_view(env, &base);
  int *scratch = nullptr;
  if (m < 8192) {   // small batches: several warps per edge (needs a scratch word per edge)
    if ((size_t)m * sizeof(int) > env->fh.cap) SFFG_CUDA(cudaStreamSynchronize((cudaStream_t)stream));   // (growing frees the old block)
    rc = env->fh.reserve((size_t)m * sizeof(int));
    if (rc != SFFG_OK) return rc;
    scratch = (int *)env->fh.p;
  }
  SFFG_CUDA(launch_check_edges(v, d_starts, d_ends, m, sample_dist, rot_mode, d_free_out, d_first_hit_out,
                               (cudaStream_t)stream, env->cfg, env->count, base, scratch));
  return env_leave(env, (cudaStream_t)stream);
}

static int check_edges_impl(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                            uint8_t *free_out, int32_t *first_hit_out, bool async);
int sffg_check_edges(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                     uint8_t *free_out, int32_t *first_hit_out) {
  return check_edges_impl(env, starts, ends, m, sample_dist, rot_mode, free_out, first_hit_out, false);
}
int sffg_check_edges_begin(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                           uint8_t *free_out, int32_t *first_hit_out) {
  return check_edges_impl(env, starts, ends, m, sample_dist, rot_mode, free_out, first_hit_out, true);
}

// completes the asynchronous call pending on this environment (no-op when none is)
int sffg_env_end(sffg_env *env) {
  if (!env) return fail(SFFG_ERR_ARG, "sffg_env_end: null environment");
  if (env->pend.kind == 0) return SFFG_OK;
  const sffg_env::Pending c = env->pend;
  env->pend.kind = 0;
  SFFG_CUDA(cudaStreamSynchronize(env->streams[0].get()));
  const EnvStaging h = env->staging();
  if (c.kind == 1) {
    std::memcpy(c.out, h.edge_free(c.m), (size_t)c.m);
    if (c.first_out) std::memcpy(c.first_out, h.edge_first_hit(), (size_t)c.m * 4);
  } else {
    const uint8_t *h_free = h.move_free(), *h_hit = h.move_hit(c.m);
    for (int64_t i = 0; i < c.m; ++i) c.out[i] = (uint8_t)(h_free[i] && !h_hit[i]);
  }
  return check_status(env);
}

// planner-sized edge and move calls: the end points go to device memory (starts, then ends) with one DMA from the
// staging area, because every warp that shares an edge re-reads them
static int stage_segments(sffg_env *env, const double *starts, const double *ends, int64_t m, double **ds, double **de) {
  int rc = env->in[0].reserve((size_t)m * 96);
  if (rc == SFFG_OK) rc = env->fh.reserve((size_t)m * sizeof(int));
  if (rc != SFFG_OK) return rc;
  unsigned char *h_in = env->staging().in();
  std::memcpy(h_in, starts, (size_t)m * 48);
  std::memcpy(h_in + (size_t)m * 48, ends, (size_t)m * 48);
  *ds = (double *)env->in[0].p;
  *de = *ds + 6 * m;
  SFFG_CUDA(cudaMemcpyAsync(*ds, h_in, (size_t)m * 96, cudaMemcpyHostToDevice, env->streams[0].get()));
  return SFFG_OK;
}

// the last step of a planner-sized edge or move call, once all of it is enqueued on the first stream: the blocking form
// completes it, the asynchronous form leaves it pending for sffg_env_end (*_device launches issued before the end call are
// ordered behind it)
static int env_commit(sffg_env *env, const sffg_env::Pending &p, bool async) {
  if (async) {
    const int rc = env_leave(env, env->streams[0].get());
    if (rc != SFFG_OK) return rc;
  }
  env->pend = p;
  return async ? SFFG_OK : sffg_env_end(env);
}

// Host-pointer edge calls too large for the staging area run in chunks of 2^18 edges on the environment's two streams in
// turn.  run(s, off, cnt, ds, de, st) enqueues the kernels of one chunk, whose end points are at ds / de in device memory,
// and the copies of its results on st (the buffers of stream s are free again when it is called).
extern "C++" {   // (a template cannot have C linkage)
template <class Run>
static int edge_call_chunks(sffg_env *env, const double *starts, const double *ends, int64_t m, const Run &run) {
  const int64_t chunk = 1 << 18;
  int s = 0;
  for (int64_t off = 0; off < m; off += chunk, s ^= 1) {
    const int64_t cnt = std::min(chunk, m - off);
    cudaStream_t st = env->streams[s].get();
    SFFG_CUDA(cudaStreamSynchronize(st));
    int rc = env->in[s].reserve((size_t)cnt * 96);
    if (rc != SFFG_OK) return rc;
    double *ds = (double *)env->in[s].p, *de = ds + 6 * cnt;
    SFFG_CUDA(cudaMemcpyAsync(ds, starts + 6 * off, (size_t)cnt * 48, cudaMemcpyHostToDevice, st));
    SFFG_CUDA(cudaMemcpyAsync(de, ends + 6 * off, (size_t)cnt * 48, cudaMemcpyHostToDevice, st));
    if ((rc = run(s, off, cnt, ds, de, st)) != SFFG_OK) return rc;
  }
  for (const Stream &st : env->streams) SFFG_CUDA(cudaStreamSynchronize(st.get()));
  return check_status(env);
}
}  // extern "C++"

static int check_edges_impl(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                            uint8_t *free_out, int32_t *first_hit_out, bool async) {
  int rc = check_segment_args(env, starts, ends, m, sample_dist, rot_mode, free_out, "sffg_check_edges");
  if (rc != SFFG_OK || m == 0) return rc;
  if ((rc = env_enter_host(env)) != SFFG_OK) return rc;
  unsigned *base;
  if ((size_t)m * 96 <= EnvStaging::kInBytes && (size_t)m * 5 <= EnvStaging::kOutBytes) {
    // planner-sized call: the results are written straight into pinned mapped memory
    const EnvStaging h = env->staging();
    double *ds, *de;
    if ((rc = stage_segments(env, starts, ends, m, &ds, &de)) != SFFG_OK) return rc;
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch_check_edges(v, ds, de, m, sample_dist, rot_mode, h.edge_free(m), h.edge_first_hit(), env->streams[0].get(),
                                 env->cfg, env->count, base, (int *)env->fh.p));
    return env_commit(env, sffg_env::Pending{1, m, free_out, first_hit_out}, async);
  }
  return edge_call_chunks(env, starts, ends, m, [&](int s, int64_t off, int64_t cnt, double *ds, double *de, cudaStream_t st) {
    int rc2 = env->out[s].reserve((size_t)cnt);
    if (rc2 == SFFG_OK) rc2 = env->aux[s].reserve((size_t)cnt * 4);
    if (rc2 != SFFG_OK) return rc2;
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch_check_edges(v, ds, de, cnt, sample_dist, rot_mode, (uint8_t *)env->out[s].p,
                                 (int32_t *)env->aux[s].p, st, env->cfg, env->count, base, nullptr));
    SFFG_CUDA(cudaMemcpyAsync(free_out + off, env->out[s].p, (size_t)cnt, cudaMemcpyDeviceToHost, st));
    if (first_hit_out)
      SFFG_CUDA(cudaMemcpyAsync(first_hit_out + off, env->aux[s].p, (size_t)cnt * 4, cudaMemcpyDeviceToHost, st));
    return SFFG_OK;
  });
}

// ---- separation distance per edge --------------------------------------------------------------------------------
static int distance_edges_args(const sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist,
                               int rot_mode, double max_dist, const double *dist_out, const char *who) {
  const int rc = check_segment_args(env, starts, ends, m, sample_dist, rot_mode, dist_out, who);
  if (rc != SFFG_OK) return rc;
  if (!(max_dist > 0)) return fail(SFFG_ERR_ARG, std::string(who) + ": bad arguments (max_dist must be > 0)");
  return SFFG_OK;
}

// scratch of an edge distance call in environment memory: the verdict launch's first hits and free flags and, when its
// edges may be split over several warps (`split`), the verdict launch's per-edge word and the distance kernel's records.
// Growing frees the old block, so `st` (ordered behind every earlier launch of the environment) is drained first.
static int edge_distance_scratch(sffg_env *env, int64_t m, bool split, cudaStream_t st, EdgeDistScratch *scr) {
  const size_t rec = split ? distance_edges_rec_bytes(m, env->cfg) : 0;
  const size_t fh = split ? (size_t)m * sizeof(int) : 0;
  if ((size_t)m * 5 > env->edge_scr.cap || rec > env->edge_rec.cap || fh > env->fh.cap) SFFG_CUDA(cudaStreamSynchronize(st));
  int rc = env->edge_scr.reserve((size_t)m * 5);
  if (rc == SFFG_OK) rc = env->fh.reserve(fh);
  if (rc == SFFG_OK) rc = env->edge_rec.reserve(rec);
  if (rc != SFFG_OK) return rc;
  scr->first_hit = (int32_t *)env->edge_scr.p;
  scr->free = (uint8_t *)env->edge_scr.p + (size_t)m * 4;
  scr->fh = split ? (int *)env->fh.p : nullptr;
  scr->recs = rec ? env->edge_rec.p : nullptr;
  return SFFG_OK;
}

int sffg_distance_edges(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                        double max_dist, double *dist_out, int32_t *index_out, double *points_out) {
  int rc = distance_edges_args(env, starts, ends, m, sample_dist, rot_mode, max_dist, dist_out, "sffg_distance_edges");
  if (rc != SFFG_OK || m == 0) return rc;
  if ((rc = env_enter_host(env)) != SFFG_OK) return rc;
  unsigned *base;
  if ((size_t)m * 96 <= EnvStaging::kInBytes && (size_t)m * 60 <= EnvStaging::kOutBytes) {
    // planner-sized call: both kernels on one stream, results straight into pinned mapped memory, one synchronisation
    cudaStream_t st = env->streams[0].get();
    const EnvStaging h = env->staging();
    EdgeDistScratch scr;
    double *ds, *de;
    if ((rc = edge_distance_scratch(env, m, true, st, &scr)) != SFFG_OK) return rc;
    if ((rc = stage_segments(env, starts, ends, m, &ds, &de)) != SFFG_OK) return rc;
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch_distance_edges(v, ds, de, m, sample_dist, rot_mode, max_dist, h.edge_dist(), index_out ? h.edge_index(m) : nullptr,
                                    points_out ? h.edge_points(m) : nullptr, st, env->cfg, base, scr));
    SFFG_CUDA(cudaStreamSynchronize(st));
    std::memcpy(dist_out, h.edge_dist(), (size_t)m * 8);
    if (index_out) std::memcpy(index_out, h.edge_index(m), (size_t)m * 4);
    if (points_out) std::memcpy(points_out, h.edge_points(m), (size_t)m * 48);
    return check_status(env);
  }
  return edge_call_chunks(env, starts, ends, m, [&](int s, int64_t off, int64_t cnt, double *ds, double *de, cudaStream_t st) {
    // out[s]: distances [cnt], points [cnt][6], indices [cnt]; aux[s]: the verdict launch's first hits and free flags
    int rc2 = env->out[s].reserve((size_t)cnt * 60);
    if (rc2 == SFFG_OK) rc2 = env->aux[s].reserve((size_t)cnt * 5);
    if (rc2 != SFFG_OK) return rc2;
    double *d_dist = (double *)env->out[s].p, *d_points = d_dist + cnt;
    int32_t *d_index = (int32_t *)(d_points + 6 * cnt);
    const EdgeDistScratch scr{(uint8_t *)env->aux[s].p + (size_t)cnt * 4, (int32_t *)env->aux[s].p, nullptr, nullptr};
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch_distance_edges(v, ds, de, cnt, sample_dist, rot_mode, max_dist, d_dist, index_out ? d_index : nullptr,
                                    points_out ? d_points : nullptr, st, env->cfg, base, scr));
    SFFG_CUDA(cudaMemcpyAsync(dist_out + off, d_dist, (size_t)cnt * 8, cudaMemcpyDeviceToHost, st));
    if (index_out) SFFG_CUDA(cudaMemcpyAsync(index_out + off, d_index, (size_t)cnt * 4, cudaMemcpyDeviceToHost, st));
    if (points_out) SFFG_CUDA(cudaMemcpyAsync(points_out + 6 * off, d_points, (size_t)cnt * 48, cudaMemcpyDeviceToHost, st));
    return SFFG_OK;
  });
}

int sffg_distance_edges_device(sffg_env *env, const double *d_starts, const double *d_ends, int64_t m, double sample_dist,
                               int rot_mode, double max_dist, double *d_dist_out, int32_t *d_index_out, double *d_points_out,
                               void *stream) {
  int rc = distance_edges_args(env, d_starts, d_ends, m, sample_dist, rot_mode, max_dist, d_dist_out, "sffg_distance_edges_device");
  if (rc != SFFG_OK) return rc;
  unsigned *base;
  rc = env_enter(env, (cudaStream_t)stream);
  if (rc != SFFG_OK) return rc;
  // small batches: several warps per edge, as sffg_check_edges_device
  EdgeDistScratch scr;
  if ((rc = edge_distance_scratch(env, m, m < 8192, (cudaStream_t)stream, &scr)) != SFFG_OK) return rc;
  EnvDev v = env_view(env, &base);
  SFFG_CUDA(launch_distance_edges(v, d_starts, d_ends, m, sample_dist, rot_mode, max_dist, d_dist_out, d_index_out, d_points_out,
                                  (cudaStream_t)stream, env->cfg, base, scr));
  return env_leave(env, (cudaStream_t)stream);
}

// ---- continuous edge check -----------------------------------------------------------------------------------------
// margin: positive, finite and at least 1e-6 max(1, max |obstacle coordinate|), which bounds the steps per edge
static int sweep_args(const sffg_env *env, const double *starts, const double *ends, int64_t m, int rot_mode, double margin,
                      const uint8_t *clear_out, const char *who) {
  const int rc = check_segment_args(env, starts, ends, m, 0.0, rot_mode, clear_out, who, false);
  if (rc != SFFG_OK) return rc;
  if (!(margin > 0) || !std::isfinite(margin) || margin < 1e-6 * std::max(1.0, env->obst_max_abs))
    return fail(SFFG_ERR_ARG, std::string(who) + ": bad arguments (margin must be finite and >= 1e-6 max(1, max |obstacle "
                              "coordinate|) = " + std::to_string(1e-6 * std::max(1.0, env->obst_max_abs)) + ")");
  return SFFG_OK;
}

// scratch of a sweep call whose edges may be split over several warps: the per-edge stop word and the per-warp records.
// Growing frees the old block, so `st` (ordered behind every earlier launch of the environment) is drained first.
static int sweep_scratch(sffg_env *env, int64_t m, bool split, cudaStream_t st, SweepScratch *scr) {
  const size_t rec = split ? sweep_edges_rec_bytes(m, env->cfg) : 0;
  const size_t fh = split ? (size_t)m * sizeof(int) : 0;
  if (rec > env->edge_rec.cap || fh > env->fh.cap) SFFG_CUDA(cudaStreamSynchronize(st));
  int rc = env->fh.reserve(fh);
  if (rc == SFFG_OK) rc = env->edge_rec.reserve(rec);
  if (rc != SFFG_OK) return rc;
  scr->stop = rec ? (int *)env->fh.p : nullptr;
  scr->recs = rec ? env->edge_rec.p : nullptr;
  return SFFG_OK;
}

int sffg_sweep_edges(sffg_env *env, const double *starts, const double *ends, int64_t m, int rot_mode, double margin,
                     uint8_t *clear_out, double *t_out, double *dist_out) {
  int rc = sweep_args(env, starts, ends, m, rot_mode, margin, clear_out, "sffg_sweep_edges");
  if (rc != SFFG_OK || m == 0) return rc;
  if ((rc = env_enter_host(env)) != SFFG_OK) return rc;
  unsigned *base;
  if ((size_t)m * 96 <= EnvStaging::kInBytes && (size_t)m * 17 <= EnvStaging::kOutBytes) {
    // planner-sized call: results straight into pinned mapped memory, one synchronisation
    cudaStream_t st = env->streams[0].get();
    const EnvStaging h = env->staging();
    SweepScratch scr;
    double *ds, *de;
    if ((rc = sweep_scratch(env, m, true, st, &scr)) != SFFG_OK) return rc;
    if ((rc = stage_segments(env, starts, ends, m, &ds, &de)) != SFFG_OK) return rc;
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch_sweep_edges(v, ds, de, m, rot_mode, margin, h.sweep_clear(m), t_out ? h.sweep_t() : nullptr,
                                 dist_out ? h.sweep_dist(m) : nullptr, st, env->cfg, base, scr));
    SFFG_CUDA(cudaStreamSynchronize(st));
    std::memcpy(clear_out, h.sweep_clear(m), (size_t)m);
    if (t_out) std::memcpy(t_out, h.sweep_t(), (size_t)m * 8);
    if (dist_out) std::memcpy(dist_out, h.sweep_dist(m), (size_t)m * 8);
    return check_status(env);
  }
  return edge_call_chunks(env, starts, ends, m, [&](int s, int64_t off, int64_t cnt, double *ds, double *de, cudaStream_t st) {
    // out[s]: stop parameters [cnt], distances [cnt], clear flags [cnt]; one warp per edge (no scratch)
    const int rc2 = env->out[s].reserve((size_t)cnt * 17);
    if (rc2 != SFFG_OK) return rc2;
    double *d_t = (double *)env->out[s].p, *d_dist = d_t + cnt;
    uint8_t *d_clear = (uint8_t *)(d_dist + cnt);
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch_sweep_edges(v, ds, de, cnt, rot_mode, margin, d_clear, t_out ? d_t : nullptr, dist_out ? d_dist : nullptr, st,
                                 env->cfg, base, SweepScratch{nullptr, nullptr}));
    SFFG_CUDA(cudaMemcpyAsync(clear_out + off, d_clear, (size_t)cnt, cudaMemcpyDeviceToHost, st));
    if (t_out) SFFG_CUDA(cudaMemcpyAsync(t_out + off, d_t, (size_t)cnt * 8, cudaMemcpyDeviceToHost, st));
    if (dist_out) SFFG_CUDA(cudaMemcpyAsync(dist_out + off, d_dist, (size_t)cnt * 8, cudaMemcpyDeviceToHost, st));
    return SFFG_OK;
  });
}

int sffg_sweep_edges_device(sffg_env *env, const double *d_starts, const double *d_ends, int64_t m, int rot_mode, double margin,
                            uint8_t *d_clear_out, double *d_t_out, double *d_dist_out, void *stream) {
  int rc = sweep_args(env, d_starts, d_ends, m, rot_mode, margin, d_clear_out, "sffg_sweep_edges_device");
  if (rc != SFFG_OK) return rc;
  unsigned *base;
  rc = env_enter(env, (cudaStream_t)stream);
  if (rc != SFFG_OK) return rc;
  // small batches: several warps per edge, as sffg_check_edges_device
  SweepScratch scr;
  if ((rc = sweep_scratch(env, m, m < 8192, (cudaStream_t)stream, &scr)) != SFFG_OK) return rc;
  EnvDev v = env_view(env, &base);
  SFFG_CUDA(launch_sweep_edges(v, d_starts, d_ends, m, rot_mode, margin, d_clear_out, d_t_out, d_dist_out, (cudaStream_t)stream,
                               env->cfg, base, scr));
  return env_leave(env, (cudaStream_t)stream);
}

static int check_moves_impl(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                            uint8_t *ok_out, bool async);
int sffg_check_moves(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                     uint8_t *ok_out) {
  return check_moves_impl(env, starts, ends, m, sample_dist, rot_mode, ok_out, false);
}
int sffg_check_moves_begin(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                           uint8_t *ok_out) {
  return check_moves_impl(env, starts, ends, m, sample_dist, rot_mode, ok_out, true);
}
static int check_moves_impl(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist, int rot_mode,
                            uint8_t *ok_out, bool async) {
  int rc = check_segment_args(env, starts, ends, m, sample_dist, rot_mode, ok_out, "sffg_check_moves");
  if (rc != SFFG_OK || m == 0) return rc;
  if ((rc = env_enter_host(env)) != SFFG_OK) return rc;
  if ((size_t)m * 96 <= EnvStaging::kInBytes && (size_t)m * 6 <= EnvStaging::kOutBytes) {
    // planner-sized call: one upload, the pose kernel on the end points and the edge kernel on the segments back to back
    // on one stream, results straight into pinned mapped memory, one synchronisation
    cudaStream_t st = env->streams[0].get();
    const EnvStaging h = env->staging();
    double *ds, *de;
    if ((rc = stage_segments(env, starts, ends, m, &ds, &de)) != SFFG_OK) return rc;
    unsigned *base;
    EnvDev v = env_view(env, &base);
    SFFG_CUDA(launch_collide_poses(v, de, 1, m, h.move_hit(m), st, env->cfg, env->count, base));
    EnvDev w = env_view(env, &base);
    SFFG_CUDA(launch_check_edges(w, ds, de, m, sample_dist, rot_mode, h.move_free(), nullptr, st, env->cfg, env->count, base,
                                 (int *)env->fh.p));
    return env_commit(env, sffg_env::Pending{2, m, ok_out, nullptr}, async);
  }
  std::vector<uint8_t> hit((size_t)m);
  rc = sffg_collide_poses_f64(env, ends, m, hit.data());
  if (rc == SFFG_OK) rc = sffg_check_edges(env, starts, ends, m, sample_dist, rot_mode, ok_out, nullptr);
  if (rc != SFFG_OK) return rc;
  for (int64_t i = 0; i < m; ++i) ok_out[i] = (uint8_t)(ok_out[i] && !hit[(size_t)i]);
  return SFFG_OK;
}

int sffg_gen_poses_device(uint64_t seed, uint64_t first_index, int64_t n, const float range[6], float *d_poses_out,
                          void *stream) {
  if (n < 0 || !range || (n > 0 && !d_poses_out)) return fail(SFFG_ERR_ARG, "sffg_gen_poses_device: bad arguments");
  int rc = ensure_runtime();
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(launch_gen_poses(seed, first_index, n, range, d_poses_out, (cudaStream_t)stream));
  return SFFG_OK;
}

// ---- neighbour index ------------------------------------------------------------------------------------------
int sffg_index_create(int dim, sffg_index **out) {
  if (!out || (dim != 2 && dim != 6)) return fail(SFFG_ERR_ARG, "sffg_index_create: dim must be 2 or 6");
  int rc = ensure_runtime();
  if (rc != SFFG_OK) return rc;
  std::unique_ptr<sffg_index, int (*)(sffg_index *)> idx(new sffg_index(), sffg_index_destroy);   // released on every error return
  idx->dim = dim;
  const char *pr = std::getenv("SFFG_KNN_PRUNING");
  idx->pruning = !(pr && pr[0] == '0');
  SFFG_CUDA(make_stream(idx->stream));
  SFFG_CUDA(make_event(idx->ev));
  SFFG_CUDA(make_event(idx->add_ev));
  SFFG_CUDA(dev_alloc(idx->d_total, sizeof(unsigned long long)));
  SFFG_CUDA(host_alloc(idx->h_small, kSmallBytes));
  // storage exists from the start: the scan kernels may touch the first block of an empty index
  idx->cap = 4096 + 128;
  SFFG_CUDA(dev_alloc(idx->d_coords, (size_t)idx->cap * dim * sizeof(float)));
  SFFG_CUDA(cudaMemset(idx->d_coords.get(), 0, (size_t)idx->cap * dim * sizeof(float)));
  SFFG_CUDA(dev_alloc(idx->d_amax, 256));
  SFFG_CUDA(cudaMemset(idx->d_amax.get(), 0, 256));
  *out = idx.release();
  return SFFG_OK;
}

int sffg_index_destroy(sffg_index *idx) {
  if (!idx) return SFFG_OK;
  if (idx->stream) cudaStreamSynchronize(idx->stream.get());
  delete idx;
  return SFFG_OK;
}

int64_t sffg_index_size(const sffg_index *idx) { return idx ? idx->n : -1; }

static int index_grow(sffg_index *idx, int64_t need, cudaStream_t st) {
  if (need + 128 <= idx->cap) return SFFG_OK;
  int64_t ncap = std::max<int64_t>({need, idx->cap * 2, 4096});
  ncap = (ncap + 31) / 32 * 32 + 128;   // spare blocks: the scan kernels prefetch up to 3 blocks past the end of a slice
  DevPtr<float> nc;
  SFFG_CUDA(dev_alloc(nc, (size_t)ncap * idx->dim * sizeof(float)));
  for (int c = 0; c < idx->dim && idx->n > 0; ++c)
    SFFG_CUDA(cudaMemcpyAsync(nc.get() + (size_t)c * ncap, idx->d_coords.get() + (size_t)c * idx->cap, (size_t)idx->n * sizeof(float),
                              cudaMemcpyDeviceToDevice, st));
  SFFG_CUDA(cudaStreamSynchronize(st));
  idx->d_coords = std::move(nc);
  idx->cap = ncap;
  return SFFG_OK;
}

int sffg_index_add_device(sffg_index *idx, const float *d_pts, int64_t n, void *stream) {
  if (!idx || n < 0 || (n > 0 && !d_pts)) return fail(SFFG_ERR_ARG, "sffg_index_add_device: bad arguments");
  if (n == 0) return SFFG_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = index_grow(idx, idx->n + n, st);
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(launch_index_append(idx->d_coords.get(), idx->cap, idx->dim, idx->n, d_pts, n, idx->d_amax.get(), st));
  idx->n += n;
  return SFFG_OK;
}

int sffg_index_add(sffg_index *idx, const float *pts, int64_t n) {
  if (!idx || n < 0 || (n > 0 && !pts)) return fail(SFFG_ERR_ARG, "sffg_index_add: bad arguments");
  if (n == 0) return SFFG_OK;
  int rc = index_busy(idx, "sffg_index_add");
  if (rc != SFFG_OK) return rc;
  rc = idx->stage.reserve((size_t)n * idx->dim * sizeof(float));
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(cudaMemcpyAsync(idx->stage.p, pts, (size_t)n * idx->dim * sizeof(float), cudaMemcpyHostToDevice, idx->stream.get()));
  rc = sffg_index_add_device(idx, (const float *)idx->stage.p, n, idx->stream.get());
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(cudaStreamSynchronize(idx->stream.get()));
  return SFFG_OK;
}

int sffg_index_add_multi_begin(sffg_index *const *idx, const int64_t *n_per, int n_idx, const float *pts) {
  if (!idx || !n_per || n_idx < 1) return fail(SFFG_ERR_ARG, "sffg_index_add_multi: bad arguments");
  int64_t total = 0;
  const int dim = idx[0] ? idx[0]->dim : 0;
  for (int i = 0; i < n_idx; ++i) {
    if (!idx[i] || idx[i]->dim != dim || n_per[i] < 0) return fail(SFFG_ERR_ARG, "sffg_index_add_multi: bad index / count");
    total += n_per[i];
  }
  if (total == 0) return SFFG_OK;
  if (!pts) return fail(SFFG_ERR_ARG, "sffg_index_add_multi: null points");
  int rc;
  sffg_index *lead = idx[0];   // one staging buffer, one upload, one synchronisation for all indices
  for (int i = 0; i < n_idx; ++i)
    if ((rc = index_busy(idx[i], "sffg_index_add_multi")) != SFFG_OK) return rc;
  cudaStream_t st = lead->stream.get();
  const size_t bytes = (size_t)total * dim * sizeof(float);
  rc = lead->stage.reserve(bytes);
  if (rc != SFFG_OK) return rc;
  // (small batches: the whole staging area holds the rows)
  SFFG_CUDA(upload_async(lead->stage.p, pts, bytes, bytes <= kSmallBytes ? lead->h_small.get() : nullptr, st));
  int64_t off = 0;
  for (int i = 0; i < n_idx; ++i) {
    if (n_per[i] == 0) continue;
    rc = sffg_index_add_device(idx[i], (const float *)lead->stage.p + off * dim, n_per[i], st);
    if (rc != SFFG_OK) return rc;
    off += n_per[i];
  }
  // the appends ran on the lead's stream: later work on the other indices' own streams is ordered behind them
  SFFG_CUDA(cudaEventRecord(lead->add_ev.get(), st));
  for (int i = 0; i < n_idx; ++i)
    if (idx[i] != lead && n_per[i] > 0) SFFG_CUDA(cudaStreamWaitEvent(idx[i]->stream.get(), lead->add_ev.get(), 0));
  sffg_index::Pending p{};
  p.kind = 3;   // (the staging area of the lead is in use until sffg_index_end)
  lead->pend = p;
  return SFFG_OK;
}

int sffg_index_add_multi(sffg_index *const *idx, const int64_t *n_per, int n_idx, const float *pts) {
  const int rc = sffg_index_add_multi_begin(idx, n_per, n_idx, pts);
  if (rc != SFFG_OK) return rc;
  return idx[0]->pend.kind == 3 ? sffg_index_end(idx[0]) : SFFG_OK;
}

static IndexDev index_view(const sffg_index *idx) {
  return IndexDev{idx->d_coords.get(), idx->cap, idx->n, idx->dim, idx->d_amax.get()};
}

static SortedDev sorted_view(const sffg_index *idx) {
  SortedDev sv;
  sv.coords = (const float *)idx->s_coords.p;
  sv.ids = (const int *)idx->s_ids.p;
  sv.bb = (const float *)idx->s_bb.p;
  sv.cap_s = idx->s_cap;
  sv.nblk_cap = idx->s_nblk_cap;
  sv.nsb_cap = idx->s_nblk_cap / 32 + 2;
  sv.sbb = sv.bb + (size_t)idx->s_nblk_cap * 2 * (idx->dim == 6 ? 3 : 2);
  sv.n_sorted = (int)idx->n_sorted;
  sv.nblk = (int)((idx->n_sorted + 31) / 32);
  sv.amax = idx->d_amax.get();
  sv.bounds = (const int *)idx->s_bounds.p;
  return sv;
}

constexpr int64_t kSortMinNodes = 8192;   // below this the exhaustive scan is already latency-bound

// (re)builds the Morton-sorted view when the index is large and too many nodes were appended since the last build
static int ensure_sorted(sffg_index *idx, cudaStream_t st) {
  if (!idx->pruning || idx->n < kSortMinNodes) return SFFG_OK;
  const int64_t tail = idx->n - idx->n_sorted;
  if (idx->n_sorted > 0 && tail <= std::max<int64_t>(2048, idx->n_sorted / 4)) return SFFG_OK;
  const int n = (int)idx->n;
  const int lin = idx->dim == 6 ? 3 : 2;
  if (n > idx->s_cap) {
    idx->s_cap = ((int64_t)n * 3 / 2 + 31) / 32 * 32 + 128;
    idx->s_nblk_cap = idx->s_cap / 32 + 32;
    idx->s_coords.release();
    idx->s_ids.release();
    idx->s_bb.release();
    idx->s_keys.release();
    idx->s_vals.release();
  }
  int rc = idx->s_coords.reserve((size_t)idx->s_cap * idx->dim * 4);
  if (rc == SFFG_OK) rc = idx->s_ids.reserve((size_t)idx->s_cap * 4);
  // block boxes followed by superblock boxes (one per 32 blocks)
  if (rc == SFFG_OK) rc = idx->s_bb.reserve(((size_t)idx->s_nblk_cap + (size_t)(idx->s_nblk_cap / 32 + 2)) * 2 * lin * 4);
  if (rc == SFFG_OK) rc = idx->s_keys.reserve((size_t)idx->s_cap * 8);
  if (rc == SFFG_OK) rc = idx->s_vals.reserve((size_t)idx->s_cap * 8);
  if (rc == SFFG_OK) rc = idx->s_temp.reserve(sorted_build_temp_bytes((int)idx->s_cap));
  if (rc == SFFG_OK) rc = idx->s_bounds.reserve(64);
  if (rc != SFFG_OK) return rc;
  SortedBuildBuffers b;
  b.bounds = (int *)idx->s_bounds.p;
  b.keys_in = (unsigned *)idx->s_keys.p;
  b.keys_out = b.keys_in + idx->s_cap;
  b.vals_in = (unsigned *)idx->s_vals.p;
  b.vals_out = b.vals_in + idx->s_cap;
  b.temp = idx->s_temp.p;
  b.temp_bytes = idx->s_temp.cap;
  b.s_coords = (float *)idx->s_coords.p;
  b.cap_s = idx->s_cap;
  b.s_ids = (int *)idx->s_ids.p;
  b.bb = (float *)idx->s_bb.p;
  b.nblk_cap = idx->s_nblk_cap;
  b.nsb_cap = idx->s_nblk_cap / 32 + 2;
  b.sbb = b.bb + (size_t)idx->s_nblk_cap * 2 * lin;
  const IndexDev v = index_view(idx);
  SFFG_CUDA(launch_sorted_build(v, n, b, st));
  idx->n_sorted = n;
  return SFFG_OK;
}

static int knn_rows_device(sffg_index *idx, const float *d_queries, int64_t nq, int k, const RowDests &out, cudaStream_t st) {
  const IndexDev v = index_view(idx);
  int rc = ensure_sorted(idx, st);
  if (rc != SFFG_OK) return rc;
  if (idx->n_sorted > 0) {
    const SortedDev sv = sorted_view(idx);
    const PrunedPlan plan = plan_pruned(nq, sv, idx->n - idx->n_sorted, g_rt.sm_count);
    rc = idx->scratch.reserve(pruned_scratch_bytes(plan, nq, k));
    if (rc != SFFG_OK) return rc;
    SFFG_CUDA(launch_knn_pruned(v, sv, d_queries, nq, k, out, idx->scratch.p, plan, st));
    return SFFG_OK;
  }
  KnnPlan plan = plan_knn(nq, idx->n, g_rt.sm_count);
  rc = idx->scratch.reserve(knn_scratch_bytes(plan, nq, k));
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(launch_knn(v, d_queries, nq, k, out, idx->scratch.p, plan, st));
  return SFFG_OK;
}

int sffg_knn_device(sffg_index *idx, const float *d_queries, int64_t nq, int k, int32_t *d_ids_out, float *d_d2_out,
                    void *stream) {
  if (!idx || nq < 0 || k < 1 || k > SFFG_MAX_K || (nq > 0 && (!d_queries || !d_ids_out || !d_d2_out)))
    return fail(SFFG_ERR_ARG, "sffg_knn_device: bad arguments (1 <= k <= 128)");
  if (nq == 0) return SFFG_OK;
  return knn_rows_device(idx, d_queries, nq, k, single_dest(d_ids_out, d_d2_out), (cudaStream_t)stream);
}

int sffg_knn_gather_device(sffg_index *idx, const float *d_queries, int64_t nq, int k, int32_t *const *d_ids_dests,
                           float *const *d_d2_dests, int n_dests, void *stream) {
  if (!idx || nq < 0 || k < 1 || k > SFFG_MAX_K || !d_ids_dests || !d_d2_dests || n_dests < 1 || n_dests > kMaxRowDests ||
      (nq > 0 && !d_queries))
    return fail(SFFG_ERR_ARG, "sffg_knn_gather_device: bad arguments (1 <= k <= 128, 1..8 destinations)");
  RowDests out{};
  out.n = n_dests;
  for (int r = 0; r < n_dests; ++r) {
    if (!d_ids_dests[r] || !d_d2_dests[r]) return fail(SFFG_ERR_ARG, "sffg_knn_gather_device: null destination");
    out.ids[r] = d_ids_dests[r];
    out.d2[r] = d_d2_dests[r];
  }
  if (nq == 0) return SFFG_OK;
  return knn_rows_device(idx, d_queries, nq, k, out, (cudaStream_t)stream);
}

int sffg_knn(sffg_index *idx, const float *queries, int64_t nq, int k, int32_t *ids_out, float *d2_out) {
  if (!idx || nq < 0 || k < 1 || k > SFFG_MAX_K || (nq > 0 && (!queries || !ids_out || !d2_out)))
    return fail(SFFG_ERR_ARG, "sffg_knn: bad arguments (1 <= k <= 128)");
  if (nq == 0) return SFFG_OK;
  int rc = index_busy(idx, "sffg_knn");
  if (rc != SFFG_OK) return rc;
  const size_t qbytes = (size_t)nq * idx->dim * 4, obytes = (size_t)nq * k * 4;
  if (qbytes <= IndexStaging::kQueryBytes && 2 * obytes <= IndexStaging::kKnnOutBytes) {
    // planner-sized call: queries and results live in pinned mapped memory, one synchronisation
    const IndexStaging h = idx->staging();
    std::memcpy(h.queries(), queries, qbytes);
    int32_t *h_ids = h.knn_ids();
    float *h_d2 = h.knn_d2(obytes);
    rc = sffg_knn_device(idx, reinterpret_cast<const float *>(h.queries()), nq, k, h_ids, h_d2, idx->stream.get());
    if (rc != SFFG_OK) return rc;
    SFFG_CUDA(cudaStreamSynchronize(idx->stream.get()));
    std::memcpy(ids_out, h_ids, obytes);
    std::memcpy(d2_out, h_d2, obytes);
    return SFFG_OK;
  }
  const int64_t chunk = 1 << 17;
  for (int64_t off = 0; off < nq; off += chunk) {
    const int64_t cnt = std::min(chunk, nq - off);
    rc = idx->q.reserve((size_t)cnt * idx->dim * 4);
    if (rc == SFFG_OK) rc = idx->ids.reserve((size_t)cnt * k * 4);
    if (rc == SFFG_OK) rc = idx->d2.reserve((size_t)cnt * k * 4);
    if (rc != SFFG_OK) return rc;
    SFFG_CUDA(cudaMemcpyAsync(idx->q.p, queries + off * idx->dim, (size_t)cnt * idx->dim * 4, cudaMemcpyHostToDevice, idx->stream.get()));
    rc = sffg_knn_device(idx, (const float *)idx->q.p, cnt, k, (int32_t *)idx->ids.p, (float *)idx->d2.p, idx->stream.get());
    if (rc != SFFG_OK) return rc;
    SFFG_CUDA(cudaMemcpyAsync(ids_out + off * k, idx->ids.p, (size_t)cnt * k * 4, cudaMemcpyDeviceToHost, idx->stream.get()));
    SFFG_CUDA(cudaMemcpyAsync(d2_out + off * k, idx->d2.p, (size_t)cnt * k * 4, cudaMemcpyDeviceToHost, idx->stream.get()));
    SFFG_CUDA(cudaStreamSynchronize(idx->stream.get()));
  }
  return SFFG_OK;
}

int sffg_knn_multi_begin(sffg_index *const *idx, const int64_t *nq_per, int n_idx, const float *queries, int k, int32_t *ids_out,
                         float *d2_out) {
  if (!idx || !nq_per || n_idx < 1 || k < 1 || k > SFFG_MAX_K) return fail(SFFG_ERR_ARG, "sffg_knn_multi: bad arguments");
  int64_t total = 0;
  const int dim = idx[0] ? idx[0]->dim : 0;
  for (int i = 0; i < n_idx; ++i) {
    if (!idx[i] || idx[i]->dim != dim || nq_per[i] < 0) return fail(SFFG_ERR_ARG, "sffg_knn_multi: bad index / count");
    total += nq_per[i];
  }
  if (total == 0) return SFFG_OK;
  if (!queries || !ids_out || !d2_out) return fail(SFFG_ERR_ARG, "sffg_knn_multi: null buffers");
  int rc;
  sffg_index *lead = idx[0];   // its stream and staging carry the whole call
  for (int i = 0; i < n_idx; ++i)
    if ((rc = index_busy(idx[i], "sffg_knn_multi")) != SFFG_OK) return rc;
  cudaStream_t st = lead->stream.get();
  const size_t qbytes = (size_t)total * dim * 4, obytes = (size_t)total * k * 4;
  const bool small = qbytes <= IndexStaging::kQueryBytes && 2 * obytes <= IndexStaging::kKnnOutBytes;
  const IndexStaging h = lead->staging();
  rc = lead->q.reserve(qbytes);
  if (rc == SFFG_OK) rc = lead->ids.reserve(obytes);
  if (rc == SFFG_OK) rc = lead->d2.reserve(obytes);
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(upload_async(lead->q.p, queries, qbytes, small ? h.queries() : nullptr, st));
  // fork: every index searches on its own stream once the queries have arrived; join: the lead stream waits for all
  SFFG_CUDA(cudaEventRecord(lead->ev.get(), st));
  int64_t off = 0;
  for (int i = 0; i < n_idx; ++i) {
    if (nq_per[i] == 0) continue;
    cudaStream_t si = idx[i] == lead ? st : idx[i]->stream.get();
    if (si != st) SFFG_CUDA(cudaStreamWaitEvent(si, lead->ev.get(), 0));
    rc = sffg_knn_device(idx[i], (const float *)lead->q.p + off * dim, nq_per[i], k, (int32_t *)lead->ids.p + off * k,
                         (float *)lead->d2.p + off * k, si);
    if (rc != SFFG_OK) return rc;
    if (si != st) {
      SFFG_CUDA(cudaEventRecord(idx[i]->ev.get(), si));
      SFFG_CUDA(cudaStreamWaitEvent(st, idx[i]->ev.get(), 0));
    }
    off += nq_per[i];
  }
  sffg_index::Pending p{};
  p.kind = 1;
  if (small) {
    SFFG_CUDA(cudaMemcpyAsync(h.knn_ids(), lead->ids.p, obytes, cudaMemcpyDeviceToHost, st));
    SFFG_CUDA(cudaMemcpyAsync(h.knn_d2(obytes), lead->d2.p, obytes, cudaMemcpyDeviceToHost, st));
    p.copy[0] = {ids_out, h.knn_ids(), obytes};
    p.copy[1] = {d2_out, h.knn_d2(obytes), obytes};
    p.n_copy = 2;
  } else {
    SFFG_CUDA(cudaMemcpyAsync(ids_out, lead->ids.p, obytes, cudaMemcpyDeviceToHost, st));
    SFFG_CUDA(cudaMemcpyAsync(d2_out, lead->d2.p, obytes, cudaMemcpyDeviceToHost, st));
  }
  lead->pend = p;
  return SFFG_OK;
}

int sffg_knn_multi(sffg_index *const *idx, const int64_t *nq_per, int n_idx, const float *queries, int k, int32_t *ids_out,
                   float *d2_out) {
  const int rc = sffg_knn_multi_begin(idx, nq_per, n_idx, queries, k, ids_out, d2_out);
  if (rc != SFFG_OK) return rc;
  return idx[0]->pend.kind == 1 ? sffg_index_end(idx[0]) : SFFG_OK;
}

// fill and per-row sort of a radius call once idx->offsets holds the row offsets: the sorted rows go to ids_dst / d2_dst
static int radius_fill_sort(sffg_index *idx, bool pruned, int64_t nq, float r2, int32_t *ids_dst, float *d2_dst) {
  cudaStream_t st = idx->stream.get();
  const IndexDev v = index_view(idx);
  const float *q = (const float *)idx->q.p;
  const int64_t *offs = (const int64_t *)idx->offsets.p;
  int32_t *cursor = (int32_t *)idx->cursor.p;
  unsigned long long *keys = (unsigned long long *)idx->keys.p;
  SFFG_CUDA(cudaMemsetAsync(cursor, 0, (size_t)nq * 4, st));
  if (pruned) SFFG_CUDA(launch_radius_fill_pruned(v, sorted_view(idx), q, nq, r2, offs, cursor, keys, g_rt.sm_count, st));
  else SFFG_CUDA(launch_radius_fill(v, q, nq, r2, offs, cursor, keys, plan_knn(nq, idx->n, g_rt.sm_count), st));
  SFFG_CUDA(launch_radius_sort(keys, offs, (const int32_t *)idx->counts.p, nq, ids_dst, d2_dst, st));
  return SFFG_OK;
}

// second half of a radius call once the counts are on the host: exclusive scan, fill, per-row sort, download
static int radius_fill_from_host_counts(sffg_index *idx, const sffg_index::Pending &c, int64_t total) {
  cudaStream_t st = idx->stream.get();
  const IndexStaging h = idx->staging();
  const size_t cbytes = (size_t)c.nq * 4;
  std::vector<int64_t> offs((size_t)c.nq);
  int64_t run = 0;
  for (int64_t i = 0; i < c.nq; ++i) {
    offs[(size_t)i] = run;
    run += c.counts_out[i];
  }
  int rc = idx->offsets.reserve((size_t)c.nq * 8);
  if (rc == SFFG_OK) rc = idx->cursor.reserve(cbytes);
  if (rc == SFFG_OK) rc = idx->keys.reserve((size_t)total * 8);
  if (rc == SFFG_OK) rc = idx->ids.reserve((size_t)total * 4);
  if (rc == SFFG_OK) rc = idx->d2.reserve((size_t)total * 4);
  if (rc != SFFG_OK) return rc;
  // two-sync staging: the row offsets in the query part (free again), the rows without a head
  const bool small_out = c.small && (size_t)c.nq * 8 <= IndexStaging::kQueryBytes && (size_t)total * 8 <= IndexStaging::kRowsBytes;
  SFFG_CUDA(upload_async(idx->offsets.p, offs.data(), (size_t)c.nq * 8, small_out ? h.queries() : nullptr, st));
  rc = radius_fill_sort(idx, c.pruned, c.nq, c.r2, (int32_t *)idx->ids.p, (float *)idx->d2.p);
  if (rc != SFFG_OK) return rc;
  int32_t *ids_dst = small_out ? h.rows_ids(0) : c.ids_out;
  float *d2_dst = small_out ? h.rows_d2(0, total) : c.d2_out;
  SFFG_CUDA(cudaMemcpyAsync(ids_dst, idx->ids.p, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
  SFFG_CUDA(cudaMemcpyAsync(d2_dst, idx->d2.p, (size_t)total * 4, cudaMemcpyDeviceToHost, st));
  SFFG_CUDA(cudaStreamSynchronize(st));
  if (small_out) {
    std::memcpy(c.ids_out, ids_dst, (size_t)total * 4);
    std::memcpy(c.d2_out, d2_dst, (size_t)total * 4);
  }
  return SFFG_OK;
}

constexpr int64_t kFusedRadiusMaxNodes = 32768;   // above this the pruned count / fill kernels win over one exhaustive pass

static int radius_begin_impl(sffg_index *idx, const float *queries, int64_t nq, float r2, int32_t *counts_out, int32_t *ids_out,
                             float *d2_out, int64_t capacity, int64_t *total_out, bool allow_fused) {
  if (!idx || nq < 0 || (nq > 0 && (!queries || !counts_out)) || (ids_out && !d2_out))
    return fail(SFFG_ERR_ARG, "sffg_radius: bad arguments");
  if (total_out) *total_out = 0;
  if (nq == 0) return SFFG_OK;
  int rc = index_busy(idx, "sffg_radius");
  if (rc != SFFG_OK) return rc;
  cudaStream_t st = idx->stream.get();
  const IndexDev v = index_view(idx);
  const IndexStaging h = idx->staging();
  const size_t qbytes = (size_t)nq * idx->dim * 4, cbytes = (size_t)nq * 4;
  // planner-sized calls stage through pinned memory so that every copy is an asynchronous DMA
  const bool small = qbytes <= IndexStaging::kQueryBytes && cbytes <= IndexStaging::kCountBytes;
  sffg_index::Pending c{};
  c.kind = 2;
  c.nq = nq;
  c.capacity = capacity;
  c.r2 = r2;
  c.queries = queries;
  c.counts_out = counts_out;
  c.ids_out = ids_out;
  c.d2_out = d2_out;
  c.total_out = total_out;
  c.small = small;
  if (small) c.copy[c.n_copy++] = {counts_out, h.counts(), cbytes};
  const size_t rowoff_bytes = (size_t)nq * sizeof(int64_t);
  if (allow_fused && small && ids_out && capacity > 0 && idx->n <= kFusedRadiusMaxNodes && qbytes <= IndexStaging::kFlagAt &&
      rowoff_bytes + 64 <= IndexStaging::kRowsBytes / 2) {
    // planner-sized search on a small index: ONE kernel (block per query) that reads the queries from and writes counts,
    // row offsets and sorted rows to pinned mapped memory -- one stream operation besides zeroing the row allocator, one
    // host synchronisation.  Staging: [queries | flag] [counts] [row offsets | ids | d2].
    std::memcpy(h.queries(), queries, qbytes);
    *h.fused_flag() = 0;
    c.fused = true;
    c.cap1 = IndexStaging::rows_cap(rowoff_bytes);
    SFFG_CUDA(cudaMemsetAsync(idx->d_total.get(), 0, sizeof(unsigned long long), st));
    SFFG_CUDA(launch_radius_fused(v, reinterpret_cast<const float *>(h.queries()), nq, r2, c.cap1, h.counts(), h.rows_head(),
                                  h.rows_ids(rowoff_bytes), h.rows_d2(rowoff_bytes, c.cap1), idx->d_total.get(), h.fused_flag(), st));
    idx->pend = c;
    return SFFG_OK;
  }
  rc = idx->q.reserve(qbytes);
  if (rc == SFFG_OK) rc = idx->counts.reserve(cbytes);
  if (rc != SFFG_OK) return rc;
  SFFG_CUDA(upload_async(idx->q.p, queries, qbytes, small ? h.queries() : nullptr, st));
  SFFG_CUDA(cudaMemsetAsync(idx->counts.p, 0, cbytes, st));
  rc = ensure_sorted(idx, st);
  if (rc != SFFG_OK) return rc;
  c.pruned = idx->n_sorted > 0;
  const float *q = (const float *)idx->q.p;
  if (c.pruned) SFFG_CUDA(launch_radius_count_pruned(v, sorted_view(idx), q, nq, r2, (int32_t *)idx->counts.p, g_rt.sm_count, st));
  else SFFG_CUDA(launch_radius_count(v, q, nq, r2, (int32_t *)idx->counts.p, plan_knn(nq, idx->n, g_rt.sm_count), st));
  SFFG_CUDA(cudaMemcpyAsync(small ? (void *)h.counts() : (void *)counts_out, idx->counts.p, cbytes, cudaMemcpyDeviceToHost, st));
  // Planner-sized call with result buffers: the exclusive scan of the counts runs on the device, so that count, scan, fill
  // and sort are enqueued back to back and the call costs ONE host synchronisation.  The rows land in pinned mapped
  // memory ([total][ids][d2] in the rows part of the staging area); when they do not fit there, or not into the
  // caller's capacity, the kernels after the scan do nothing and sffg_index_end takes the two-synchronisation route.
  c.cap1 = std::min<int64_t>(capacity, IndexStaging::rows_cap(sizeof(int64_t)));
  c.one_sync = small && ids_out && c.cap1 > 0;
  if (c.one_sync) {
    rc = idx->offsets.reserve((size_t)nq * 8);
    if (rc == SFFG_OK) rc = idx->cursor.reserve(cbytes);
    if (rc == SFFG_OK) rc = idx->keys.reserve((size_t)c.cap1 * 8);
    if (rc != SFFG_OK) return rc;
    *h.rows_head() = -1;
    SFFG_CUDA(launch_radius_offsets((const int32_t *)idx->counts.p, nq, c.cap1, (int64_t *)idx->offsets.p, h.rows_head(), st));
    rc = radius_fill_sort(idx, c.pruned, nq, r2, h.rows_ids(sizeof(int64_t)), h.rows_d2(sizeof(int64_t), c.cap1));
    if (rc != SFFG_OK) return rc;
  }
  idx->pend = c;
  return SFFG_OK;
}

int sffg_radius_begin(sffg_index *idx, const float *queries, int64_t nq, float r2, int32_t *counts_out, int32_t *ids_out,
                      float *d2_out, int64_t capacity, int64_t *total_out) {
  return radius_begin_impl(idx, queries, nq, r2, counts_out, ids_out, d2_out, capacity, total_out, true);
}

// completes the asynchronous call pending on this index (no-op when none is)
int sffg_index_end(sffg_index *idx) {
  if (!idx) return fail(SFFG_ERR_ARG, "sffg_index_end: null index");
  if (idx->pend.kind == 0) return SFFG_OK;
  const sffg_index::Pending c = idx->pend;
  idx->pend.kind = 0;
  SFFG_CUDA(cudaStreamSynchronize(idx->stream.get()));
  for (int i = 0; i < c.n_copy; ++i) std::memcpy(c.copy[i].dst, c.copy[i].src, c.copy[i].bytes);
  if (c.kind != 2) return SFFG_OK;
  const IndexStaging h = idx->staging();
  int64_t total = 0;
  if (c.fused) {
    const int flag = *reinterpret_cast<const volatile int *>(h.fused_flag());
    for (int64_t i = 0; i < c.nq; ++i) total += c.counts_out[i];
    if (c.total_out) *c.total_out = total;
    if (total == 0) return SFFG_OK;
    if (c.capacity < total)
      return fail(SFFG_ERR_CAPACITY, "sffg_radius: result buffers hold " + std::to_string(c.capacity) + " entries, " +
                                         std::to_string(total) + " needed");
    if (flag) {   // a row longer than the kernel's shared buffer, or rows beyond the staging area: the general path
      const int rc = radius_begin_impl(idx, c.queries, c.nq, c.r2, c.counts_out, c.ids_out, c.d2_out, c.capacity, c.total_out, false);
      return rc != SFFG_OK ? rc : sffg_index_end(idx);
    }
    const size_t rowoff_bytes = (size_t)c.nq * sizeof(int64_t);
    const int64_t *h_rowoff = h.rows_head();
    const int32_t *h_ids = h.rows_ids(rowoff_bytes);
    const float *h_d2 = h.rows_d2(rowoff_bytes, c.cap1);
    int64_t run = 0;
    for (int64_t i = 0; i < c.nq; ++i) {   // rows were packed in the order the blocks finished: back into query order
      const int64_t n_i = c.counts_out[i];
      if (n_i) {
        std::memcpy(c.ids_out + run, h_ids + h_rowoff[i], (size_t)n_i * 4);
        std::memcpy(c.d2_out + run, h_d2 + h_rowoff[i], (size_t)n_i * 4);
      }
      run += n_i;
    }
    return SFFG_OK;
  }
  if (c.one_sync) {
    total = *h.rows_head();
    if (total < 0) return fail(SFFG_ERR_INTERNAL, "sffg_radius: the device-side scan did not report a total");
    if (c.total_out) *c.total_out = total;
    if (total == 0) return SFFG_OK;
    if (total <= c.cap1) {
      std::memcpy(c.ids_out, h.rows_ids(sizeof(int64_t)), (size_t)total * 4);
      std::memcpy(c.d2_out, h.rows_d2(sizeof(int64_t), c.cap1), (size_t)total * 4);
      return SFFG_OK;
    }
  } else {
    for (int64_t i = 0; i < c.nq; ++i) total += c.counts_out[i];
    if (c.total_out) *c.total_out = total;
    if (!c.ids_out || total == 0) return SFFG_OK;
  }
  if (c.capacity < total)
    return fail(SFFG_ERR_CAPACITY, "sffg_radius: result buffers hold " + std::to_string(c.capacity) + " entries, " +
                                       std::to_string(total) + " needed");
  return radius_fill_from_host_counts(idx, c, total);
}

int sffg_radius(sffg_index *idx, const float *queries, int64_t nq, float r2, int32_t *counts_out, int32_t *ids_out,
                float *d2_out, int64_t capacity, int64_t *total_out) {
  const int rc = sffg_radius_begin(idx, queries, nq, r2, counts_out, ids_out, d2_out, capacity, total_out);
  if (rc != SFFG_OK) return rc;
  return idx->pend.kind == 2 ? sffg_index_end(idx) : SFFG_OK;
}

}  // extern "C"
