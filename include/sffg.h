/*
 * sffg.h -- C ABI of the B200 collision-and-neighbour engine for the Space-Filling Forest* planner.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types, never throws.  Every entry
 * point names the reference interface it replaces (paths relative to the reference repository root).
 * The library (libsffg.so) is CUDA-only: there is NO CPU fallback; every compute call returns
 * SFFG_ERR_NO_DEVICE when no sm_100 device is usable.
 *
 * Conventions
 *   - all functions return an int status (SFFG_OK == 0) unless stated; sffg_last_error() gives the text
 *   - triangle soups are double [n][9] = p1.xyz p2.xyz p3.xyz, already offset+scaled the way
 *     Obstacle<T>::addPoint does it (src/environment.h:198-211)
 *   - poses are [n][6] = x y z yaw pitch roll (Point<T>, src/primitives.h:86-102), angles in radians; any finite
 *     angle is accepted and the verdict is exact for it (no range reduction by the caller: a double angle of 1000 rad is
 *     judged at that angle, not at its float neighbour)
 *   - "host" calls take caller-owned host pointers and block until results are in the output arrays
 *   - "_device" calls take device pointers + a cudaStream_t (as void*), enqueue, and return immediately
 *   - one host thread per handle at a time
 */
#ifndef SFFG_H_
#define SFFG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SFFG_API __attribute__((visibility("default")))
#else
#define SFFG_API
#endif

#define SFFG_OK 0
#define SFFG_ERR_NO_DEVICE 1    /* no CUDA device / wrong architecture: the engine refuses to run            */
#define SFFG_ERR_CUDA 2         /* a CUDA runtime call failed (text in sffg_last_error)                        */
#define SFFG_ERR_ARG 3          /* bad argument (null pointer, negative size, dim not 2 or 6, k out of range)  */
#define SFFG_ERR_IO 4           /* mesh file unreadable / malformed                                            */
#define SFFG_ERR_CAPACITY 5     /* caller-provided result buffer too small (needed size is reported)           */
#define SFFG_ERR_DOMAIN 6       /* reserved (no longer returned: the metric is exact for every float angle)    */
#define SFFG_ERR_INTERNAL 7     /* traversal stack overflow or similar -- a bug, never a silent wrong answer   */

#define SFFG_ROT_REFERENCE 0    /* interior edge samples carry identity rotation (src/problemStruct.h:157-163) */
#define SFFG_ROT_INTERPOLATE 1  /* opt-in: angles interpolated along the wrapped difference                    */

#define SFFG_MAX_K 128

typedef struct sffg_env sffg_env;       /* obstacle BVH + robot mesh resident on one GPU  (Environment<T>)     */
typedef struct sffg_index sffg_index;   /* append-only node set resident on one GPU        (flann::Index)      */

/* ---- threads and streams ----------------------------------------------------------------------------------
 * A handle (sffg_env, sffg_index) may be used from one host thread at a time; different handles may be used from
 * different threads.  Host-pointer calls block until their results are in the caller's buffers.  The *_device calls
 * only enqueue work on the caller's stream.  Launches of ONE environment share launch state (a ring of work counters,
 * scratch for small edge batches), so the library keeps them in order across streams: a *_device call on another stream
 * than the previous call of that environment first waits (on the device, cudaStreamWaitEvent) for that previous launch.
 * Use one environment per stream for launches that should overlap.  An sffg_index is bound the same way to the stream
 * of its last call for as long as work is in flight (its scratch buffers are reused by the next search).              */

/* ---- library ------------------------------------------------------------------------------------------ */
SFFG_API int sffg_version(void);
SFFG_API const char *sffg_last_error(void);              /* thread-local, valid until the next call on this thread      */
SFFG_API int sffg_init(int device);                      /* bind this process/thread to a GPU; checks sm_100            */
SFFG_API int sffg_device_count(void);

/* ---- meshes: Obstacle<T>::ParseOBJFile / ParseMapFile / addPoint / addFacet, src/environment.h:125-223 -- */
/* is_obj != 0: OBJ (every token starting with 'v' is a vertex, only the first 3 indices of an 'f' line are
 * used, 'o' never changes the index offset); is_obj == 0: 2-D ".tri" map (x1 y1 x2 y2 x3 y3, z = 0).
 * vertex = (file value + position[i]) * scale.  *tris_out is malloc'ed by the library: free with sffg_free.
 * bbox_out (optional) = minX maxX minY maxY minZ maxZ over all parsed vertices (Obstacle::localRange).       */
#define SFFG_MESH_TRI 0        /* 2-D ".tri" map                                                                     */
#define SFFG_MESH_OBJ 1        /* OBJ exactly as the reference reads it (parity mode)                                 */
#define SFFG_MESH_OBJ_FIXED 2  /* opt-in: only "v" lines are vertices, polygons are fan-triangulated (a quad gives two
                                * triangles), negative indices are relative -- what the files mean, not what the
                                * reference loads; leaves parity with the reference's triangle soup                   */
SFFG_API int sffg_mesh_load(const char *path, int is_obj, const double position[3], double scale,
                   double **tris_out, int64_t *n_tris_out, double bbox_out[6]);
SFFG_API void sffg_free(void *p);

/* ---- environment: RAPID_model::{BeginModel,AddTri,EndModel} (call sites src/environment.h:102-114,:222) -- */
/* The obstacle soup is the union of all Obstacles (the reference ORs over them, src/environment.h:312-314;
 * all sit at identity).  n_obst == 0 reproduces HasMap == false: nothing ever collides (:307-309).           */
SFFG_API int sffg_env_create(const double *obst_tris, int64_t n_obst, const double *robot_tris, int64_t n_robot,
                    sffg_env **out);
SFFG_API int sffg_env_destroy(sffg_env *env);

/* where the obstacle hierarchy is built (RAPID builds its OBB tree on the host at EndModel(), src/environment.h:114):
 * HOST = binned-SAH builder on the CPU (best traversal, ~1 us per triangle); DEVICE = Morton-ordered builder on the GPU
 * (a few ms for millions of triangles: large maps, obstacles that move every frame); AUTO = HOST below 2^18 triangles.
 * Verdicts do not depend on the builder -- both hierarchies are conservative and every surviving pair is tested exactly. */
#define SFFG_BUILD_AUTO 0
#define SFFG_BUILD_HOST 1
#define SFFG_BUILD_DEVICE 2
SFFG_API int sffg_env_create_ex(const double *obst_tris, int64_t n_obst, const double *robot_tris, int64_t n_robot,
                       int build_mode, sffg_env **out);
/* replaces the obstacle soup of an existing environment (moving / re-scanned obstacles; the reference would have to
 * delete and re-create its Obstacle objects, src/main.cpp:254): rebuilds hierarchy, triangle arrays and clearance grid,
 * keeps robot, streams, staging buffers and counters.  Blocks until the device is idle, then until the rebuild is done. */
SFFG_API int sffg_env_set_obstacles(sffg_env *env, const double *obst_tris, int64_t n_obst, int build_mode);
/* the same n_obst triangles in the same order, at new positions (rigid motion or deformation between frames): the
 * hierarchy keeps its topology and only the triangle arrays, every slot box (bottom-up, outward rounded), the top cut,
 * the root box and the clearance grid are recomputed on the GPU -- several times cheaper than a rebuild.  Verdicts stay
 * exact whatever the motion (boxes are refitted conservatively, every surviving pair is still tested exactly); only the
 * culling power degrades as the soup drifts away from the shape the topology was built for -- rebuild from time to time.
 * SFFG_ERR_ARG when the triangle count differs from the current set.                                               */
SFFG_API int sffg_env_refit_obstacles(sffg_env *env, const double *obst_tris, int64_t n_obst);

typedef struct {
  int64_t n_obst_tris, n_robot_tris;
  int64_t n_nodes;          /* 8-wide BVH nodes                                                               */
  int32_t depth;            /* levels of the wide BVH                                                         */
  int64_t device_bytes;     /* HBM held by this environment                                                   */
  double build_ms;          /* host BVH build + upload + clearance grid                                       */
  int64_t grid_cells;       /* cells of the free-space (clearance) grid, 0 when disabled                      */
  double grid_cell_size;
  int32_t built_on_device;  /* 1 if the hierarchy came from the GPU builder                                   */
} sffg_env_info_t;
SFFG_API int sffg_env_info(const sffg_env *env, sffg_env_info_t *out);

/* ---- pose verdicts: Environment<T>::Collide(Point<T>), src/environment.h:306-316
 *      = RAPID_Collide(I, 0, obstacle, R(pose), T(pose), robot) != 0 contacts, :269-276 ---------------------- */
SFFG_API int sffg_collide_poses_f32(sffg_env *env, const float *poses, int64_t n, uint8_t *verdict_out);
SFFG_API int sffg_collide_poses_f64(sffg_env *env, const double *poses, int64_t n, uint8_t *verdict_out);
/* RAPID_Collide's own argument form: rt = [n][12] doubles, R2 row-major (9) then T2 (3).  Model 1 (the obstacle soup) sits
 * at identity -- the only placement the planner ever passes (eyeRotation and a zero vector, src/environment.h:89, :270,
 * :274).  This is what the RAPID.H shim forwards; the shim terminates the process (like the reference's own fatal paths,
 * src/main.cpp:427-433) when a caller hands RAPID_Collide a model 1 that is rotated or translated, because this engine
 * bakes the obstacle placement into the hierarchy at sffg_env_create. */
SFFG_API int sffg_collide_transforms_f64(sffg_env *env, const double *rt, int64_t n, uint8_t *verdict_out);
SFFG_API int sffg_collide_poses_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n,
                              uint8_t *d_verdict_out, void *stream);

/* ---- separation distance per pose (what PQP / FCL distance queries answer; no counterpart in the reference) -------
 * dist_out[i] = distance between the robot at poses[i] ([n][6] x y z yaw pitch roll, float or double as poses_are_f64
 * says) and the obstacle soup, capped at max_dist (> 0, +INFINITY allowed):
 *   - contact gives exactly 0: dist_out[i] == 0.0 exactly when sffg_collide_poses_* gives verdict 1 for the same pose in
 *     the same format (the same code decides both)
 *   - a free pose gets min(d, max_dist), d = minimum over all (obstacle triangle, robot triangle) pairs of their
 *     Euclidean distance in double precision, the robot placed by the pose's double transform (ZYX Euler,
 *     FillRotationMatrix, the transform of the exact contact stage).  A free pose never reports 0: where d evaluates to 0
 *     for a pair the contact test separated, the smallest positive double is reported
 *   - accuracy: |dist - d| <= 1e-9 * S, S = max(1, max |obstacle coordinate|, |T| + robot radius)
 *   - when d >= max_dist the output is max_dist exactly; with no obstacles every pose gets max_dist (+inf included)
 *   - points_out (optional, NULL allowed) [n][6]: a nearest point on the robot, then a nearest point on the obstacles,
 *     world frame; written when 0 < dist < max_dist, NaN otherwise
 *   - max_dist <= 0 or NaN, or a null pointer with n > 0: SFFG_ERR_ARG.  A traversal stack overflow raises
 *     SFFG_ERR_INTERNAL (at once for the host call, at sffg_env_sync_check for the _device call), never a wrong answer
 *   - streams and threads as for every other call (see above); the matrix pose form is not offered */
SFFG_API int sffg_distance_poses(sffg_env *env, const void *poses, int poses_are_f64, int64_t n, double max_dist,
                                 double *dist_out, double *points_out);
SFFG_API int sffg_distance_poses_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n, double max_dist,
                                        double *d_dist_out, double *d_points_out, void *stream);

/* ---- separation distance per edge: the clearance of the segments isPathFree checks ---------------------------------
 * The samples of edge e are exactly the poses sffg_check_edges tests for the same (start, end, sample_dist, rot_mode);
 * D(e, k) is what sffg_distance_poses returns for sample k as a double pose at the same max_dist (in reference mode the
 * sample's angles are 0).
 *   - dist_out[e] = minimum of D(e, k) over the samples of e, bit for bit.  So dist_out[e] == 0 exactly where
 *     sffg_check_edges reports free == 0; an edge without samples, and every edge when there are no obstacles, gets
 *     max_dist.  The end points are not samples (as in isPathFree): a path's clearance is the minimum of its edges'
 *     distances and sffg_distance_poses of its nodes
 *   - index_out (optional, NULL allowed): the first colliding sample (first_hit_out of sffg_check_edges) when dist == 0;
 *     the lowest k with D(e, k) == dist_out[e] when 0 < dist < max_dist; 0 otherwise
 *   - points_out (optional, NULL allowed) [m][6]: a nearest point on the robot at sample index_out[e], then a nearest
 *     point on the obstacles, world frame, as sffg_distance_poses gives them for that sample; NaN unless 0 < dist <
 *     max_dist.  Where pairs tie, any of the tied points may be reported
 *   - the argument errors of sffg_check_edges, and max_dist <= 0 or NaN: SFFG_ERR_ARG.  A traversal stack overflow raises
 *     SFFG_ERR_INTERNAL (at once for the host call, at sffg_env_sync_check for the _device call)
 *   - streams and threads as for every other call; no begin / end form and no counters */
SFFG_API int sffg_distance_edges(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist,
                                 int rot_mode, double max_dist, double *dist_out, int32_t *index_out, double *points_out);
SFFG_API int sffg_distance_edges_device(sffg_env *env, const double *d_starts, const double *d_ends, int64_t m,
                                        double sample_dist, int rot_mode, double max_dist, double *d_dist_out,
                                        int32_t *d_index_out, double *d_points_out, void *stream);

/* ---- continuous edge check: a certificate for the whole motion, not only for the samples isPathFree checks -----------
 * sffg_check_edges tests poses sample_dist apart and says nothing between them: a thin wall or a pole crossed between two
 * samples is missed.  This call certifies the motion itself by conservative advancement on the pose distance.
 *   - the motion of edge e, tau in [0, 1]: position x_k(tau) = s_k + tau * (f_k - s_k) (s = starts[e], f = ends[e]), each
 *     operation rounded to nearest, no FMA.  SFFG_ROT_REFERENCE: identity rotation for every tau, end points included (how
 *     isPathFree places its samples).  SFFG_ROT_INTERPOLATE: angles s_{3+k} + tau * wrap(f_{3+k} - s_{3+k}), wrap as in
 *     sffg_check_edges.  Every sample sffg_check_edges tests lies on this curve, up to rounding, for any sample_dist
 *   - margin = m > 0.  clear_out[e] = 1: every pose of the motion is at distance >= m / 2 from the obstacles, up to the
 *     accuracy of sffg_distance_poses (1e-9 S); in particular the whole motion is collision free.  t_out[e] = 1.0 and
 *     dist_out[e] = m then
 *   - clear_out[e] = 0: t_out[e] = tau* in [0, 1) where the distance of pose(tau*) is < m, every pose with tau < tau* is at
 *     distance >= m / 2 (same accuracy), and dist_out[e] is, bit for bit, what sffg_distance_poses returns for pose(tau*)
 *     as a double pose at max_dist = m (in reference mode its angles are 0).  So dist_out[e] == 0 exactly when
 *     sffg_collide_poses_f64 reports contact at pose(tau*)
 *   - a motion that comes within m / 2 of the obstacles is never clear, one that stays >= m away is always clear; in
 *     between either answer can come back, each certified as stated.  An edge with a non-finite coordinate (that the
 *     motion uses) is never clear: t = 0, dist = NaN.  With no obstacles every edge is clear
 *   - t_out and dist_out are optional (NULL allowed).  No points, no begin / end form, no counters
 *   - clear, t and dist do not depend on the batch size, the split of edges over warps, host chunking, the host or device
 *     form, the hierarchy builder or timing
 *   - work: at most 32 + 2 mu / m pose distance evaluations per edge, mu = |f_xyz - s_xyz| (reference mode) plus
 *     rho (|dyaw| + |dpitch| + |droll|) with wrapped differences (interpolate mode), rho = the robot's bounding radius
 *   - SFFG_ERR_ARG: the argument errors of sffg_check_edges (sample_dist aside); margin <= 0, NaN or infinite; margin <
 *     1e-6 max(1, max |obstacle coordinate|) (the coordinate rounded up to float).  A traversal stack overflow raises
 *     SFFG_ERR_INTERNAL (at once for the host call, at sffg_env_sync_check for the _device call), never a wrong answer
 *   - streams and threads as for every other call */
SFFG_API int sffg_sweep_edges(sffg_env *env, const double *starts, const double *ends, int64_t m, int rot_mode,
                              double margin, uint8_t *clear_out, double *t_out, double *dist_out);
SFFG_API int sffg_sweep_edges_device(sffg_env *env, const double *d_starts, const double *d_ends, int64_t m, int rot_mode,
                                     double margin, uint8_t *d_clear_out, double *d_t_out, double *d_dist_out, void *stream);

/* ---- multi-GPU (SURVEY 8e): pose batches are split over ranks, every rank needs all verdicts.  Instead of a separate
 * all-gather, the kernel stores verdict i to d_outs[r][i] for EVERY destination r: the local result buffer and the same
 * slice of every peer's buffer, mapped into this process through CUDA IPC -- the exchange rides on the kernel's own stores
 * over NVLink while it computes -- and the last CTA to finish publishes a completion epoch to every rank.  One process per
 * GPU:
 *   sffg_peer_buffer_create   cudaMalloc'ed (zeroed) buffer + its 64-byte IPC handle (ship it to the peers, e.g. with
 *                             torch.distributed.all_gather_object)
 *   sffg_peer_buffer_open     map a peer's buffer into this process; _close unmaps; _destroy frees an own buffer
 *   sffg_collide_poses_gather_device        as sffg_collide_poses_device with n_outs (1..8) destinations, 4-byte aligned
 *   sffg_collide_poses_gather_sync_device   the same with the handshake fused in.  d_flags[r] = rank r's array of 8 uint32 in a
 *                             peer buffer, d_done_counter = a zeroed local uint32.  Before touching the destinations the
 *                             kernel waits until every rank has published an epoch >= wait_epoch (0 = do not wait); when
 *                             its last CTA finishes it publishes signal_epoch (> 0, growing by 1 per call) to every rank.
 *                             With B result buffers used round-robin, call j (1-based epoch j) may pass wait_epoch =
 *                             j - B + 2 provided every rank reads the results of call s before it enqueues call s + 2:
 *                             B = 4 lets a rank run a full kernel ahead of the slowest one instead of meeting it at a
 *                             barrier after every call.
 *   sffg_peer_wait_device     enqueue "wait until every rank has published >= epoch": what a consumer of call `epoch`'s
 *                             gathered results puts in front of its work
 *   sffg_peer_barrier_device  signal + wait in one call (stand-alone barrier on the same flag words)
 *                             env may be NULL for both (a barrier between index searches): a timeout then aborts the
 *                             launch (the next CUDA call of the process fails) instead of raising the env's status
 * A rank that never arrives raises SFFG_ERR_INTERNAL at the next sffg_env_sync_check after 10 s instead of hanging the GPU. */
SFFG_API int sffg_peer_buffer_create(int64_t bytes, void **d_ptr_out, uint8_t handle_out[64]);
SFFG_API int sffg_peer_buffer_open(const uint8_t handle[64], void **d_ptr_out);
SFFG_API int sffg_peer_buffer_close(void *d_ptr);
SFFG_API int sffg_peer_buffer_destroy(void *d_ptr);
SFFG_API int sffg_collide_poses_gather_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n,
                                     uint8_t *const *d_outs, int n_outs, void *stream);
SFFG_API int sffg_collide_poses_gather_sync_device(sffg_env *env, const void *d_poses, int poses_are_f64, int64_t n,
                                          uint8_t *const *d_outs, uint32_t *const *d_flags, int n_ranks, int my_rank,
                                          uint32_t signal_epoch, uint32_t wait_epoch, uint32_t *d_done_counter,
                                          void *stream);
SFFG_API int sffg_peer_wait_device(sffg_env *env, uint32_t *const *d_flags, int n_ranks, int my_rank, uint32_t epoch,
                          void *stream);
SFFG_API int sffg_peer_barrier_device(sffg_env *env, uint32_t *const *d_flags, int n_ranks, int my_rank, uint32_t epoch,
                             void *stream);

/* ---- edge verdicts: Solver<T,R>::isPathFree(start, finish), src/problemStruct.h:154-168 -------------------
 * parts = distance6(start, finish) / sample_dist; samples index = 1 .. (index < parts); position =
 * start + index * dir / parts; stops at the first colliding sample.  free_out[i] = 1 if no sample collides;
 * first_hit_out (optional) = index of the first colliding sample, 0 if free.
 * The reference hard-codes sample_dist = 0.1 (collisionSampleSize, :121).                                     */
SFFG_API int sffg_check_edges(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist,
                     int rot_mode, uint8_t *free_out, int32_t *first_hit_out);
SFFG_API int sffg_check_edges_device(sffg_env *env, const double *d_starts, const double *d_ends, int64_t m,
                            double sample_dist, int rot_mode, uint8_t *d_free_out, int32_t *d_first_hit_out,
                            void *stream);

/* a move start -> end as every expansion step of the reference validates it: the end pose must be collision free AND the
 * segment must pass the local planner -- `env.Collide(newPoint) || !isPathFree(node, newPoint)` rejects
 * (src/forest.h:246, src/rrt.h:149, src/lazy.h:197).  ok_out[i] = 1 when move i is valid.  One call, one upload, both
 * kernels on one stream, one synchronisation.                                                                          */
SFFG_API int sffg_check_moves(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist,
                     int rot_mode, uint8_t *ok_out);

/* work counters of the last call on this env (debug/roofline): poses past the root cull, BVH child-box tests,
 * triangle-pair FP32 SAT tests, FP64 exact re-tests                                                          */
typedef struct {
  int64_t poses, poses_past_root, box_tests, pair_tests, exact_tests;
  int64_t traversal_steps, triangle_passes, triangles_transformed;   /* warp-level steps of the two inner loops */
  int64_t exact_run;   /* FP64 pair tests actually executed (exact_tests counts pairs FP32 SAT left undecided) */
  int64_t poses_past_grid;   /* poses neither culled by the obstacle AABB nor proven free by the clearance grid */
} sffg_counters_t;
SFFG_API int sffg_env_enable_counters(sffg_env *env, int on);
/* after *_device calls: waits for the device and reports a traversal failure (SFFG_ERR_INTERNAL) if one was flagged */
SFFG_API int sffg_env_sync_check(sffg_env *env);
SFFG_API int sffg_env_read_counters(sffg_env *env, sffg_counters_t *out);

/* ---- synthetic pose stream (SURVEY 8d): Philox4x32-10(seed, index); distribution of
 *      RandGen<T>::randomPointInSpace, src/randGen.h:123-146.  range = minX maxX minY maxY minZ maxZ --------- */
SFFG_API int sffg_gen_poses_device(uint64_t seed, uint64_t first_index, int64_t n, const float range[6], float *d_poses_out,
                          void *stream);

/* ---- neighbour index: flann::Index<D6Distance<float>> as used by the planner
 *      ctor+buildIndex src/forest.h:72-73; addPoints :367; knnSearch :317; radiusSearch :266-267
 *      (API lib/flann/src/cpp/flann/flann.hpp:101-115,:149-152,:289-296,:361-368).
 * Exact search with the INTENDED metric (src/primitives.h:404-438 with += ; == squared Point::distance
 * in float); ids are 0-based insertion order; distances are squared; ties resolve to the lower id. ---------- */
SFFG_API int sffg_index_create(int dim /* 2 or 6 */, sffg_index **out);
SFFG_API int sffg_index_destroy(sffg_index *idx);
SFFG_API int sffg_index_add(sffg_index *idx, const float *pts /* [n][dim] */, int64_t n);   /* copies; ids continue */
SFFG_API int sffg_index_add_device(sffg_index *idx, const float *d_pts, int64_t n, void *stream);
/* appends to several indices in one call (one upload, one synchronisation): pts holds n_per[0] rows for idx[0], then
 * n_per[1] rows for idx[1], ... -- the planner appends every new node to its tree's index (src/forest.h:367)        */
SFFG_API int sffg_index_add_multi(sffg_index *const *idx, const int64_t *n_per, int n_idx, const float *pts);
SFFG_API int64_t sffg_index_size(const sffg_index *idx);

/* k nearest, ascending (d2,id); rows shorter than k (index smaller than k) are padded with id -1, d2 +inf */
SFFG_API int sffg_knn(sffg_index *idx, const float *queries, int64_t nq, int k, int32_t *ids_out, float *d2_out);
SFFG_API int sffg_knn_device(sffg_index *idx, const float *d_queries, int64_t nq, int k, int32_t *d_ids_out, float *d2_out,
                    void *stream);
/* multi-GPU form of sffg_knn_device (node set replicated, query rows split over the ranks): the kernel that finishes a
 * row stores it to d_ids_dests[r] / d_d2_dests[r] for every r < n_dests -- this rank's row range inside every rank's
 * gathered [Q][k] buffers (sffg_peer_buffer_create / _open) -- so the row exchange rides on the search's own stores over
 * NVLink.  Follow it with sffg_peer_barrier_device(NULL, ...) on the same stream before anyone reads the gathered rows;
 * with two sets of gathered buffers used alternately and results read (on that stream) before the next call but one,
 * no further synchronisation is needed.                                                                            */
SFFG_API int sffg_knn_gather_device(sffg_index *idx, const float *d_queries, int64_t nq, int k, int32_t *const *d_ids_dests,
                           float *const *d_d2_dests, int n_dests, void *stream);

/* several indices in one call (the planner keeps one index per tree, src/forest.h:72): queries are concatenated in index
 * order, nq_per[i] rows for idx[i]; one upload, the per-index searches run concurrently on the indices' own streams, one
 * download, one synchronisation. */
SFFG_API int sffg_knn_multi(sffg_index *const *idx, const int64_t *nq_per, int n_idx, const float *queries, int k,
                            int32_t *ids_out, float *d2_out);

/* all points with d2 < r2 (strict), each row sorted by (d2,id); rows packed in query order.
 * counts_out[nq] is always written; *total_out = sum(counts).  Pass ids_out == NULL to size the buffers
 * (two-call protocol); otherwise capacity must be >= total or SFFG_ERR_CAPACITY is returned.                */
SFFG_API int sffg_radius(sffg_index *idx, const float *queries, int64_t nq, float r2, int32_t *counts_out,
                int32_t *ids_out, float *d2_out, int64_t capacity, int64_t *total_out);

/* ---- asynchronous forms for planner rounds --------------------------------------------------------------
 * The callers of this path (SpaceForest::expandNode, src/forest.h:240-376; RapidExpTree::expandNode, src/rrt.h:137-235)
 * ask one question after the other; the batched hosts ask them per round, and the questions of one round that do not
 * depend on each other (the radius search over all trees, the per-tree k nearest, the edges of the crowding rule,
 * appending the round's new nodes) can be in flight together.  A *_begin call enqueues the whole call -- upload,
 * kernels, download -- and returns; the results are in the caller's buffers (which, like the inputs, must stay alive) once the matching
 * end call has returned: sffg_index_end(idx) for sffg_radius_begin, sffg_index_end(idx[0]) for sffg_knn_multi_begin and
 * sffg_index_add_multi_begin, sffg_env_end(env) for sffg_check_edges_begin / sffg_check_moves_begin.  Between begin
 * and end, calls on OTHER objects run concurrently on the GPU (every index and every environment has its own stream);
 * a second host-pointer call on an object with a pending call is refused with SFFG_ERR_ARG (of the indices of a multi
 * call only idx[0] holds the pending call; the others stay usable without an end call); *_device launches on an
 * environment with a pending call are ordered behind it by the library (like all launches of one environment), *_device
 * calls on an index with a pending call share that index's scratch buffers and are the caller's to order.  Appends are ordered before
 * every later search on the indices they went to without any host synchronisation.  Batches too large for the pinned
 * staging area are simply executed by the begin call; the end call is then a no-op.  The blocking calls above are
 * begin + end.  sffg_radius (both forms) costs one host synchronisation for planner-sized batches: on indices of up to
 * 32 768 nodes the whole search is one kernel (a block per query), on larger ones the exclusive scan of the per-query
 * counts runs on the device between the count and the fill kernel.                                                     */
SFFG_API int sffg_radius_begin(sffg_index *idx, const float *queries, int64_t nq, float r2, int32_t *counts_out,
                               int32_t *ids_out, float *d2_out, int64_t capacity, int64_t *total_out);
SFFG_API int sffg_knn_multi_begin(sffg_index *const *idx, const int64_t *nq_per, int n_idx, const float *queries, int k,
                                  int32_t *ids_out, float *d2_out);
SFFG_API int sffg_index_add_multi_begin(sffg_index *const *idx, const int64_t *n_per, int n_idx, const float *pts);
SFFG_API int sffg_index_end(sffg_index *idx);
SFFG_API int sffg_check_edges_begin(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist,
                                    int rot_mode, uint8_t *free_out, int32_t *first_hit_out);
SFFG_API int sffg_check_moves_begin(sffg_env *env, const double *starts, const double *ends, int64_t m, double sample_dist,
                                    int rot_mode, uint8_t *ok_out);
SFFG_API int sffg_env_end(sffg_env *env);

#ifdef __cplusplus
}
#endif
#endif /* SFFG_H_ */
