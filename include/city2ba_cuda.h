/* city2ba_cuda.h — C ABI of libcity2ba_cuda.so: the B200 (sm_100a) replacement for city2ba's
 * visibility / observation-generation hot path and its elementwise noise pass.
 *
 * This is what a `build.rs` + `ffi.rs` on the Rust side would bind (see INTEGRATION.md).
 * Each entry point names the reference interface it replaces (paths relative to the
 * tkonolige/city2ba source tree).  Plain pointers and sizes only; no exceptions cross this
 * boundary; every function returns C2B_OK (0) or a negative c2b_status and leaves a message
 * retrievable with c2b_last_error() (thread local).  Calls are blocking.  One c2b_ctx drives
 * one GPU; issue calls from one host thread at a time per ctx.  Several GPUs of one box: c2b_init_multi /
 * c2b_visibility_graph_multi (one process, one ctx and worker thread per GPU, NCCL for the two exchanges), or one
 * process per GPU with each rank passing its own contiguous camera range to c2b_visibility_graph.
 *
 * There is NO CPU fallback: c2b_init fails with C2B_ERR_NO_DEVICE when no sm_100 GPU is
 * visible, and nothing else works without a ctx.
 */
#ifndef CITY2BA_CUDA_H
#define CITY2BA_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define C2B_ABI_VERSION 3

typedef enum {
  C2B_OK = 0,
  C2B_ERR_INVALID = -1,   /* bad argument (null pointer, index out of range, ...)        */
  C2B_ERR_NO_DEVICE = -2, /* no usable CUDA device                                        */
  C2B_ERR_CUDA = -3,      /* a CUDA runtime call or kernel failed; message has the detail */
  C2B_ERR_OOM = -4,       /* device or pinned-host allocation failed                      */
  C2B_ERR_EMPTY = -5,     /* empty problem (reference: Error::EmptyProblem, src/baproblem.rs:36) */
  C2B_ERR_NCCL = -6,      /* libnccl.so.2 could not be loaded, or an NCCL call failed (multi-GPU entries only) */
  C2B_ERR_IO = -7,        /* a file could not be created or opened, or a write was short (reference: Error::IOError) */
  C2B_ERR_PARSE = -8      /* a BAL file does not follow its grammar or ends early (reference: Error::ParseError) */
} c2b_status;

typedef struct c2b_ctx c2b_ctx;
typedef struct c2b_scene c2b_scene;

/* camera record = 15 doubles: R column-major [9] (cgmath Matrix3 {x,y,z} columns of
 * SnavelyCamera::dir), t [3] (SnavelyCamera::loc), f,k1,k2 (SnavelyCamera::intrin)
 * — src/baproblem.rs:131-138 */
#define C2B_CAM_STRIDE 15

/* ---- lifetime ------------------------------------------------------------------------------ */
/* replaces embree_rs::Device::new(), src/bin/city2ba.rs:515.  device = CUDA ordinal. */
int c2b_init(int device, c2b_ctx **out);
void c2b_shutdown(c2b_ctx *ctx);
const char *c2b_last_error(void);
int c2b_abi_version(void);
/* number of CUDA kernels this library has launched in this process so far */
uint64_t c2b_kernel_launches(void);
/* Measurement / test hooks.  Defaults are the product's behaviour; each hook is also read ONCE from the
 * environment in c2b_init (upper case, C2B_ prefix: C2B_BATCHES=1 ...).  name = "reset" restores the defaults.
 *   parts_log2 (-1 auto | 0..2)  tickets per camera in the fused kernel = 2^k
 *   trilist_cap (128)            leaf-list entries per camera before the camera traverses the BVH instead
 *   max_pairs (2^32-1)           pairs inside max_dist one resident pass may hold (lower: forces range splits)
 *   hoist_max (64)               leaf lists up to this length get per-camera triangle records
 *   packet_bvh (1)               list overflow: 1 lane = node packet traversal, 0 per-ray stackless walk
 *   trilist_warp (-1 auto|0|1)   leaf lists built by one warp / one thread per camera
 *   batches (0 auto)             camera batches of the host-buffer call
 *   grid_cell_factor (0.25)      point-grid cell side / max_dist
 *   grid_x_split (8)             point-grid cells in x are 1/k of the side (rounded down to a power of two, at most
 *                                64; halved while the grid would exceed 2^22 cells)
 *   optimistic (1)               later passes on a ctx launch their kernels without waiting for the plan's totals
 *                                (sizes and kernel variant from the previous pass, checked by the kernels)
 *   cold_staged (1)              first host-buffer call on a ctx: CSR in unpinned memory through a pinned ring
 *   stage_threads (4)            host threads staging a PAGEABLE input array through the pinned ring (0: leave
 *                                the pageable copy to the driver)
 *   bal_chunk_bytes (2^25)       byte budget of one chunk of c2b_write_bal* and c2b_read_bal_resident (device buffer
 *                                and pinned ring slot);
 *                                at least 4096, rounded down to a multiple of 8
 * Unknown names are C2B_ERR_INVALID. */
int c2b_tune(c2b_ctx *ctx, const char *name, double value);
/* measurement aid (SURVEY 8d): sustained rate of independent f64 FMAs on this device, in DFMA/s
 * (one fused multiply-add per thread counted as one).  The secondary bound of the exhaustive cull, whose
 * hot loop is FP64-issue-bound; not part of the reference's surface. */
int c2b_probe_fp64(c2b_ctx *ctx, double *dfma_per_s);

/* ---- scene (triangle mesh -> GPU LBVH) ----------------------------------------------------------
 * replaces Scene::new + model_to_geometry + attach_geometry + commit
 * (src/generate.rs:74-105, src/bin/city2ba.rs:515-521).  xyz = 3*nv tightly packed f32 (tobj
 * positions), tri = 3*nt u32 (all OBJ objects concatenated, indices already offset).  Triples
 * with a repeated index (tobj's 2-index `l` records padded into triples) can never be hit and
 * are dropped; a triple touching a vertex >= nv is C2B_ERR_INVALID.  nt may be 0. */
int c2b_scene_create(c2b_ctx *ctx, const float *xyz, uint64_t nv, const uint32_t *tri, uint64_t nt,
                     c2b_scene **out);
/* replaces CommittedScene::bounds(), src/generate.rs:237 */
int c2b_scene_bounds(const c2b_scene *scene, float lower[3], float upper[3]);
uint64_t c2b_scene_num_triangles(const c2b_scene *scene);
uint64_t c2b_scene_num_nodes(const c2b_scene *scene);
void c2b_scene_destroy(c2b_scene *scene);

/* ---- ray-level entries (parity tooling + camera placement) -------------------------------------
 * Embree-compatible 48-byte AoS ray (RTCRay): replaces CommittedScene::occluded_stream_aos
 * (src/generate.rs:472): on a hit tfar is set to -inf, otherwise the ray is left untouched.
 * tnear is honoured as 0 (the reference never sets it). */
typedef struct {
  float org_x, org_y, org_z, tnear;
  float dir_x, dir_y, dir_z, time;
  float tfar;
  uint32_t mask, id, flags;
} c2b_ray48;
int c2b_occluded(c2b_ctx *ctx, const c2b_scene *scene, c2b_ray48 *rays, uint64_t n_rays);
/* Embree rtcIntersect1 as a batch: closest hit of every ray through the BVH.  On a hit tfar = distance
 * and flags = 1; otherwise the ray is left untouched and flags = 0. */
int c2b_intersect(c2b_ctx *ctx, const c2b_scene *scene, c2b_ray48 *rays, uint64_t n_rays);
/* replaces CommittedScene::intersect on a single ray (src/generate.rs:253-262): closest hit;
 * *hit = 1 and *tfar = distance when something is hit, else *hit = 0. */
int c2b_intersect1(c2b_ctx *ctx, const c2b_scene *scene, const float org[3], const float dir[3],
                   int *hit, float *tfar);

/* ---- the hot path: visibility graph ------------------------------------------------------------
 * replaces city2ba::generate::visibility_graph (src/generate.rs:424-481) for one contiguous
 * camera range. */
typedef enum {
  C2B_CULL_GRID = 0,      /* default: points binned in a uniform grid, each camera scans only the
                             cells its max_dist ball touches, then the exact f64 predicates */
  C2B_CULL_EXHAUSTIVE = 1 /* every camera x point pair is tested, like the reference's loop at
                             src/generate.rs:446 */
} c2b_cull_mode;

typedef enum {
  C2B_OCC_MESH = 0,    /* rays against the scene's BVH (generate path) */
  C2B_OCC_NONE = 1,    /* no occlusion (synthetic_line, src/synthetic.rs:353-379) */
  C2B_OCC_ANALYTIC = 2 /* 2-D wall test of `synthetic` (src/synthetic.rs:52-124) */
} c2b_occlusion;

typedef enum {
  C2B_PRED_WATERTIGHT = 0, /* default: watertight edge-function test (what the north star asks for) */
  C2B_PRED_MT = 1          /* Moeller-Trumbore in the form of Embree 3's default intersector — what the
                              reference's default scene runs (src/bin/city2ba.rs:515-521, src/generate.rs:472);
                              restated from the published algorithm, not watertight on shared edges */
} c2b_predicate;

typedef struct {
  int cull_mode;          /* c2b_cull_mode */
  int occlusion;          /* c2b_occlusion; MESH needs a scene */
  int endpoint_guard_rel; /* 0 = reference: tfar = f32(|d|) - 1e-6f (src/generate.rs:464);
                             1 = additionally tfar *= (1 - 2^-18) (documented, non-default) */
  int count_traversal;    /* 1 = count BVH nodes visited / triangles tested (slower) */
  double block_length;    /* C2B_OCC_ANALYTIC only */
  double block_inset;     /* C2B_OCC_ANALYTIC only */
  int predicate;          /* c2b_predicate; C2B_OCC_MESH only */
  int reserved;           /* 0 */
} c2b_vis_options;
void c2b_vis_options_default(c2b_vis_options *opt);

typedef struct {
  /* CSR of visible observations, camera-major, ascending point index inside each camera
   * (the order src/generate.rs:446,473-478 produces).  Host memory owned by the ctx (pinned; the first
   * host-buffer call on a ctx uses unpinned memory filled through a pinned ring, because pinning a large result
   * takes longer than producing it — hook cold_staged): valid until the next c2b_visibility_graph* call on the
   * same ctx or c2b_shutdown. */
  uint64_t n_cameras;
  uint64_t n_obs;
  uint64_t *offsets;   /* [n_cameras+1] */
  uint32_t *point_idx; /* [n_obs]; 32-bit on purpose: P < 2^32 is enforced, and the result crosses PCIe
                          (20 instead of 24 bytes per observation); the binding widens to usize */
  double *uv;          /* [2*n_obs] u,v interleaved (normalised image coordinates) */
  /* statistics of this call */
  uint64_t n_candidates;    /* pairs that passed distance/front/frustum (= rays cast)      */
  uint64_t pairs_evaluated; /* camera x point pairs the cull kernel actually tested          */
  uint64_t nodes_visited;   /* warp-level BVH node visits (count_traversal only)            */
  uint64_t tris_tested;     /* warp-level triangle tests  (count_traversal only)            */
  uint64_t h2d_bytes, d2h_bytes;
  /* device time of each stage, CUDA events on the ctx stream, milliseconds */
  float ms_h2d, ms_prep, ms_cull, ms_sort, ms_traverse, ms_compact, ms_d2h, ms_total;
} c2b_obs;

/* one call, host buffers in, host CSR out (what the Rust visibility_graph body would call).
 * cams: C x 15 doubles; pts: P x 3 doubles (cgmath Point3<f64> is repr(C)).  pts == NULL with P equal to
 * the number of points already resident (c2b_upload_points / c2b_upload_points_device) reuses them. */
int c2b_visibility_graph(c2b_ctx *ctx, const c2b_scene *scene, const double *cams, uint64_t C,
                         const double *pts, uint64_t P, double max_dist,
                         const c2b_vis_options *opt, c2b_obs *out);
void c2b_obs_free(c2b_ctx *ctx, c2b_obs *obs);

/* the same path split in three so a caller can keep inputs/outputs resident in HBM
 * (bench `value`, multi-pass pipelines).  upload -> run (device CSR stays in the ctx) -> download. */
int c2b_upload_points(c2b_ctx *ctx, const double *pts, uint64_t P);
/* the same from a DEVICE pointer on the ctx's GPU (e.g. the output of an NCCL all-gather when every
 * rank uploaded 1/N of the points over its own PCIe link); the caller's stream must have finished
 * writing d_pts.  The data is copied; d_pts may be reused afterwards. */
int c2b_upload_points_device(c2b_ctx *ctx, const double *d_pts, uint64_t P);
/* zero-copy variant: the ctx's own device array of xyz records (room for `capacity` points) for a caller
 * that fills it on the device — c2b_visibility_graph_multi all-gathers the per-GPU shards straight into it —
 * then c2b_points_commit(P) once the writes are ordered before the ctx's work (same stream or synchronised). */
int c2b_points_device_buffer(c2b_ctx *ctx, uint64_t capacity, double **d_out);
int c2b_points_commit(c2b_ctx *ctx, uint64_t P);
int c2b_upload_cameras(c2b_ctx *ctx, const double *cams, uint64_t C);
/* The point grid (cells of side max_dist/4) is derived data that the ctx keeps between calls on the same
 * points and max_dist.  This forgets it, so that the next resident pass pays the build again (ms_prep):
 * what a one-shot `visibility_graph` call costs; bench.py's `value` is measured this way. */
int c2b_drop_point_grid(c2b_ctx *ctx);
int c2b_visibility_graph_resident(c2b_ctx *ctx, const c2b_scene *scene, double max_dist,
                                  const c2b_vis_options *opt, c2b_obs *stats_out);
int c2b_download_obs(c2b_ctx *ctx, c2b_obs *out);
/* the resident CSR into CALLER-owned arrays (pinned for full PCIe rate; pageable works): offsets_dst receives
 * n_cameras entries (+ the closing one if with_end), each increased by obs_base — the slot of a camera range
 * inside a larger CSR; idx_dst / uv_dst receive n_obs entries.  ms_d2h (optional): device time of the copies. */
int c2b_download_obs_into(c2b_ctx *ctx, uint64_t obs_base, uint64_t *offsets_dst, uint32_t *idx_dst,
                          double *uv_dst, int with_end, float *ms_d2h);

/* ---- the same path on several GPUs of one box (SURVEY 8e) -------------------------------------------
 * replaces the rayon par_iter over cameras (src/generate.rs:434-441) and its order-preserving collect
 * (:479-481).  ONE process drives n_gpus devices: one c2b_ctx + stream set + host thread per device and one
 * NCCL communicator (ncclCommInitAll; libnccl.so.2 is loaded with dlopen the first time, so single-GPU users
 * need no NCCL).  Mesh / BVH and points are replicated, every GPU owns a contiguous camera range — equal ranges at
 * first, then sized in proportion to the rate at which each GPU's slab reached host memory in the previous call
 * (the GPUs of a box do not all reach host memory equally fast; C2B_MULTI_ADAPTIVE=0 keeps them equal).  Data exchanged over NVLink: (1) every GPU uploads 1/G of the point
 * array over its own PCIe link and the shards are all-gathered (ncclAllGather) into each GPU's point array;
 * (2) ONE ncclAllGather of the per-GPU observation counts, from which every GPU rebases its CSR offsets on
 * the device and learns where its slab starts; every GPU then copies its slab into the SAME pinned host CSR
 * at that offset.  The result is identical to c2b_visibility_graph's, bit for bit. */
typedef struct c2b_multi c2b_multi;
typedef struct c2b_multi_scene c2b_multi_scene;
#define C2B_MAX_GPUS 16
/* devices == NULL: ordinals 0 .. n_gpus-1 */
int c2b_init_multi(int n_gpus, const int *devices, c2b_multi **out);
void c2b_shutdown_multi(c2b_multi *m);
int c2b_multi_num_gpus(const c2b_multi *m);
/* the per-GPU context (valid until c2b_shutdown_multi), e.g. for c2b_tune or the single-GPU entries */
c2b_ctx *c2b_multi_ctx(c2b_multi *m, int g);
/* the BVH is built on every GPU (the build is deterministic: identical copies) */
int c2b_scene_create_multi(c2b_multi *m, const float *xyz, uint64_t nv, const uint32_t *tri, uint64_t nt,
                           c2b_multi_scene **out);
void c2b_scene_destroy_multi(c2b_multi_scene *scene);
/* GPU g's copy (owned by the multi scene), e.g. for c2b_intersect on c2b_multi_ctx(m, g) */
c2b_scene *c2b_multi_scene_get(const c2b_multi_scene *scene, int g);
typedef struct {
  int n_gpus;
  uint64_t cam_begin[C2B_MAX_GPUS], cam_end[C2B_MAX_GPUS]; /* camera range of GPU g                     */
  uint64_t n_obs[C2B_MAX_GPUS];                            /* its observation count = slab length         */
  uint64_t obs_base[C2B_MAX_GPUS];                         /* its slab's start in the host CSR (from the
                                                              all-gathered counts, computed on the device) */
  float ms_points[C2B_MAX_GPUS];  /* shard H2D + point all-gather + SoA / bounds                          */
  float ms_compute[C2B_MAX_GPUS]; /* resident pass (grid build, plan, fused kernel, sort + write)         */
  float ms_exchange[C2B_MAX_GPUS];/* count all-gather + offset rebase                                     */
  float ms_d2h[C2B_MAX_GPUS];     /* slab -> host CSR                                                     */
  float ms_wall;                  /* host wall clock of the whole call                                    */
} c2b_multi_stats;
/* out: the ONE host CSR (pinned, owned by `m`, valid until the next call or c2b_shutdown_multi); the stage
 * timers of `out` are the maxima over GPUs.  stats may be NULL. */
int c2b_visibility_graph_multi(c2b_multi *m, const c2b_multi_scene *scene, const double *cams, uint64_t C,
                               const double *pts, uint64_t P, double max_dist, const c2b_vis_options *opt,
                               c2b_obs *out, c2b_multi_stats *stats);

/* total_reprojection_error (src/baproblem.rs:265-279) of the resident problem, norm 1 or 2 fast
 * paths, anything else through pow(). */
int c2b_reprojection_error_resident(c2b_ctx *ctx, double norm, double *out);

/* ---- noise pass (src/noise.rs:35-177) ------------------------------------------------------------
 * In place on host arrays: cams C x 15, pts P x 3, uv O x 2.  Randomness is Philox4x32-10 keyed
 * by `seed` with counter (element index, stream, slot) — the reference uses thread_rng(), which
 * cannot be seeded, so parity is exact against the oracle's identical stream and distributional
 * against the reference: a direction (the reference's normalised Gaussian pair / triple) is drawn uniformly
 * on the circle / sphere, a magnitude by Box-Muller (city2ba_b200/csrc/c2b_noise.cuh). */
/* replaces noise::add_drift (src/noise.rs:68-116) */
int c2b_add_drift(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, double strength,
                  double angle_strength, double std, const double dir[3], uint64_t seed);
/* replaces noise::add_drift_normalized (src/noise.rs:47-56) */
int c2b_add_drift_normalized(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P,
                             double strength, double angle_strength, double std, uint64_t seed);
/* replaces noise::add_noise (src/noise.rs:119-177) */
int c2b_add_noise(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, double *uv,
                  uint64_t O, double translation_std, double rotation_std, double point_std,
                  double observations_std, uint64_t seed);
/* replaces noise::add_sin_noise (src/noise.rs:388-416): every camera centre / point x moves by
 * sin(dot(x / dimensions, dir) * frequency * pi) * strength * normalize(noise_dir), dimensions =
 * BAProblem::dimensions (src/baproblem.rs:307-337; zero extents count as 1e-8).  Deterministic. */
int c2b_add_sin_noise(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, const double dir[3],
                      const double noise_dir[3], double strength, double frequency);
/* The same passes on the RESIDENT problem — the cameras and points of the last c2b_upload_* calls and the
 * (u, v) of the last c2b_visibility_graph_resident — in place in HBM: `generate -> noise` without crossing PCIe.
 * dir == NULL in c2b_add_drift_resident is add_drift_normalized.  Afterwards c2b_download_problem /
 * c2b_download_obs fetch the noised problem and c2b_reprojection_error_resident measures it. */
int c2b_add_drift_resident(c2b_ctx *ctx, double strength, double angle_strength, double std, const double *dir,
                           uint64_t seed);
int c2b_add_noise_resident(c2b_ctx *ctx, double translation_std, double rotation_std, double point_std,
                           double observations_std, uint64_t seed);
int c2b_add_sin_noise_resident(c2b_ctx *ctx, const double dir[3], const double noise_dir[3], double strength,
                               double frequency);
/* cameras (C x 15) and points (P x 3) of the resident problem -> host */
int c2b_download_problem(c2b_ctx *ctx, double *cams_out, double *pts_out);
/* device time of the last noise call on this ctx (CUDA events on its stream), milliseconds:
 * ms[0] upload, ms[1] statistics + elementwise kernels, ms[2] download */
int c2b_noise_timing(c2b_ctx *ctx, float ms[3]);
/* BAProblem::mean / std (src/baproblem.rs:282-304) */
int c2b_mean_std(c2b_ctx *ctx, const double *cams, uint64_t C, const double *pts, uint64_t P,
                 double mean[3], double std[3]);

/* ---- graph post-processing -------------------------------------------------------------------------
 * replaces BAProblem::cull (src/baproblem.rs:538-549) = largest_connected_component (:456-534, with its
 * observation filter at :523 as written: the point index looked up as an entity index without the camera offset)
 * then remove_singletons (:426-453), to a fixed point.  Components are labelled by their smallest entity
 * (cameras 0..C-1, then points C..C+P-1); the largest wins, the lowest label on a tie (the reference's HashMap
 * order is unspecified).  Records, points and (u, v) are copied, never recomputed: the result equals the host
 * mirrors' bit for bit.  Bounds: C + P < 2^32 - 1 and O < 2^32 - 1 (C2B_ERR_INVALID otherwise).
 * After c2b_visibility_graph_multi the graph is spread over the GPUs: cull its host CSR with c2b_cull_problem on
 * c2b_multi_ctx(m, 0). */
typedef struct {
  uint64_t n_cameras, n_points, n_obs; /* after the cull */
  uint32_t iterations;                 /* applications of LCC + remove_singletons, as the reference's loop */
  uint32_t reserved;
  float ms_h2d, ms_compute, ms_d2h;    /* device time (CUDA events on the ctx stream); h2d/d2h 0 when resident;
                                          ms_h2d includes the input check */
} c2b_cull_stats;
/* in place on host arrays: the culled problem is written into the prefixes of cams / pts / offsets /
 * point_idx / uv.  O = offsets[C], and point_idx / uv must hold O entries: they are read up to that length before
 * anything is checked, so offsets[C] has to be the arrays' length even when other offsets are wrong.  Rejects offsets[0] != 0, decreasing offsets and point_idx >= P
 * (from_visibility's asserts) with C2B_ERR_INVALID and leaves the arrays untouched.  Does not touch the
 * ctx's resident problem.  out may be NULL. */
int c2b_cull_problem(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, uint64_t *offsets,
                     uint32_t *point_idx, double *uv, c2b_cull_stats *out);
/* the same on the resident problem: the cameras / points of the last c2b_upload_* calls and the CSR of the last
 * c2b_visibility_graph_resident.  Afterwards c2b_download_obs / c2b_download_problem /
 * c2b_reprojection_error_resident / c2b_add_*_resident see the culled problem, and a new
 * c2b_visibility_graph_resident computes the culled problem's graph.  C2B_ERR_INVALID without a resident result,
 * and after the host-buffer c2b_visibility_graph (which leaves only its last camera batch resident). */
int c2b_cull_problem_resident(c2b_ctx *ctx, c2b_cull_stats *out);

/* ---- noise::add_incorrect_correspondences (src/noise.rs:180-226) ------------------------------------------------
 * In every camera of more than one observation, observation i is selected with probability mismatch_chance and swaps
 * its point index with observation j of the same camera, drawn with weight maxd - |uv_i - uv_j| (maxd the largest such
 * distance; i itself weighs maxd).  (u, v), offsets, cameras and points are not changed.  Deterministic in seed:
 * one Philox4x32-10 block per observation (key seed, counter (o lo, o hi, 6, 0)); u from words 0-1 (53 bits) selects
 * when u <= mismatch_chance; weights are quantised to floor(w / maxd * 2^32) and j is found from words 2-3 by an
 * integer prefix sum (DESIGN.md §4, "Mismatched correspondences").  The transpositions apply per camera in ascending i.
 * A selected observation whose distances are not all finite fails with NegativeWeight, one whose distances are all 0
 * with AllWeightsZero (Rng::weighted): C2B_ERR_INVALID, the message names the lowest such observation and its camera
 * and ends in "called `Result::unwrap()` on an `Err` value: <kind>"; nothing is changed then. */
typedef struct {
  uint64_t n_selected;               /* observations selected (in cameras of more than one observation) */
  uint64_t n_swapped;                /* selections whose partner is another observation */
  float ms_h2d, ms_compute, ms_d2h;  /* device time (CUDA events on the ctx stream); h2d/d2h 0 when resident;
                                        ms_h2d includes the input check */
} c2b_mismatch_stats;
/* in place on host arrays: point_idx / uv hold O = offsets[C] entries.  Rejects offsets[0] != 0 and decreasing
 * offsets with C2B_ERR_INVALID and leaves point_idx untouched.  C and O below 2^32 - 1.  Does not touch the ctx's
 * resident problem.  out may be NULL. */
int c2b_add_incorrect_correspondences(c2b_ctx *ctx, const uint64_t *offsets, uint64_t C, uint32_t *point_idx,
                                      const double *uv, double mismatch_chance, uint64_t seed,
                                      c2b_mismatch_stats *out);
/* the same on the resident CSR, in HBM; afterwards c2b_download_obs, c2b_reprojection_error_resident,
 * c2b_cull_problem_resident and c2b_write_bal_resident see the edited graph.  Refuses in the cases
 * c2b_cull_problem_resident refuses. */
int c2b_add_incorrect_correspondences_resident(c2b_ctx *ctx, double mismatch_chance, uint64_t seed,
                                               c2b_mismatch_stats *out);

/* ---- noise::join_landmarks (src/noise.rs:323-378) ---------------------------------------------------------------
 * n = floor(join_percent * P) (0 when join_percent is negative or NaN) observations, min(n, O) of them, drawn over all
 * O observations, are each re-pointed at one of the 10 nearest other landmarks of the landmark they see.  Points,
 * offsets and (u, v) are not changed.  Deterministic in seed (DESIGN.md §4, "Joined landmarks"): one Philox4x32-10
 * block per observation o (key seed, counter (o lo, o hi, 7, 0)); the selected observations are the min(n, O) smallest
 * pairs (w0 | w1 << 32, o); the neighbour list is the m = min(11, P) smallest pairs (d2, k) over all points, d2 the
 * squared distance to the landmark seen, rounded to nearest in the order (dx dx + dy dy) + dz dz; the observation
 * takes list[1 + mulhi64(w2 | w3 << 32, m - 1)], the search is exact.  With at least one selection, P < 2 fails with a
 * message ending in "No neighbors?!" and a point with a coordinate that is not finite fails naming the lowest such
 * point: C2B_ERR_INVALID, nothing is changed then. */
typedef struct {
  uint64_t n_selected;               /* observations selected: min(n, O) */
  uint64_t n_changed;                /* selections whose new point differs from the one they saw */
  float ms_h2d, ms_compute, ms_d2h;  /* device time (CUDA events on the ctx stream); h2d/d2h 0 when resident;
                                        ms_h2d includes the input check */
} c2b_join_stats;
/* in place on host arrays: pts holds P points (x, y, z), point_idx O = offsets[C] entries.  Rejects offsets[0] != 0,
 * decreasing offsets and indices >= P with C2B_ERR_INVALID and leaves point_idx untouched.  C + P and O below
 * 2^32 - 1.  Does not touch the ctx's resident problem.  out may be NULL. */
int c2b_join_landmarks(c2b_ctx *ctx, const double *pts, uint64_t P, const uint64_t *offsets, uint64_t C,
                       uint32_t *point_idx, double join_percent, uint64_t seed, c2b_join_stats *out);
/* the same on the resident points and CSR, in HBM; afterwards c2b_download_obs, c2b_reprojection_error_resident,
 * c2b_cull_problem_resident and c2b_write_bal_resident see the edited graph.  Refuses in the cases
 * c2b_cull_problem_resident refuses. */
int c2b_join_landmarks_resident(c2b_ctx *ctx, double join_percent, uint64_t seed, c2b_join_stats *out);

/* ---- BAL files (BAProblem::write, src/baproblem.rs:709-764) ----------------------------------------------------
 * The file is encoded on the device and streamed to disk in chunks of at most bal_chunk_bytes: the D2H copy and
 * the host write of one chunk overlap the encoding of the next, and the device and pinned memory of the encoder
 * do not grow with the problem.  The bytes are the reference's:
 *   C2B_BAL_TEXT    header "C P O", then "c p u v" per observation, the 9-vector (to_vec) of every camera and the
 *                   3 coordinates of every point, one line each; every f64 as Rust's `{}` prints it: the shortest
 *                   digits that round-trip, positional (1e21 -> 1000000000000000000000, 5e-324 -> 0.000...005),
 *                   "NaN", "inf", "-inf", "-0"
 *   C2B_BAL_BINARY  big-endian u64 C P O, per camera its observation count then (u64 point, f64 u, f64 v) records,
 *                   the camera 9-vectors, the points
 * The camera 9-vectors are computed on the host by c2b_camera_to_vec. */
typedef enum { C2B_BAL_TEXT = 0, C2B_BAL_BINARY = 1 } c2b_bal_format;
typedef struct {
  uint64_t bytes;      /* size of the file written */
  uint64_t chunks;
  float ms_encode;     /* device time of the encoding kernels, summed over chunks (CUDA events) */
  float ms_d2h;        /* device time of the chunk copies to pinned memory, summed */
  float ms_write;      /* host wall time spent in write(2), summed */
} c2b_bal_stats;
/* host arrays in the layout of c2b_cull_problem (cams C x 15, pts P x 3, offsets C + 1, point_idx / uv
 * offsets[C] entries); offsets[0] != 0, decreasing offsets and point_idx >= P are C2B_ERR_INVALID and no file
 * is created.  Does not touch the ctx's resident problem.  out may be NULL. */
int c2b_write_bal(c2b_ctx *ctx, const char *path, int format, const double *cams, uint64_t C, const double *pts,
                  uint64_t P, const uint64_t *offsets, const uint32_t *point_idx, const double *uv,
                  c2b_bal_stats *out);
/* the resident problem (after c2b_visibility_graph_resident, and after a resident cull or noise pass); refuses
 * in the cases c2b_cull_problem_resident refuses */
int c2b_write_bal_resident(c2b_ctx *ctx, const char *path, int format, c2b_bal_stats *out);

/* ---- reading BAL files (BAProblem::from_file, src/baproblem.rs:580-706) -----------------------------------------
 * The file is streamed to the device in chunks of at most bal_chunk_bytes (pinned ring -> device buffer), parsed
 * there, and becomes the ctx's RESIDENT problem: cameras (c2b_camera_from_vec of the file's 9-vectors, on the host),
 * points, and the CSR grouped by camera in file order (BAProblem::new, src/baproblem.rs:342-355).  Afterwards
 * c2b_download_obs[_into], c2b_download_problem, c2b_reprojection_error_resident, c2b_add_*_resident,
 * c2b_cull_problem_resident and c2b_write_bal_resident work on it.
 *   C2B_BAL_TEXT    tokens separated by ASCII whitespace: "C P O", O x "c p u v", 9C camera numbers, 3P point
 *                   numbers; tokens after them are ignored.  Indices are digits only (nom's digit1, fitting a u64);
 *                   numbers follow Rust's f64::from_str ([+-]? digits with optional '.', optional exponent, or
 *                   inf / infinity / nan in any case), correctly rounded (round half to even) for any digit count.
 *                   A token longer than bal_chunk_bytes is C2B_ERR_PARSE.
 *   C2B_BAL_BINARY  the layout c2b_write_bal writes; doubles are copied bit for bit; trailing bytes are ignored.
 * C2B_ERR_PARSE: a malformed token (the message names the byte offset of the first), too few tokens, header counts
 * the file cannot hold, a truncated binary file, binary counts that exceed what is left or do not sum to O.
 * C2B_ERR_INVALID: an observation's camera or point index out of range (BAProblem::new's asserts), C, P or O not
 * below 2^32 - 1, an unknown format.  C2B_ERR_IO: the file cannot be opened or read.  After any failure there is no
 * resident problem (the entries above refuse with C2B_ERR_INVALID).  out may be NULL. */
typedef struct {
  uint64_t n_cameras, n_points, n_obs;
  uint64_t bytes;       /* bytes of the file read */
  uint64_t chunks;
  uint64_t slow_tokens; /* numbers the device could not round on its own, converted on the host (std::from_chars) */
  uint32_t regrouped;   /* 1 when the observations were not in camera order and were grouped on the device */
  uint32_t reserved;
  float ms_read;        /* host wall time in pread(2), summed */
  float ms_h2d;         /* device time of the chunk copies, summed (CUDA events) */
  float ms_parse;       /* device time of the parse kernels, summed (CUDA events) */
} c2b_bal_read_stats;
int c2b_read_bal_resident(c2b_ctx *ctx, const char *path, int format, c2b_bal_read_stats *out);

/* ---- input generation on the GPU -------------------------------------------------------------------
 * replaces generate_world_points_uniform (src/generate.rs:356-420): num_points world points, each
 * on an area-weighted random triangle (all index triples of all models, concatenated), uniform
 * inside it (random_point_in_triangle, :314-326), kept only if some camera centre lies within
 * max_dist (the R-tree query at :396-400, dist^2 <= max_dist^2).  Candidate k is a pure function of
 * (seed, k) — Philox4x32-10 — and accepted candidates are returned in candidate order, so the result is
 * deterministic (the reference's thread_rng() is not seedable: parity with it is distributional, with
 * the oracle exact).  Errors mirror the reference's panics: no cameras; more than 10 * num_points
 * rejections before num_points acceptances ("Failed to generate enough points ..."). */
int c2b_generate_world_points_uniform(c2b_ctx *ctx, const float *xyz, uint64_t nv, const uint32_t *tri,
                                      uint64_t nt, const double *cams, uint64_t C, uint64_t num_points,
                                      double max_dist, uint64_t seed, double *pts_out, uint64_t *n_out);

/* ---- host-side input generators (no GPU work) ----------------------------------------------------
 * camera/point lattices of synthetic_grid / synthetic_line (src/synthetic.rs:178-258, 323-344)
 * and the city-block box mesh used as the synthetic triangle scene. */
uint64_t c2b_grid_num_cameras(uint64_t cameras_per_block, uint64_t num_blocks);
uint64_t c2b_grid_num_points(uint64_t points_per_block, uint64_t num_blocks);
int c2b_grid_cameras(uint64_t cameras_per_block, uint64_t num_blocks, double block_length,
                     double camera_height, double *cams_out);
int c2b_grid_points(uint64_t points_per_block, uint64_t num_blocks, double block_length,
                    double block_inset, double point_height, double *pts_out);
int c2b_line_cameras(uint64_t num_cameras, double length, double camera_height, double *cams_out);
int c2b_line_points(uint64_t num_points, double length, double point_offset, double point_height,
                    double *pts_out);
int c2b_city_mesh(uint64_t num_blocks, double block_length, double block_inset, double height,
                  float *xyz_out /* 3*8*n^2 */, uint32_t *tri_out /* 3*12*n^2 */);

/* SnavelyCamera helpers on the host (src/baproblem.rs:141-176) — used by the host mirror */
void c2b_camera_center(const double *cam, double out[3]);
void c2b_camera_project_world(const double *cam, const double p[3], double out[3]);
void c2b_camera_project(const double *cam, const double pc[3], double out[2]);
void c2b_camera_from_position_direction(const double pos[3], const double R[9], double *cam_out);
void c2b_camera_transform(const double *cam, const double dR[9], const double dloc[3],
                          double *cam_out);
/* SnavelyCamera::to_vec (src/baproblem.rs:192-202): [rodrigues 3, translation 3, f, k1, k2], the same operations
 * as include/city2ba.hpp's to_vec, bit for bit */
void c2b_camera_to_vec(const double *cam, double out[9]);
/* SnavelyCamera::from_vec (src/baproblem.rs:180-190): the record of a 9-vector, the same operations as
 * include/city2ba.hpp's from_vec (both branches of from_rodrigues), bit for bit */
void c2b_camera_from_vec(const double v[9], double *cam_out);

#ifdef __cplusplus
}
#endif
#endif /* CITY2BA_CUDA_H */
