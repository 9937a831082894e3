// c2b_fused.cuh — the grid schedule of c2b_visibility_graph as ONE pass per camera:
// cull + projection (src/generate.rs:446-454), ray construction (:456-464), occlusion (:472) and
// the visible-point list (:473-478) without a candidate pool in between.
//
//   k_cam_plan          one thread per camera: the x-contiguous cell rows its max_dist ball touches, each
//                       trimmed by what is linear in x along a row (in front of the camera, the four
//                       side planes of the image, the ball); the trimmed (start, end) point ranges are
//                       kept for the fused pass, their total (an upper bound of the camera's visible
//                       count) -> exclusive scan -> the camera's slice of the scratch index array.
//   k_visibility_fused  persistent warps drawing cameras from a ticket.  Per camera the warp scans the
//                       planned rows 32 grid-ordered points at a time, evaluates the exact f64 predicate
//                       per lane and stages the survivors in shared memory.  Every 32 survivors form a
//                       ray packet that is resolved at once: the rays are built from the coordinates
//                       just read (L1 hits), the camera's leaf list (k_cam_trilist) is filtered against
//                       the packet's segment box and direction box with lane = triangle, and lane = ray
//                       runs the 9-FMA edge-function test on the survivors' origin-relative records
//                       (TriRec; computed once per camera when the list has <= 64 entries, else once per
//                       packet; cameras whose list overflows traverse the BVH with lane = node).
//                       Visible point indices go to the camera's scratch slice; no atomics.
//   k_sort_write        one warp per camera: warp-private LSD radix sort of the visible indices
//                       (ascending point index, src/generate.rs:446), (u, v) recomputed with the
//                       cull kernel's device function (bit-identical), CSR records written coalesced.
#pragma once
#include "c2b_common.cuh"
#include "c2b_compact.cuh"
#include "c2b_cull.cuh"
#include "c2b_math.cuh"
#include "c2b_traverse.cuh"

namespace c2b {

struct FusedArgs {
  // cameras
  const double *cams;                   // [15*C]
  const double *cen_x, *cen_y, *cen_z;  // [C]
  uint64_t C;
  // grid-ordered points
  const double *gx, *gy, *gz;  // [P]
  const uint32_t *gidx;        // [P] original index
  const uint32_t *cell_start;  // [n_cells + 1]
  GridDesc g;
  double max_dist;
  double t_star;  // m2 < t_star  <=>  sqrt_rn(m2) < max_dist (exact)
  // occlusion
  const float4 *nodes;
  const float4 *tris;
  int n_nodes;
  float scene_absmax;
  const uint32_t *tri_list;   // [C * tri_cap] leaf node indices (k_cam_trilist)
  const uint32_t *tri_count;  // [C]
  uint32_t tri_cap;
  uint32_t hoist_max;  // leaf lists up to this length (<= FU_HOIST) get per-camera records
  int packet_bvh;      // list overflow: 1 = lane = node packet traversal, 0 = per-ray stackless walk
  int endpoint_guard_rel;
  double block_length, block_inset;  // analytic occlusion (src/synthetic.rs:52-124)
  // plan + output.  A camera's rows are split into 2^parts_log2 contiguous blocks, one TICKET each (1, 2
  // or 4: more than one only when there are fewer cameras than persistent warps, so that the extra
  // per-ticket work runs on warps that would otherwise idle); slot = (camera << parts_log2) | part owns
  // its own scratch slice and visible count.  Part p holds rows [nrows*p >> log2, nrows*(p+1) >> log2).
  int parts_log2;
  // the plan also leaves every camera's trimmed row ranges behind (cameras with <= FU_ROWS rows), so that
  // the fused pass starts a camera with one coalesced load instead of recomputing them
  uint2 *rows;          // [C * FU_ROWS] (start, end) of row r of the camera, r = (z - lo.z) * ny + (y - lo.y)
  uint32_t *row_count;  // [C] number of rows; 0 = nothing to scan; FU_ROWS_MANY = more than FU_ROWS (recompute)
  uint32_t *ev_count;         // [slots+1] points on the slot's rows (k_cam_plan), then its exclusive scan
  uint32_t *scratch_idx;      // visible point indices, slot s at [ev_off[s], ev_off[s] + vis_count[s])
  uint64_t scratch_cap;       // entries scratch_idx holds (a slice beyond it raises counters[12] bit 0)
  uint32_t *vis_count;        // [slots+1]
  unsigned long long *counters;  // [1] pairs evaluated, [2] list entries / nodes, [3] warp triangle tests,
                                 // [4] candidates (rays), [5] scratch slice overflow flag, [7] camera ticket,
                                 // [8]-[11] unused;
                                 // [12] optimistic-launch flags (FU_FLAG_*): the host sized a buffer or chose a
                                 // kernel variant from the previous pass and this pass does not fit
};
enum { FU_FLAG_SCRATCH = 1, FU_FLAG_NEED_WALK = 2, FU_FLAG_OUT = 4 };

// camera_cell_range / camera_row run in BOTH k_cam_plan (which sizes each camera's scratch slice) and
// k_visibility_fused (which scans the rows), so they must round identically in both inlined copies:
// every operation is an explicit round-to-nearest intrinsic that the compiler cannot contract.
// cells whose points can lie within max_dist of the centre; false = none
__device__ __forceinline__ bool camera_cell_range(const GridDesc &g, const double cc[3], double max_dist,
                                                  int lo[3], int hi[3]) {
  bool empty = !(max_dist > 0.0);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    // every point with |p - c| < max_dist has c_k - r - eps < p_k < c_k + r + eps, and grid_coord is
    // monotone, so [coord(a0), coord(a1)] holds its cell; eps covers the rounding of a0 / a1
    const double eps = dadd(dmul(1e-9, dadd(fabs(cc[k]), fabs(max_dist))), 1e-300);
    const double a0 = dsub(dsub(cc[k], max_dist), eps), a1 = dadd(dadd(cc[k], max_dist), eps);
    if (a0 > g.max_c[k] || a1 < g.min_c[k]) empty = true;  // ball misses the populated slab
    lo[k] = grid_coord(g, k, a0);
    hi[k] = grid_coord(g, k, a1);
  }
  if (!(cc[0] == cc[0] && cc[1] == cc[1] && cc[2] == cc[2])) empty = true;  // NaN centre sees nothing
  return !empty;
}

// ---- per-row trimming ---------------------------------------------------------------------------------
// A camera scans rows of x-contiguous cells.  Everything a visible point must satisfy that is LINEAR in
// x along a row trims the row's cell range before any point is read:
//   in front of the camera      pc.z = r2.p + tz <= 0                                (src/generate.rs:450)
//   inside the image            |f pc.x| <= -pc.z and |f pc.y| <= -pc.z, i.e. the four half-spaces
//                               (+-f r0 + r2).p + (+-f tx + tz) <= 0, (+-f r1 + r2).p + (+-f ty + tz) <= 0
//                               (src/generate.rs:454 with `project`, src/baproblem.rs:145-151; only when
//                               k1 = k2 = 0, otherwise the image bound is not a plane)
//   within max_dist             |x - cx| <= sqrt(R^2 - d^2), d = distance of the centre from the row's
//                               (y, z) rectangle
// All of it is conservative (slack of 1e-9 of the magnitudes involved against rounding of ~1e-16), the
// exact predicate still runs on every point that is read.

// trims [x0, x1] to the cells that can hold a point with nx*x + ny*y + nz*z + off <= 0 for y in [y0, y1],
// z in [z0, z1]; xr bounds |nx*x| over the camera's ball; false = nothing on this row qualifies
__device__ __forceinline__ bool trim_halfspace(const GridDesc &g, double cell_h, double nx, double ny, double nz,
                                               double off, double xr, double mag_floor, double y0, double y1,
                                               double z0, double z1, int &x0, int &x1) {
  // smallest value ny*y + nz*z + off can take on the row (0 * inf is avoided explicitly)
  const double my = ny == 0.0 ? 0.0 : dmul(ny, ny > 0.0 ? y0 : y1);
  const double mz = nz == 0.0 ? 0.0 : dmul(nz, nz > 0.0 ? z0 : z1);
  const double bmin = dadd(dadd(my, mz), off);
  const double mag = dadd(dadd(dadd(dadd(fabs(my), fabs(mz)), fabs(off)), xr), mag_floor);
  if (bmin == bmin && fabs(bmin) < INFINITY) {
    const double slack = dadd(dmul(1e-9, mag), 1e-300);
    if (xr <= slack) {
      if (bmin > dmul(2.0, slack)) return false;  // the whole row is outside
    } else {
      const double xlim = ddiv(-dsub(bmin, slack), nx);  // nx*x <= -(bmin - slack)
      if (xlim == xlim) {
        const double xs = dmul(1e-9, dadd(fabs(xlim), cell_h));
        if (nx > 0.0) {
          const double xe = dadd(xlim, xs);
          if (xe < g.lo[0]) return false;
          const int xc = grid_coord(g, 0, xe);
          x1 = xc < x1 ? xc : x1;
        } else {
          const double xe = dsub(xlim, xs);
          if (xe > g.max_c[0]) return false;
          const int xc = grid_coord(g, 0, xe);
          x0 = xc > x0 ? xc : x0;
        }
        if (x0 > x1) return false;
      }
    }
  }
  return true;
}

constexpr int FU_ROWS = 32;
constexpr uint32_t FU_ROWS_MANY = 0xffffffffu;

struct RowRange {
  uint32_t start, end;  // grid-ordered points [start, end) of the trimmed row; start >= end: nothing
};

// The trimmed point range of row (y, z) for the camera record c (15 doubles) with centre cc.  Runs in BOTH
// k_cam_plan (which sizes each camera's scratch slice) and k_visibility_fused (which scans the rows), so it
// must round identically in both inlined copies: every operation is an explicit round-to-nearest intrinsic
// that the compiler cannot contract.
__device__ __forceinline__ RowRange camera_row(const GridDesc &g, const uint32_t *__restrict__ cell_start,
                                               const double *c, const double cc[3], double max_dist,
                                               const int lo[3], const int hi[3], double cell_h, int y, int z) {
  RowRange r{0u, 0u};
  int x0 = lo[0], x1 = hi[0];
  // bounds of the row's cells in y and z; edge cells also hold the clamped coordinates, so they
  // extend to the data bounds
  const double sl = dmul(1e-6, cell_h);
  const double y0 = y == 0 ? g.min_c[1] : dsub(dadd(g.lo[1], dmul((double)y, cell_h)), sl);
  const double y1 = y == g.n[1] - 1 ? g.max_c[1] : dadd(dadd(g.lo[1], dmul((double)(y + 1), cell_h)), sl);
  const double z0 = z == 0 ? g.min_c[2] : dsub(dadd(g.lo[2], dmul((double)z, cell_h)), sl);
  const double z1 = z == g.n[2] - 1 ? g.max_c[2] : dadd(dadd(g.lo[2], dmul((double)(z + 1), cell_h)), sl);
  const double reach = dadd(fabs(cc[0]), fabs(max_dist));
  // the ball
  {
    const double dy = fmax(fmax(dsub(y0, cc[1]), dsub(cc[1], y1)), 0.0);
    const double dz = fmax(fmax(dsub(z0, cc[2]), dsub(cc[2], z1)), 0.0);
    const double rem = dsub(dmul(dmul(max_dist, max_dist), 1.000000001), dadd(dmul(dy, dy), dmul(dz, dz)));
    if (rem < 0.0) return r;
    if (rem == rem && rem < INFINITY) {
      const double w = dadd(dmul(dsqrt(rem), 1.000000001), dmul(1e-9, reach));
      const double xa = dsub(cc[0], w), xb = dadd(cc[0], w);
      if (xa > g.max_c[0] || xb < g.min_c[0]) return r;
      const int ca = grid_coord(g, 0, xa), cb = grid_coord(g, 0, xb);
      x0 = ca > x0 ? ca : x0;
      x1 = cb < x1 ? cb : x1;
      if (x0 > x1) return r;
    }
  }
  // magnitudes the rounding errors of the exact predicate scale with: (|f| + 1) (|R| |p| + |t|)
  const double f = c[12];
  const bool planar_image = c[13] == 0.0 && c[14] == 0.0 && fabs(f) < INFINITY;
  double rmax = 0.0;
#pragma unroll
  for (int k = 0; k < 12; ++k) rmax = fmax(rmax, fabs(c[k]));
  const double span = dadd(dadd(dadd(fabs(cc[0]), fabs(cc[1])), fabs(cc[2])), dmul(3.0, fabs(max_dist)));
  const double mag_floor = dmul(dadd(planar_image ? fabs(f) : 0.0, 1.0), dmul(rmax, dadd(span, 1.0)));
  // in front of the camera
  if (!trim_halfspace(g, cell_h, c[2], c[5], c[8], c[11], dmul(fabs(c[2]), reach), mag_floor, y0, y1, z0, z1, x0, x1))
    return r;
  if (planar_image) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int row = k >> 1;  // 0: u (camera x), 1: v (camera y)
      const double sf = (k & 1) ? -f : f;
      const double nx = dadd(dmul(sf, c[row]), c[2]), ny = dadd(dmul(sf, c[3 + row]), c[5]);
      const double nz = dadd(dmul(sf, c[6 + row]), c[8]), off = dadd(dmul(sf, c[9 + row]), c[11]);
      if (!trim_halfspace(g, cell_h, nx, ny, nz, off, dmul(fabs(nx), reach), mag_floor, y0, y1, z0, z1, x0, x1))
        return r;
    }
  }
  const uint32_t rowbase = ((uint32_t)z * g.n[1] + y) * g.n[0];
  r.start = cell_start[rowbase + x0];
  r.end = cell_start[rowbase + x1 + 1];
  return r;
}

// The cull predicate of src/generate.rs:450-454 with the two f64 divisions of `project` replaced by
// a CLASSIFICATION: 1/pc.z is taken from the f32 reciprocal (relative error < 2e-7), (u, v) follow
// in f64 with a propagated error bound, and only a pair whose |u| or |v| lies within that bound of
// the frustum edge (or whose magnitudes leave the f32 range, or NaN) runs the exact operation
// sequence.  The returned bool is therefore identical to cull_project_thr's; (u, v) themselves are
// produced later by `observe` for the visible pairs only.
__device__ __forceinline__ bool cull_predicate(const double *cam, V3 center, V3 p, double t_star) {
  const V3 d{dsub(center.x, p.x), dsub(center.y, p.y), dsub(center.z, p.z)};
  if (!(mag2(d) < t_star)) return false;
  // project_world, z row first (same operation order as mat_vec)
  const double pcz = dadd(dadd(dadd(dmul(cam[2], p.x), dmul(cam[5], p.y)), dmul(cam[8], p.z)), cam[11]);
  if (!(pcz <= 0.0)) return false;
  const double pcx = dadd(dadd(dadd(dmul(cam[0], p.x), dmul(cam[3], p.y)), dmul(cam[6], p.z)), cam[9]);
  const double pcy = dadd(dadd(dadd(dmul(cam[1], p.x), dmul(cam[4], p.y)), dmul(cam[7], p.z)), cam[10]);
  const double f = cam[12], k1 = cam[13], k2 = cam[14];
  const double az = fabs(pcz);
  if (az > 1e-30 && az < 1e30) {
    const double iz = (double)__frcp_rn(__double2float_rn(pcz));
    const double a = pcx * iz, b = pcy * iz;  // -(p_) up to 2e-7; only magnitudes matter below
    double ua, va, bu, bv;
    if (k1 == 0.0 && k2 == 0.0) {
      ua = fabs(f * a);
      va = fabs(f * b);
      bu = 2e-6 * ua;
      bv = 2e-6 * va;
    } else {
      const double m2p = a * a + b * b;
      const double r = 1.0 + k1 * m2p + k2 * (m2p * m2p);
      const double rb = 1.0 + fabs(k1) * m2p + fabs(k2) * (m2p * m2p);
      ua = fabs(f * r * a);
      va = fabs(f * r * b);
      bu = 2e-6 * fabs(f * a) * rb;
      bv = 2e-6 * fabs(f * b) * rb;
    }
    if (ua <= 1.0 - bu && va <= 1.0 - bv) return true;  // NaN falls through to the exact path
    if (ua > 1.0 + bu || va > 1.0 + bv) return false;
  }
  double u, v;
  project(f, k1, k2, V3{pcx, pcy, pcz}, u, v);
  return u >= -1.0 && u <= 1.0 && v >= -1.0 && v <= 1.0;
}

// out-of-line copy for the fused kernel: called once per 32 rows, and kept out of the register
// allocation of its 64-register hot loops (same operations, same results)
__device__ __noinline__ RowRange camera_row_call(const GridDesc &g, const uint32_t *__restrict__ cell_start,
                                                 const double *c, const double *cc, double max_dist, const int *lo,
                                                 const int *hi, double cell_h, int y, int z) {
  return camera_row(g, cell_start, c, cc, max_dist, lo, hi, cell_h, y, z);
}

// ---- plan -------------------------------------------------------------------------------------------
// one thread per camera, rows in sequence (a warp per camera with lane = row leaves most lanes idle and
// measured 0.19 ms at cfg4 against 0.03 ms for this form)
__global__ void __launch_bounds__(128, 5) k_cam_plan(FusedArgs a) {
  const uint64_t cam = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int S = 1 << a.parts_log2;
  unsigned long long n0 = 0, n1 = 0, n2 = 0, n3 = 0;
  if (cam < a.C) {
    const double cc[3] = {a.cen_x[cam], a.cen_y[cam], a.cen_z[cam]};
    int lo[3], hi[3];
    a.row_count[cam] = 0u;
    if (camera_cell_range(a.g, cc, a.max_dist, lo, hi)) {
      double c[15];
#pragma unroll
      for (int k = 0; k < 15; ++k) c[k] = a.cams[15 * cam + k];
      const double cell_h = ddiv(1.0, a.g.inv_h);
      const int nrows = (hi[1] - lo[1] + 1) * (hi[2] - lo[2] + 1);
      const bool keep = nrows <= FU_ROWS;
      a.row_count[cam] = keep ? (uint32_t)nrows : FU_ROWS_MANY;
      int ri = 0;
      for (int z = lo[2]; z <= hi[2]; ++z)
        for (int y = lo[1]; y <= hi[1]; ++y, ++ri) {
          const RowRange rr = camera_row(a.g, a.cell_start, c, cc, a.max_dist, lo, hi, cell_h, y, z);
          if (keep) a.rows[cam * FU_ROWS + ri] = make_uint2(rr.start, rr.end);
          if (rr.end > rr.start) {
            const unsigned long long m = rr.end - rr.start;
            int part = 0;  // the block of rows ri falls in (same split as k_visibility_fused)
            for (int q = 1; q < S; ++q)
              if (ri >= (nrows * q) >> a.parts_log2) part = q;
            n0 += part == 0 ? m : 0ull;
            n1 += part == 1 ? m : 0ull;
            n2 += part == 2 ? m : 0ull;
            n3 += part == 3 ? m : 0ull;
          }
        }
    }
    uint32_t *out = a.ev_count + (cam << a.parts_log2);  // each < 2^32 (<= P)
    out[0] = (uint32_t)n0;
    if (S > 1) out[1] = (uint32_t)n1;
    if (S > 2) {
      out[2] = (uint32_t)n2;
      out[3] = (uint32_t)n3;
    }
  }
  if (cam == a.C) a.ev_count[cam << a.parts_log2] = 0u;  // closes the scan
  // 64-bit total, so the host can tell when the u32 scan would wrap
  unsigned long long n = n0 + n1 + n2 + n3;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(&a.counters[1], n);
}

// ---- warp-private radix sort of a camera's visible point indices (k_sort_write) -----------------------
struct SortWriteArgs {
  const uint32_t *ev_off;     // [C+1] scratch slice starts
  const uint32_t *seg_off;    // [C+1] exclusive scan of vis_count = CSR offsets
  uint64_t C;
  const uint32_t *scratch_idx;
  const double *cams;
  const double *p_aos;  // xyz records, original point order
  uint64_t *out_offsets;
  uint32_t *out_idx;
  double2 *out_uv;
  int key_bits;    // bits of the largest point index: the radix passes cover exactly these
  int parts_log2;  // slots per camera (FusedArgs::parts_log2); ev_off / seg_off are indexed by slot
  uint64_t out_cap;            // observations out_idx / out_uv hold
  unsigned long long *flags;   // counters[12]: FU_FLAG_OUT when a camera's records do not fit
};

// a camera's visible list is the concatenation of its slots' scratch slices
struct CamSlices {
  uint32_t base, n;         // CSR segment of the camera
  uint32_t sub[4], eo[4];   // slot q starts at list position sub[q] and at scratch_idx[eo[q]]
};
// MULTI = false: one slot per camera (parts_log2 == 0), the common case, compiled without the slot search
template <bool MULTI>
__device__ __forceinline__ CamSlices cam_slices(const SortWriteArgs &s, uint64_t cam) {
  CamSlices cs;
  if (!MULTI) {
    cs.base = s.seg_off[cam];
    cs.n = s.seg_off[cam + 1] - cs.base;
    cs.sub[0] = 0u;
    cs.eo[0] = s.ev_off[cam];
    return cs;
  }
  const uint64_t slot0 = cam << s.parts_log2;
  const int S = 1 << s.parts_log2;
  cs.base = s.seg_off[slot0];
  cs.n = s.seg_off[slot0 + S] - cs.base;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    cs.sub[q] = q < S ? s.seg_off[slot0 + q] - cs.base : 0xffffffffu;
    cs.eo[q] = q < S ? s.ev_off[slot0 + q] : 0u;
  }
  return cs;
}
template <bool MULTI>
__device__ __forceinline__ uint32_t cam_key(const SortWriteArgs &s, const CamSlices &cs, uint32_t t) {
  if (!MULTI) return s.scratch_idx[cs.eo[0] + t];
  uint32_t sub = cs.sub[0], eo = cs.eo[0];
#pragma unroll
  for (int q = 1; q < 4; ++q)
    if (t >= cs.sub[q]) {
      sub = cs.sub[q];
      eo = cs.eo[q];
    }
  return s.scratch_idx[eo + (t - sub)];
}

constexpr uint32_t SW_WARP_MAX = 1024;   // one warp per camera
constexpr uint32_t SW_BLOCK_MAX = 4096;  // shared-memory sort, one block per camera

constexpr int SW_WARPS = 4;
constexpr int SW_RADIX_BITS = 8;
constexpr int SW_BINS = 1 << SW_RADIX_BITS;

// sorted[] is indexed with one pad word per 32 (i + i/32), so that the lane*E + r stores and the
// consecutive reads are both free of bank conflicts
__device__ __forceinline__ uint32_t sw_pad(uint32_t i) { return i + (i >> 5); }

// Warp-private LSD radix sort of n <= 32*E keys, 8-bit digits.  Keys live in registers in list order
// (a[r] = key r*32 + lane); one pass = digit histogram in shared memory (ATOMS), exclusive scan of the
// 256 counters (8 per lane + one warp scan), then a stable scatter chunk by chunk: the rank of a key
// among the equal digits of its chunk is popc(__match_any_sync & lanes below), the chunk's first lane
// per digit advances the counter with one shared-memory atomic and hands the old value to its peers
// by shuffle.  About 0.4k warp instructions per pass at n = 532 against ~3k for the 1024-key bitonic network
// this replaces (profiles/r01h: k_sort_write spent 878 M warp instructions, 16.5 per observation).  The sorted
// keys end up in `sorted` (padded layout).
//   * A digit on which all keys agree needs no pass (common for the top digit: a camera's points are usually
//     close in index).  One OR and one AND reduction over the keys tell which digits vary, so a skipped pass
//     costs nothing (until r02x its histogram was built first and then found to have a single bin).
//   * The scatter handles FOUR chunks at a time: four MATCHes, then the four leaders' atomics, then four
//     shuffles + stores.  Chunk by chunk the chain MATCH -> ATOMS -> SHFL -> STS exposed its ~120 cycles of
//     latency 17 times per pass: 45 % of the kernel's stall samples sat on the instruction after a MATCH or an
//     ATOMS (profiles/r02w_sass_dynamic_sort_write.txt, short_scoreboard 7.6 warps per issue).
template <int E, bool MULTI>
__device__ __forceinline__ void sort_warp_to_smem(const SortWriteArgs &s, const CamSlices &cs, int lane,
                                                  uint32_t *sorted, uint32_t *hist) {
  static_assert(E % 4 == 0, "the scatter takes four chunks at a time");
  const uint32_t n = cs.n;
  const int key_bits = s.key_bits;
  uint32_t a[E];
  uint32_t v_or = 0u, v_and = 0xffffffffu;
#pragma unroll
  for (int r = 0; r < E; ++r) {
    const uint32_t t = r * 32 + lane;
    a[r] = 0xffffffffu;
    if (t < n) {
      a[r] = cam_key<MULTI>(s, cs, t);
      v_or |= a[r];
      v_and &= a[r];
    }
  }
  // bits in which the camera's keys differ (warp-uniform; lanes without keys contribute the neutral elements)
  const uint32_t varying = __reduce_or_sync(0xffffffffu, v_or) ^ __reduce_and_sync(0xffffffffu, v_and);
  const unsigned lt = (1u << lane) - 1u;
  bool in_smem = false;
  for (int shift = 0; shift < key_bits; shift += SW_RADIX_BITS) {
    if (((varying >> shift) & (SW_BINS - 1)) == 0u) continue;  // every key has the same digit: order unchanged
#pragma unroll
    for (int k = 0; k < SW_BINS / 32; ++k) hist[k * 32 + lane] = 0u;
    __syncwarp();
#pragma unroll
    for (int r = 0; r < E; ++r)
      if ((uint32_t)(r * 32 + lane) < n) atomicAdd(&hist[(a[r] >> shift) & (SW_BINS - 1)], 1u);
    __syncwarp();
    // exclusive scan: lane owns counters [8*lane, 8*lane + 8)
    uint32_t c[SW_BINS / 32];
    uint32_t sum = 0;
#pragma unroll
    for (int k = 0; k < SW_BINS / 32; ++k) {
      c[k] = hist[lane * (SW_BINS / 32) + k];
      sum += c[k];
    }
    uint32_t pre = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, pre, o);
      if (lane >= o) pre += v;
    }
    pre -= sum;
    __syncwarp();
#pragma unroll
    for (int k = 0; k < SW_BINS / 32; ++k) {
      hist[lane * (SW_BINS / 32) + k] = pre;
      pre += c[k];
    }
    __syncwarp();
#pragma unroll
    for (int r0 = 0; r0 < E; r0 += 4) {
      if ((uint32_t)(r0 * 32) < n) {  // warp-uniform
        uint32_t d[4], old[4];
        unsigned peers[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const bool valid = (uint32_t)((r0 + g) * 32 + lane) < n;
          d[g] = valid ? (a[r0 + g] >> shift) & (SW_BINS - 1) : (uint32_t)SW_BINS;  // padding keeps to itself
          peers[g] = __match_any_sync(0xffffffffu, d[g]);
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          old[g] = 0u;
          if (d[g] != (uint32_t)SW_BINS && lane == __ffs(peers[g]) - 1)
            old[g] = atomicAdd(&hist[d[g]], (uint32_t)__popc(peers[g]));  // warp-aggregated
          __syncwarp();  // a later chunk's leaders advance the counters after this chunk's (stable order)
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const uint32_t base = __shfl_sync(0xffffffffu, old[g], __ffs(peers[g]) - 1);
          if (d[g] != (uint32_t)SW_BINS) sorted[sw_pad(base + __popc(peers[g] & lt))] = a[r0 + g];
        }
      }
    }
    __syncwarp();
    in_smem = true;
    if (shift + SW_RADIX_BITS < key_bits && (varying >> (shift + SW_RADIX_BITS)) != 0u) {  // another pass follows
#pragma unroll
      for (int r = 0; r < E; ++r) {
        const uint32_t t = r * 32 + lane;
        if (t < n) a[r] = sorted[sw_pad(t)];
      }
      __syncwarp();
    }
  }
  if (!in_smem) {
#pragma unroll
    for (int r = 0; r < E; ++r) {
      const uint32_t t = r * 32 + lane;
      if (t < n) sorted[sw_pad(t)] = a[r];
    }
  }
}

// ---- the fused pass ---------------------------------------------------------------------------------
// Warps per CTA.  Four-warp CTAs, 7 per SM, give the kernel 72 registers at 28 warps per SM; eight-warp CTAs (until
// r02y) 64 registers at 32.  At 64 the prefetched coordinates of the next chunk and the camera centre lived in local
// memory — the spill store right behind the prefetch loads waited for them to arrive (6 % of the kernel's stall
// samples, profiles/r02x_sass_dynamic_fused.txt) — at 72 they stay in registers: 2.38 -> 2.31 ms at cfg4 on the
// same box (profiles/r02y_ab_same_box.txt).  -DC2B_FU_WARPS=8 restores the old shape.
#ifndef C2B_FU_WARPS
#define C2B_FU_WARPS 4
#endif
constexpr int FU_WARPS = C2B_FU_WARPS;
// CTAs per SM for a variant declared with m CTAs of EIGHT warps (the template argument MIN_CTAS)
constexpr int fu_min_ctas(int m) { return FU_WARPS == 8 ? m : (m == 4 ? 7 : 2 * m); }
constexpr int FU_RESIDENT_WARPS = FU_WARPS == 8 ? 32 : 28;  // per SM, of the default (mesh) variant
constexpr int FU_STAGE = 64;

enum { FU_OCC_MESH = 0, FU_OCC_NONE = 1, FU_OCC_ANALYTIC = 2 };

// warp-wide float min / max in ONE instruction: sm_100a's redux.sync.{min,max}.f32 (CREDUX.MIN.F32 / .MAX.F32,
// result in a uniform register).  Until r02w the floats went through order-preserving integer images for the
// integer REDUX (shift, xor before; compare, select, xor after: ~10 instructions per reduction, 125 per packet
// for the twelve bounds = 12 % of the kernel's warp instructions at cfg4, profiles/r02j_sass_dynamic_fused.txt).
// NaN inputs are ignored unless every lane holds one; -0 < +0.  The bounds are identical either way.
__device__ __forceinline__ float warp_min_f32(float v) {
  float r;
  asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ float warp_max_f32(float v) {
  float r;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}

__device__ __forceinline__ TriRec load_rec(const float4 *rec, int k) {
  const float4 r0 = rec[3 * k], r1 = rec[3 * k + 1], r2 = rec[3 * k + 2];
  TriRec t;
  t.ux = r0.x; t.uy = r0.y; t.uz = r0.z;
  t.vx = r0.w; t.vy = r1.x; t.vz = r1.y;
  t.wx = r1.z; t.wy = r1.w; t.wz = r2.x;
  t.T = r2.y;
  return t;
}

// range of n . d over the direction box [dlo, dhi] (interval arithmetic; the caller adds slack)
__device__ __forceinline__ void dot_range(float nx, float ny, float nz, float lx, float ly, float lz, float hx,
                                          float hy, float hz, float &mn, float &mx) {
  const float ax = nx * lx, bx = nx * hx, ay = ny * ly, by = ny * hy, az = nz * lz, bz = nz * hz;
  mn = fminf(ax, bx) + fminf(ay, by) + fminf(az, bz);
  mx = fmaxf(ax, bx) + fmaxf(ay, by) + fmaxf(az, bz);
}

// ---- per-camera triangle records ("hoisted" mode, the camera's leaf list has <= FU_HOIST entries) ----
// Every ray of a camera starts at the same origin, so the origin-relative record of a triangle is a
// per-(camera, triangle) constant.  The warp computes the records of its camera's whole leaf list
// once, lane = triangle, into shared memory (SoA: four float4 planes of FU_HOIST entries, so that
// both the lane = triangle reads and the broadcast reads of the test loop are conflict-free):
//   plane 0 {ux uy uz vx}  plane 1 {vy vz wx wy}  plane 2 {wz T lo.x lo.y}  plane 3 {lo.z hi.x hi.y hi.z}
constexpr int FU_HOIST = 64;

// (l0, l1: this lane's list entries lane and lane + 32, loaded by the caller together with the camera's other
// per-camera words so that their latencies overlap)
__device__ __forceinline__ void hoist_records(const FusedArgs &a, uint32_t l0, uint32_t l1,
                                              uint32_t n_list, float ox, float oy, float oz, float4 *rec,
                                              int lane) {
  static_assert(FU_HOIST == 64, "two list entries per lane");
  for (uint32_t j = lane; j < n_list; j += 32) {
    const uint32_t node = j < 32 ? l0 : l1;
    const float4 lo = __ldg(&a.nodes[2 * node]);
    const float4 hi = __ldg(&a.nodes[2 * node + 1]);
    const int slot = __float_as_int(hi.w);
    const float4 v0 = __ldg(&a.tris[3 * slot]);
    const float4 v1 = __ldg(&a.tris[3 * slot + 1]);
    const float4 v2 = __ldg(&a.tris[3 * slot + 2]);
    const TriRec t = tri_record(ox, oy, oz, v0.x, v0.y, v0.z, v1.x, v1.y, v1.z, v2.x, v2.y, v2.z);
    rec[j] = make_float4(t.ux, t.uy, t.uz, t.vx);
    rec[FU_HOIST + j] = make_float4(t.vy, t.vz, t.wx, t.wy);
    rec[2 * FU_HOIST + j] = make_float4(t.wz, t.T, lo.x, lo.y);
    rec[3 * FU_HOIST + j] = make_float4(lo.z, hi.x, hi.y, hi.z);
  }
  __syncwarp();
}

__device__ __forceinline__ TriRec unpack_rec(float4 r0, float4 r1, float4 r2) {
  TriRec t;
  t.ux = r0.x; t.uy = r0.y; t.uz = r0.z;
  t.vx = r0.w; t.vy = r1.x; t.vz = r1.y;
  t.wx = r1.z; t.wy = r1.w; t.wz = r2.x;
  t.T = r2.y;
  return t;
}

// can any direction of the box [dl, dh] give edge functions that are all >= 0 or all <= 0?
__device__ __forceinline__ bool direction_box_may_hit(const TriRec &t, float dlx, float dly, float dlz,
                                                      float dhx, float dhy, float dhz) {
  float umn, umx, vmn, vmx, wmn, wmx;
  dot_range(t.ux, t.uy, t.uz, dlx, dly, dlz, dhx, dhy, dhz, umn, umx);
  dot_range(t.vx, t.vy, t.vz, dlx, dly, dlz, dhx, dhy, dhz, vmn, vmx);
  dot_range(t.wx, t.wy, t.wz, dlx, dly, dlz, dhx, dhy, dhz, wmn, wmx);
  // slack: rounding of the per-ray FMA chain and of the interval sums, a few ulps of sum |n_k d_k|
  const float su = 2e-6f * (fabsf(t.ux) + fabsf(t.uy) + fabsf(t.uz));
  const float sv = 2e-6f * (fabsf(t.vx) + fabsf(t.vy) + fabsf(t.vz));
  const float sw = 2e-6f * (fabsf(t.wx) + fabsf(t.wy) + fabsf(t.wz));
  const bool some_neg = umx < -su || vmx < -sv || wmx < -sw;  // an edge function < 0 for every ray
  const bool some_pos = umn > su || vmn > sv || wmn > sw;     // an edge function > 0 for every ray
  return !(some_neg && some_pos);                             // NaN bounds keep the triangle
}

// bounding box of a packet's ray segments (origin + end points, conservatively padded) and of its
// directions, reduced over the warp with one CREDUX.F32 each
struct PacketBounds {
  float blx, bly, blz, bhx, bhy, bhz;  // segments
  float dlx, dly, dlz, dhx, dhy, dhz;  // directions
};


__device__ __forceinline__ PacketBounds packet_bounds(const Ray &ray, bool alive, float ox, float oy,
                                                      float oz, float scene_absmax) {
  float lx = INFINITY, ly = INFINITY, lz = INFINITY, hx = -INFINITY, hy = -INFINITY, hz = -INFINITY;
  float dlx = INFINITY, dly = INFINITY, dlz = INFINITY, dhx = -INFINITY, dhy = -INFINITY, dhz = -INFINITY;
  if (alive) {
    const float pad = conservative_pad(ox, oy, oz, scene_absmax) + 4e-6f * ray.tfar;
    const float ex = fmaf(ray.dx, ray.tfar, ox), ey = fmaf(ray.dy, ray.tfar, oy), ez = fmaf(ray.dz, ray.tfar, oz);
    lx = fminf(ox, ex) - pad;
    ly = fminf(oy, ey) - pad;
    lz = fminf(oz, ez) - pad;
    hx = fmaxf(ox, ex) + pad;
    hy = fmaxf(oy, ey) + pad;
    hz = fmaxf(oz, ez) + pad;
    dlx = dhx = ray.dx;
    dly = dhy = ray.dy;
    dlz = dhz = ray.dz;
  }
  PacketBounds b;
  b.blx = warp_min_f32(lx);
  b.bly = warp_min_f32(ly);
  b.blz = warp_min_f32(lz);
  b.bhx = warp_max_f32(hx);
  b.bhy = warp_max_f32(hy);
  b.bhz = warp_max_f32(hz);
  b.dlx = warp_min_f32(dlx);
  b.dly = warp_min_f32(dly);
  b.dlz = warp_min_f32(dlz);
  b.dhx = warp_max_f32(dhx);
  b.dhy = warp_max_f32(dhy);
  b.dhz = warp_max_f32(dhz);
  return b;
}

__device__ __forceinline__ bool box_meets_packet(const PacketBounds &b, float4 lo, float4 hi) {
  // written so that NaN compares keep the box (conservative)
  return !(lo.x > b.bhx || hi.x < b.blx || lo.y > b.bhy || hi.y < b.bly || lo.z > b.bhz || hi.z < b.blz);
}

// lane = triangle: lanes with `want` load triangle `slot`, build its record for the origin, drop it
// if the direction box cannot hit it, and park the survivors' records in rec[0..3*cnt);
// then lane = ray: every record is tested.  `am` = the rays of the packet that are still unoccluded, as a
// warp-uniform lane mask (one VOTE + one logic op per pair of tests; per-lane alive / occluded flags cost a dozen
// select / pack instructions per pair).  Returns false when no ray of the packet is left alive.
template <bool COUNT>
__device__ __forceinline__ bool test_leaf_chunk(const FusedArgs &a, const PacketBounds &pb, int slot, bool want,
                                                const Ray &ray, unsigned &am, float ox, float oy,
                                                float oz, float4 *rec, int lane, unsigned &n_tri) {
  TriRec t;
  if (want) {
    const float4 v0 = __ldg(&a.tris[3 * slot]);
    const float4 v1 = __ldg(&a.tris[3 * slot + 1]);
    const float4 v2 = __ldg(&a.tris[3 * slot + 2]);
    t = tri_record(ox, oy, oz, v0.x, v0.y, v0.z, v1.x, v1.y, v1.z, v2.x, v2.y, v2.z);
    want = direction_box_may_hit(t, pb.dlx, pb.dly, pb.dlz, pb.dhx, pb.dhy, pb.dhz);
  }
  const unsigned m = __ballot_sync(0xffffffffu, want);
  if (m == 0u) return true;
  if (want) {
    float4 *r = rec + 3 * __popc(m & ((1u << lane) - 1u));
    r[0] = make_float4(t.ux, t.uy, t.uz, t.vx);
    r[1] = make_float4(t.vy, t.vz, t.wx, t.wy);
    r[2] = make_float4(t.wz, t.T, 0.0f, 0.0f);
  }
  __syncwarp();
  const int cnt = __popc(m);
  if (COUNT) n_tri += cnt;
  int k = 0;
  for (; k + 1 < cnt; k += 2) {
    const TriRec t0 = load_rec(rec, k), t1 = load_rec(rec, k + 1);
    const bool h0 = ray_tri_record(ray.dx, ray.dy, ray.dz, ray.tfar, t0);
    const bool h1 = ray_tri_record(ray.dx, ray.dy, ray.dz, ray.tfar, t1);
    am &= ~__ballot_sync(0xffffffffu, h0 | h1);
    if (am == 0u) break;
  }
  if (am != 0u && (cnt & 1)) {
    const TriRec t0 = load_rec(rec, cnt - 1);
    am &= ~__ballot_sync(0xffffffffu, ray_tri_record(ray.dx, ray.dy, ray.dz, ray.tfar, t0));
  }
  __syncwarp();
  return am != 0u;
}

// list-driven any-hit for a packet of rays that share the origin (ox, oy, oz).  Returns true when
// this lane's ray is occluded.
//
// Two conservative filters run with lane = triangle before any ray is tested: (1) the leaf box must
// overlap the bounding box of the packet's ray segments; (2) with the record in hand, the three edge
// functions are bounded over the packet's direction box [dlo, dhi]: a ray can only hit if all three
// are >= 0 or all three are <= 0, so a triangle for which some edge function is negative on the whole
// box AND some edge function is positive on the whole box cannot be hit by any ray of the packet.
template <bool COUNT>
__device__ __forceinline__ bool packet_any_hit(const FusedArgs &a, const uint32_t *__restrict__ mylist,
                                               uint32_t n_list, const Ray &ray, bool have, float ox,
                                               float oy, float oz, float4 *rec, bool hoisted, int lane,
                                               unsigned &n_vis, unsigned &n_tri) {
  const bool alive = have && (ray.tfar >= 0.0f) && (ray.dx == ray.dx) && (ray.dy == ray.dy) && (ray.dz == ray.dz);
  unsigned am = __ballot_sync(0xffffffffu, alive);  // rays not yet known to be occluded (warp-uniform)
  if (am == 0u) return false;
  const PacketBounds pb = packet_bounds(ray, alive, ox, oy, oz, a.scene_absmax);
  if (hoisted) {
    for (uint32_t base = 0; base < n_list; base += 32) {
      const uint32_t j = base + lane;
      bool overlap = false;
      if (j < n_list) {
        const float4 r2 = rec[2 * FU_HOIST + j], r3 = rec[3 * FU_HOIST + j];
        overlap = box_meets_packet(pb, make_float4(r2.z, r2.w, r3.x, 0.0f), make_float4(r3.y, r3.z, r3.w, 0.0f));
        if (overlap)
          overlap = direction_box_may_hit(unpack_rec(rec[j], rec[FU_HOIST + j], r2), pb.dlx, pb.dly, pb.dlz, pb.dhx,
                                          pb.dhy, pb.dhz);
      }
      unsigned m = __ballot_sync(0xffffffffu, overlap);
      if (COUNT) {
        n_vis += min(32u, n_list - base);
        n_tri += __popc(m);
      }
      // the records' shared-memory address as ONE opaque 32-bit register: left to itself the compiler
      // re-derives it from %tid and the shared window (ten instructions) for every second triangle
      uint32_t rk_s = (uint32_t)__cvta_generic_to_shared(rec + base);
      asm volatile("" : "+r"(rk_s));
      const float4 *rk = reinterpret_cast<const float4 *>(__cvta_shared_to_generic((size_t)rk_s));
      while (m) {
        const int k0 = __ffs(m) - 1;
        m &= m - 1;
        bool h = ray_tri_record(ray.dx, ray.dy, ray.dz, ray.tfar, unpack_rec(rk[k0], rk[FU_HOIST + k0], rk[2 * FU_HOIST + k0]));
        if (m) {
          const int k1 = __ffs(m) - 1;
          m &= m - 1;
          h |= ray_tri_record(ray.dx, ray.dy, ray.dz, ray.tfar, unpack_rec(rk[k1], rk[FU_HOIST + k1], rk[2 * FU_HOIST + k1]));
        }
        // (a lane that was never alive may report a "hit" of its placeholder ray: its bit is clear already)
        am &= ~__ballot_sync(0xffffffffu, h);
        if (am == 0u) return alive;  // every live ray of the packet is occluded
      }
    }
    return alive && !((am >> lane) & 1u);
  }
  for (uint32_t base = 0; base < n_list; base += 32) {
    const uint32_t j = base + lane;
    bool overlap = false;
    int slot = 0;
    if (j < n_list) {
      const uint32_t node = mylist[j];
      const float4 lo = __ldg(&a.nodes[2 * node]);
      const float4 hi = __ldg(&a.nodes[2 * node + 1]);
      overlap = box_meets_packet(pb, lo, hi);
      slot = __float_as_int(hi.w);
    }
    if (COUNT) n_vis += min(32u, n_list - base);
    if (!test_leaf_chunk<COUNT>(a, pb, slot, overlap, ray, am, ox, oy, oz, rec, lane, n_tri)) break;
  }
  return alive && !((am >> lane) & 1u);
}

// ---- packet traversal of the BVH, lane = node --------------------------------------------------------
// For cameras whose leaf list overflows (fine meshes).  The warp keeps a LIFO of node indices in
// shared memory; each step pops up to 32 nodes, every lane tests ONE node's box against the
// packet's segment box (two LDG.128, six compares — no per-ray slab test), overlapping leaves go to
// a pending-leaf buffer, overlapping internal nodes push both children (left = node + 1, right =
// -hi.w - 1).  Whenever 32 leaves are pending (or the LIFO is empty) they are resolved with
// test_leaf_chunk.  The per-warp 4 KB region is split: records [0, 96) float4, pending leaves 64 u32,
// LIFO FU_LIFO u32.  Returns 2 if the LIFO would overflow (the caller falls back to the per-ray
// stackless walk, which needs no memory), else 0 / 1 = this lane's ray is occluded.
constexpr int FU_LIFO = 576;

template <bool COUNT>
__device__ __forceinline__ int packet_bvh_hit(const FusedArgs &a, const Ray &ray, bool have, float ox, float oy,
                                              float oz, float4 *region, int lane, unsigned &n_vis,
                                              unsigned &n_tri) {
  const bool alive = have && (ray.tfar >= 0.0f) && (ray.dx == ray.dx) && (ray.dy == ray.dy) && (ray.dz == ray.dz);
  unsigned am = __ballot_sync(0xffffffffu, alive);  // rays not yet known to be occluded (warp-uniform)
  if (am == 0u) return 0;
  const PacketBounds pb = packet_bounds(ray, alive, ox, oy, oz, a.scene_absmax);
  float4 *rec = region;
  uint32_t *pending = reinterpret_cast<uint32_t *>(region + 96);
  uint32_t *lifo = pending + 64;
  int sp = 1, np = 0;
  if (lane == 0) lifo[0] = 0u;
  __syncwarp();
  while (sp > 0 || np > 0) {
    if (sp > 0 && np <= 32) {
      const int take = sp < 32 ? sp : 32;
      const bool mine = lane < take;
      bool leaf = false, inner = false;
      int slot = 0;
      uint32_t node = 0, right = 0;
      if (mine) {
        node = lifo[sp - take + lane];
        const float4 lo = __ldg(&a.nodes[2 * node]);
        const float4 hi = __ldg(&a.nodes[2 * node + 1]);
        if (box_meets_packet(pb, lo, hi)) {
          slot = __float_as_int(hi.w);
          leaf = slot >= 0;
          inner = !leaf;
          right = (uint32_t)(-slot - 1);
        }
      }
      __syncwarp();  // every lane has read its node before anyone pushes into the same slots
      sp -= take;
      if (COUNT) n_vis += take;
      const unsigned lm = __ballot_sync(0xffffffffu, leaf), im = __ballot_sync(0xffffffffu, inner);
      if (sp + 2 * __popc(im) > FU_LIFO) return 2;
      const unsigned lt = (1u << lane) - 1u;
      if (leaf) pending[np + __popc(lm & lt)] = (uint32_t)slot;
      if (inner) {
        const int pos = sp + 2 * __popc(im & lt);
        lifo[pos] = node + 1u;
        lifo[pos + 1] = right;
      }
      np += __popc(lm);
      sp += 2 * __popc(im);
      __syncwarp();
    } else {
      const int cnt = np < 32 ? np : 32;
      const bool want = lane < cnt;
      const int slot = want ? (int)pending[np - cnt + lane] : 0;
      np -= cnt;
      if (!test_leaf_chunk<COUNT>(a, pb, slot, want, ray, am, ox, oy, oz, rec, lane, n_tri)) break;
    }
  }
  return alive && !((am >> lane) & 1u) ? 1 : 0;
}

// Persistent warps: every warp draws the next camera from a global ticket (counters[7]), so a warp
// that drew a cheap camera (city edge, few points in range) immediately gets another one and no
// warp idles waiting for the slowest camera of its block.
// WALK = the BVH traversals for cameras whose leaf list overflowed are compiled in; the host picks
// the variant without them when k_cam_trilist reported no overflow (coarse meshes), which keeps
// their registers out of the list-driven fast path.
constexpr int FU_REGION_F4 = 4 * FU_HOIST;  // 4 KB

// a warp's shared memory: triangle records (hoisted: 4 planes x FU_HOIST; chunked: 32 x 3), the camera record,
// and the ring of FU_STAGE grid positions in which the survivors of the cull wait for their packet.  (Staging the
// coordinates as well, so that the ray set-up needs no second trip through L1, was measured: 48 KB of shared
// memory per CTA instead of 36 shrink L1, 3.11 ms against 3.07 ms at cfg4.)
template <bool MESH>
struct alignas(16) FuWarpSmem {
  float4 rec[MESH ? FU_REGION_F4 : 1];
  double cam[16];
  uint32_t stage[FU_STAGE];
};

template <int OCC, bool COUNT, int MIN_CTAS, bool WALK>
__global__ void __launch_bounds__(FU_WARPS * 32, fu_min_ctas(MIN_CTAS)) k_visibility_fused(FusedArgs a) {
  // One block of shared memory per warp (FuWarpSmem), addressed through ONE opaque 32-bit register: with three
  // separate arrays indexed by the warp number the compiler re-derived every address from %tid and the shared
  // window at each use (5-10 instructions, eight times per chunk / packet: profiles/r02w_sass_dynamic_fused.txt).
  typedef FuWarpSmem<OCC == FU_OCC_MESH> WarpSmem;
  __shared__ WarpSmem s_w[FU_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t w_s = (uint32_t)__cvta_generic_to_shared(&s_w[warp]);
  asm volatile("" : "+r"(w_s));
  WarpSmem *const w = reinterpret_cast<WarpSmem *>(__cvta_shared_to_generic((size_t)w_s));
  double *const c = w->cam;
  uint32_t *stage = w->stage;
  unsigned long long found_total = 0;
  unsigned n_vis_nodes = 0, n_tri = 0;
  const double cell_h = ddiv(1.0, a.g.inv_h);
  for (;;) {
    unsigned long long ticket = 0;
    if (lane == 0) ticket = atomicAdd(&a.counters[7], 1ull);
    const uint64_t slot = __shfl_sync(0xffffffffu, ticket, 0);
    const uint64_t cam = slot >> a.parts_log2;
    if (cam >= a.C) break;
    const int part = (int)(slot & ((1u << a.parts_log2) - 1u));
    __syncwarp();
    // everything that depends on the camera index only is loaded back to back, before the first use, so
    // that the round trips overlap (the per-camera set-up is a latency chain: 0.31 ms of the 3.08 ms at cfg4
    // before this and the stored row ranges, 0.16 ms after; profiles/shard_probe.py --max-dist 0.3)
    double creg = 0.0;
    if (lane < 15) creg = __ldg(&a.cams[15 * cam + lane]);
    const V3 cen{a.cen_x[cam], a.cen_y[cam], a.cen_z[cam]};
    const uint32_t planned_rows = a.row_count[cam];
    const uint32_t ev0 = a.ev_count[slot], ev1 = a.ev_count[slot + 1];
    const uint2 myrow = a.rows[cam * FU_ROWS + lane];  // meaningful for lane < planned_rows <= FU_ROWS
    uint32_t n_list = 0, l0 = 0, l1 = 0;
    const uint32_t *mylist = nullptr;
    if (OCC == FU_OCC_MESH) {
      n_list = a.tri_count[cam];
      mylist = a.tri_list + cam * a.tri_cap;
      if ((uint32_t)lane < a.tri_cap) l0 = mylist[lane];
      if ((uint32_t)lane + 32u < a.tri_cap) l1 = mylist[lane + 32];
    }
    if (lane < 15) c[lane] = creg;
    __syncwarp();
    // launched without waiting for the plan's totals (sizes and variant from the previous pass): a camera
    // whose slice lies beyond the scratch array, or that needs the BVH walk this variant was compiled without,
    // is skipped and flagged — the host then repeats the pass with exact sizes
    const bool misfit = (uint64_t)ev1 > a.scratch_cap || (OCC == FU_OCC_MESH && !WALK && n_list == TRILIST_OVERFLOW);
    if (misfit && lane == 0)
      atomicOr(&a.counters[12], (unsigned long long)((uint64_t)ev1 > a.scratch_cap ? FU_FLAG_SCRATCH : FU_FLAG_NEED_WALK));
    if (planned_rows == 0u || misfit) {  // nothing to scan (ball outside the data, NaN centre, ...)
      if (lane == 0) a.vis_count[slot] = 0;
      continue;
    }
    const float ox = d2f(cen.x), oy = d2f(cen.y), oz = d2f(cen.z);
    const bool hoisted = OCC == FU_OCC_MESH && n_list <= a.hoist_max;  // (OVERFLOW is 2^32 - 1)
    if (hoisted) hoist_records(a, l0, l1, n_list, ox, oy, oz, w->rec, lane);
    uint32_t *out = a.scratch_idx + ev0;
    const uint32_t out_cap = ev1 - ev0;
    uint32_t nvis = 0;
    int qn = 0, head = 0;  // warp-uniform: number of staged survivors, ring position of the oldest

    auto resolve = [&](int count) {
      const bool have = lane < count;
      Ray ray;
      ray.ox = ox; ray.oy = oy; ray.oz = oz;
      ray.dx = ray.dy = ray.dz = 1.0f;
      ray.tfar = -1.0f;
      uint32_t pt = 0;
      V3 p{0.0, 0.0, 0.0};
      if (have) {
        const int e = (head + lane) & (FU_STAGE - 1);
        const uint32_t i = stage[e];
        pt = a.gidx[i];
        p = V3{a.gx[i], a.gy[i], a.gz[i]};
        if (OCC == FU_OCC_MESH) ray = make_ray(cen, p, a.endpoint_guard_rel != 0);
      }
      bool occ = false;
      if (OCC == FU_OCC_MESH) {
        if (WALK && n_list == TRILIST_OVERFLOW) {
          const int r = a.packet_bvh ? packet_bvh_hit<COUNT>(a, ray, have, ox, oy, oz, w->rec, lane, n_vis_nodes, n_tri) : 2;
          occ = r == 2 ? warp_any_hit<COUNT>(a.nodes, a.tris, a.n_nodes, ray, have, a.scene_absmax, a.counters)
                       : r == 1;
        } else
          occ = packet_any_hit<COUNT>(a, mylist, n_list, ray, have, ox, oy, oz, w->rec, hoisted, lane, n_vis_nodes, n_tri);
      } else if (OCC == FU_OCC_ANALYTIC) {
        occ = have && hits_building(cen, p, a.block_length, a.block_inset);
      }
      const bool vis = have && !occ;
      const unsigned m = __ballot_sync(0xffffffffu, vis);
      if (vis) {
        const uint32_t pos = nvis + __popc(m & ((1u << lane) - 1u));
        if (pos < out_cap)
          out[pos] = pt;
        else
          a.counters[5] = 1ull;  // cannot happen (visible <= planned row points); reported as an error
      }
      nvis += __popc(m);
    };

    // lane = row: the trimmed point ranges of up to 32 rows at a time (their cell_start loads in parallel),
    // then the warp scans the non-empty ones
    // this ticket's block of rows: ranges as the plan left them (one coalesced load), or — a camera with
    // more than FU_ROWS rows — recomputed with lane = row, 32 at a time
    int lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0}, ny = 1, nrows = (int)planned_rows;
    double cc[3] = {cen.x, cen.y, cen.z};
    if (planned_rows == FU_ROWS_MANY) {
      camera_cell_range(a.g, cc, a.max_dist, lo, hi);  // true: the plan got past it
      ny = hi[1] - lo[1] + 1;
      nrows = ny * (hi[2] - lo[2] + 1);
    }
    const int row0 = (nrows * part) >> a.parts_log2, row1 = (nrows * (part + 1)) >> a.parts_log2;
    for (int rb = planned_rows != FU_ROWS_MANY ? 0 : row0; rb < row1; rb += 32) {
      RowRange rr{0u, 0u};
      const int ri = rb + lane;
      if (ri >= row0 && ri < row1) {
        if (planned_rows != FU_ROWS_MANY) {  // at most FU_ROWS = 32 rows, one trip: lane = row index
          rr.start = myrow.x;
          rr.end = myrow.y;
        } else {
          rr = camera_row_call(a.g, a.cell_start, c, cc, a.max_dist, lo, hi, cell_h, lo[1] + ri % ny, lo[2] + ri / ny);
        }
      }
      unsigned live = __ballot_sync(0xffffffffu, rr.end > rr.start);
      if (live == 0u) continue;
      int j = __ffs(live) - 1;
      live &= live - 1;
      uint32_t base = __shfl_sync(0xffffffffu, rr.start, j), end = __shfl_sync(0xffffffffu, rr.end, j);
      // software pipeline over 32-point chunks, ACROSS rows: the next chunk (the next row's first one at a
      // row end) is in flight while the current one is evaluated
      V3 pn{0.0, 0.0, 0.0};
      if (base + lane < end) pn = V3{a.gx[base + lane], a.gy[base + lane], a.gz[base + lane]};
      for (;;) {
        uint32_t nbase = base + 32, nend = end;
        bool more = true;
        if (nbase >= end) {
          if (live) {
            j = __ffs(live) - 1;
            live &= live - 1;
            nbase = __shfl_sync(0xffffffffu, rr.start, j);
            nend = __shfl_sync(0xffffffffu, rr.end, j);
          } else {
            more = false;
          }
        }
        const uint32_t i = base + lane;
        const V3 pcur = pn;
        if (more && nbase + lane < nend) pn = V3{a.gx[nbase + lane], a.gy[nbase + lane], a.gz[nbase + lane]};
        bool pass = false;
        if (i < end) pass = cull_predicate(c, cen, pcur, a.t_star);
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (m != 0u) {
          if (pass) {
            const int e = (head + qn + __popc(m & ((1u << lane) - 1u))) & (FU_STAGE - 1);
            stage[e] = i;
          }
          qn += __popc(m);
          __syncwarp();
          if (qn >= 32) {
            resolve(32);
            __syncwarp();
            head = (head + 32) & (FU_STAGE - 1);
            qn -= 32;
            found_total += 32;
          }
        }
        if (!more) break;
        base = nbase;
        end = nend;
      }
    }
    if (qn > 0) {
      resolve(qn);
      found_total += qn;
    }
    nvis = nvis < out_cap ? nvis : out_cap;
    if (lane == 0) a.vis_count[slot] = nvis;
  }
  if (lane == 0) {
    if (found_total) atomicAdd(&a.counters[4], found_total);
    if (COUNT) {
      atomicAdd(&a.counters[2], (unsigned long long)n_vis_nodes);
      atomicAdd(&a.counters[3], (unsigned long long)n_tri);
    }
  }
}

// ---- per-camera sort + final write -------------------------------------------------------------------
template <int MIN_CTAS, bool MULTI>
__global__ void __launch_bounds__(SW_WARPS * 32, MIN_CTAS) k_sort_write(SortWriteArgs s) {
  __shared__ uint32_t s_sorted[SW_WARPS][SW_WARP_MAX + SW_WARP_MAX / 32];
  __shared__ uint32_t s_hist[SW_WARPS][SW_BINS];
  __shared__ double s_cam[SW_WARPS][16];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t cam = (uint64_t)blockIdx.x * SW_WARPS + warp;
  if (cam >= s.C) return;
  CamSlices cs = cam_slices<MULTI>(s, cam);
  // n is the same in every lane, but the compiler cannot know (it comes from memory through a per-thread
  // address); REDUX leaves it in a uniform register, so that the branches on it below are uniform branches
  // and the warp collectives inside them need no divergence scaffolding (BRA.DIV + WARPSYNC.COLLECTIVE
  // around every MATCH / SHFL were a fifth of this kernel's instructions, profiles/r01l)
  cs.n = __reduce_max_sync(0xffffffffu, cs.n);
  const uint32_t base = cs.base, n = cs.n;
  if (lane == 0) {
    s.out_offsets[cam] = base;
    if (cam == s.C - 1) s.out_offsets[s.C] = s.seg_off[s.C << s.parts_log2];
  }
  if (n == 0 || n > SW_WARP_MAX) return;
  if ((uint64_t)base + n > s.out_cap) {
    if (lane == 0) atomicOr(s.flags, (unsigned long long)FU_FLAG_OUT);
    return;
  }
  uint32_t *sorted = s_sorted[warp];
  if (n <= 128)
    sort_warp_to_smem<4, MULTI>(s, cs, lane, sorted, s_hist[warp]);
  else if (n <= 256)
    sort_warp_to_smem<8, MULTI>(s, cs, lane, sorted, s_hist[warp]);
  else if (n <= 512)
    sort_warp_to_smem<16, MULTI>(s, cs, lane, sorted, s_hist[warp]);
  else if (n <= 768)
    sort_warp_to_smem<24, MULTI>(s, cs, lane, sorted, s_hist[warp]);
  else
    sort_warp_to_smem<32, MULTI>(s, cs, lane, sorted, s_hist[warp]);
  __syncwarp();
  // Final write, two points ahead: the gathers of iterations i + 1 and i + 2 (24 B per lane from anywhere in the point array,
  // an L2 or HBM round trip) are in flight while iteration i is projected and stored.  The camera record waits in
  // shared memory (broadcast LDS.128) instead of 30 registers, which is what makes room for the extra points at
  // 64 registers; its address goes through an opaque register inside the loop, or the compiler hoists the
  // fifteen loads back into registers.  (r01: the same pipeline WITH the record in registers measured 0.85 ms
  // against 0.83 ms — it spilled.)
  double *crec = s_cam[warp];
  if (lane < 15) crec[lane] = __ldg(&s.cams[15 * cam + lane]);
  __syncwarp();
  uint32_t c_s = (uint32_t)__cvta_generic_to_shared(crec);
  // two gathers in flight per lane: (pt0, p0) is the point being written, (pt1, p1) the next one, and the loop
  // body starts the one after that
  struct Pt {
    uint32_t idx;
    double x, y, z;
  };
  auto gather = [&](uint32_t k) {
    Pt q{0u, 0.0, 0.0, 0.0};
    if (k < n) {
      q.idx = sorted[sw_pad(k)];
      const double *p = s.p_aos + 3 * (uint64_t)q.idx;
      q.x = __ldg(p);
      q.y = __ldg(p + 1);
      q.z = __ldg(p + 2);
    }
    return q;
  };
  uint32_t i = lane;
  Pt p0 = gather(i), p1 = gather(i + 32);
  while (i < n) {
    const Pt p2 = gather(i + 64);
    asm volatile("" : "+r"(c_s));
    const double *c = reinterpret_cast<const double *>(__cvta_shared_to_generic((size_t)c_s));
    s.out_idx[base + i] = p0.idx;
    s.out_uv[base + i] = observe(c, p0.x, p0.y, p0.z);
    i += 32;
    p0 = p1;
    p1 = p2;
  }
}

// cameras with SW_WARP_MAX < n <= SW_BLOCK_MAX: bitonic network in shared memory, one block each
__global__ void __launch_bounds__(256) k_sort_write_block(SortWriteArgs s) {
  __shared__ uint32_t s_sort[SW_BLOCK_MAX];
  const uint64_t cam = blockIdx.x;
  const CamSlices cs = cam_slices<true>(s, cam);
  const uint32_t base = cs.base, n = cs.n;
  if (n <= SW_WARP_MAX || n > SW_BLOCK_MAX) return;
  if ((uint64_t)base + n > s.out_cap) {
    if (threadIdx.x == 0) atomicOr(s.flags, (unsigned long long)FU_FLAG_OUT);
    return;
  }
  uint32_t n2 = 2;
  while (n2 < n) n2 <<= 1;
  for (uint32_t t = threadIdx.x; t < n2; t += blockDim.x) s_sort[t] = t < n ? cam_key<true>(s, cs, t) : 0xffffffffu;
  __syncthreads();
  for (uint32_t k = 2; k <= n2; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < n2; t += blockDim.x) {
        const uint32_t p = t ^ j;
        if (p > t) {
          const uint32_t x = s_sort[t], y = s_sort[p];
          const bool up = (t & k) == 0;
          if ((x > y) == up) {
            s_sort[t] = y;
            s_sort[p] = x;
          }
        }
      }
      __syncthreads();
    }
  }
  double c[15];
#pragma unroll
  for (int k = 0; k < 15; ++k) c[k] = __ldg(&s.cams[15 * cam + k]);
  for (uint32_t t = threadIdx.x; t < n; t += blockDim.x) {
    const uint32_t pt = s_sort[t];
    const double *p = s.p_aos + 3 * (uint64_t)pt;
    s.out_idx[base + t] = pt;
    s.out_uv[base + t] = observe(c, p[0], p[1], p[2]);
  }
}

// fallback for cameras that see more than SW_BLOCK_MAX points: 64-bit (camera, point) keys of ALL
// visible entries, radix-sorted globally, then k_write_sorted
__global__ void __launch_bounds__(256) k_expand_keys(SortWriteArgs s, int pbits, uint64_t *__restrict__ keys) {
  const int lane = threadIdx.x & 31;
  const uint64_t cam = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (cam >= s.C) return;
  const CamSlices cs = cam_slices<true>(s, cam);
  for (uint32_t t = lane; t < cs.n; t += 32) keys[cs.base + t] = (cam << pbits) | (uint64_t)cam_key<true>(s, cs, t);
}

// per-camera maximum of the visible counts (slots summed) and CSR offsets widened to u64
__global__ void k_max_cam(const uint32_t *__restrict__ seg_off, uint64_t C, int parts_log2, uint32_t *__restrict__ out) {
  uint32_t m = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < C; i += (uint64_t)gridDim.x * blockDim.x)
    m = max(m, seg_off[(i + 1) << parts_log2] - seg_off[i << parts_log2]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}
__global__ void k_widen_cam_offsets(const uint32_t *__restrict__ seg_off, uint64_t n, int parts_log2,
                                    uint64_t *__restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = seg_off[i << parts_log2];
}

}  // namespace c2b
