// c2b_cull.cuh — kernel (1): camera x point distance / front / frustum culling with the f64
// SnavelyCamera projection (src/generate.rs:446-454, src/baproblem.rs:141-151).
//
// Two schedules produce the SAME candidate set (the exact f64 predicate always decides):
//   exhaustive : every pair, like the reference loop (this file).  Camera tile in shared memory,
//                4 points per thread in registers, a conservative 7-op FMA distance reject in the
//                hot loop; survivors are queued per warp and re-tested densely with the exact
//                predicate (so the rare expensive path does not diverge the hot loop).  Candidates
//                go to an unordered pool as (key = camera << pbits | point, u, v); the pool is then
//                radix-sorted by key, which yields camera-major, ascending-point order
//                (src/generate.rs:446).
//   grid       : points binned into a grid (cells max_dist/4 in y and z, a power-of-two fraction of that
//                in x, built here); one warp per camera scans the x-contiguous cell rows its max_dist
//                ball touches and resolves occlusion in the same pass (c2b_fused.cuh).
#pragma once
#include "c2b_common.cuh"
#include "c2b_math.cuh"

namespace c2b {

struct CullArgs {
  const double *cams;              // [15*C]
  const double *cen_x, *cen_y, *cen_z;  // [C]
  const double *px, *py, *pz;      // [P] (exhaustive) or grid-sorted copies (grid)
  uint64_t C, P;
  double t_star;   // m2 < t_star  <=>  sqrt_rn(m2) < max_dist   (exact)
  double t_cons;   // conservative bound for the FMA pre-test
  int pbits;
  uint64_t *pool_key;
  double2 *pool_uv;
  uint32_t *cam_count;
  unsigned long long *counters;  // [0] pool slots used, [1] pairs evaluated, [2] nodes, [3] tris,
                                 // [4] candidates (grid schedule: slots include chunk padding)
  uint64_t pool_capacity;
};

constexpr uint64_t POOL_SENTINEL = ~0ull;  // padding slot of a 32-aligned chunk

// SnavelyCamera::center once per camera (the reference recomputes it per pair: same value)
__global__ void k_cam_prep(const double *__restrict__ cams, uint64_t C, double *__restrict__ cx,
                           double *__restrict__ cy, double *__restrict__ cz) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C) return;
  double cam[15];
#pragma unroll
  for (int k = 0; k < 15; ++k) cam[k] = cams[15 * i + k];
  V3 c = camera_center(cam);
  cx[i] = c.x;
  cy[i] = c.y;
  cz[i] = c.z;
}

// AoS xyz -> SoA
__global__ void k_aos_to_soa3(const double *__restrict__ in, uint64_t n, double *__restrict__ x,
                              double *__restrict__ y, double *__restrict__ z) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  x[i] = in[3 * i];
  y[i] = in[3 * i + 1];
  z[i] = in[3 * i + 2];
}

// exact predicate with the sqrt folded into an exact threshold on the squared distance
__device__ __forceinline__ bool cull_project_thr(const double *cam, V3 center, V3 p, double t_star,
                                                 double &u, double &v) {
  V3 d{dsub(center.x, p.x), dsub(center.y, p.y), dsub(center.z, p.z)};
  double m2 = mag2(d);
  if (!(m2 < t_star)) return false;
  V3 pc = project_world(cam, p);
  if (!(pc.z <= 0.0)) return false;
  project(cam[12], cam[13], cam[14], pc, u, v);
  return u >= -1.0 && u <= 1.0 && v >= -1.0 && v <= 1.0;
}

// warp-converged emission of candidates into the pool (every lane of the warp must call)
__device__ __forceinline__ void emit_candidates(const CullArgs &a, bool pass, uint32_t cam,
                                                uint32_t pt, double u, double v) {
  const unsigned lane = threadIdx.x & 31u;
  unsigned m = __ballot_sync(0xffffffffu, pass);
  if (m == 0u) return;
  unsigned long long base = 0;
  if (lane == (unsigned)(__ffs(m) - 1)) base = atomicAdd(&a.counters[0], (unsigned long long)__popc(m));
  base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
  if (pass) {
    unsigned long long slot = base + __popc(m & ((1u << lane) - 1u));
    if (slot < a.pool_capacity) {
      a.pool_key[slot] = ((uint64_t)cam << a.pbits) | (uint64_t)pt;
      a.pool_uv[slot] = make_double2(u, v);
      atomicAdd(&a.cam_count[cam], 1u);
    }
  }
}

// ---- exhaustive schedule --------------------------------------------------------------------------
constexpr int CB_THREADS = 256;
constexpr int CB_PPT = 4;    // points per thread
constexpr int CB_TC = 64;    // cameras per tile
constexpr int CB_QCAP = 64;  // per-warp queue entries

__device__ __forceinline__ void brute_drain(const CullArgs &a, const uint2 *q, int first, int count) {
  const int lane = threadIdx.x & 31;
  bool have = lane < count;
  bool pass = false;
  uint32_t cam = 0, pt = 0;
  double u = 0, v = 0;
  if (have) {
    uint2 e = q[first + lane];
    cam = e.x;
    pt = e.y;
    double c[15];
#pragma unroll
    for (int k = 0; k < 15; ++k) c[k] = __ldg(&a.cams[15 * (uint64_t)cam + k]);
    V3 cen{a.cen_x[cam], a.cen_y[cam], a.cen_z[cam]};
    V3 p{a.px[pt], a.py[pt], a.pz[pt]};
    pass = cull_project_thr(c, cen, p, a.t_star, u, v);
  }
  emit_candidates(a, pass, cam, pt, u, v);
}

__global__ void __launch_bounds__(CB_THREADS) k_cull_exhaustive(CullArgs a) {
  __shared__ double s_cx[CB_TC], s_cy[CB_TC], s_cz[CB_TC];
  __shared__ uint2 s_q[CB_THREADS / 32][CB_QCAP];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t cam0 = (uint64_t)blockIdx.y * CB_TC;
  const int ncam = (int)((a.C - cam0) < (uint64_t)CB_TC ? (a.C - cam0) : (uint64_t)CB_TC);
  if (threadIdx.x < ncam) {
    s_cx[threadIdx.x] = a.cen_x[cam0 + threadIdx.x];
    s_cy[threadIdx.x] = a.cen_y[cam0 + threadIdx.x];
    s_cz[threadIdx.x] = a.cen_z[cam0 + threadIdx.x];
  }
  double px[CB_PPT], py[CB_PPT], pz[CB_PPT];
  uint64_t pi[CB_PPT];
#pragma unroll
  for (int k = 0; k < CB_PPT; ++k) {
    pi[k] = (uint64_t)blockIdx.x * (CB_THREADS * CB_PPT) + (uint64_t)k * CB_THREADS + threadIdx.x;
    bool ok = pi[k] < a.P;
    px[k] = ok ? a.px[pi[k]] : 1e300;  // (1e300)^2 = inf: never passes
    py[k] = ok ? a.py[pi[k]] : 1e300;
    pz[k] = ok ? a.pz[pi[k]] : 1e300;
  }
  __syncthreads();
  uint2 *q = s_q[warp];
  int qn = 0;  // warp-uniform
  const double tc = a.t_cons;
  for (int j = 0; j < ncam; ++j) {
    const double cx = s_cx[j], cy = s_cy[j], cz = s_cz[j];
    bool pass[CB_PPT];
    bool any = false;
#pragma unroll
    for (int k = 0; k < CB_PPT; ++k) {
      double dx = px[k] - cx, dy = py[k] - cy, dz = pz[k] - cz;
      double d2 = fma(dz, dz, fma(dy, dy, dx * dx));
      pass[k] = d2 < tc;
      any |= pass[k];
    }
    if (__any_sync(0xffffffffu, any)) {
#pragma unroll
      for (int k = 0; k < CB_PPT; ++k) {
        unsigned m = __ballot_sync(0xffffffffu, pass[k]);
        if (m) {
          if (pass[k]) q[qn + __popc(m & ((1u << lane) - 1u))] = make_uint2((uint32_t)(cam0 + j), (uint32_t)pi[k]);
          qn += __popc(m);
          __syncwarp();
          if (qn >= 32) {
            brute_drain(a, q, qn - 32, 32);
            qn -= 32;
            __syncwarp();
          }
        }
      }
    }
  }
  if (qn > 0) brute_drain(a, q, 0, qn);
}

// ---- grid schedule -----------------------------------------------------------------------------------
struct GridDesc {
  double lo[3];
  double inv_h;   // 1 / cell side in y and z
  double inv_hx;  // 1 / cell side in x: inv_h times the x split (a power of two), so rows hold finer cells
  double hx;      // 1 / inv_hx (the absolute slack of the x trims, c2b_fused.cuh)
  int n[3];
  int drop;         // 1: points outside [rlo, rhi] (the cameras' reach) are not in the grid at all
  double max_c[3];  // bounds of the points IN the grid (for the ball / grid early-out, rows of edge cells)
  double min_c[3];
  double rlo[3], rhi[3];
};

__device__ __forceinline__ int grid_coord(const GridDesc &g, int k, double x) {
  // explicit rounding: binning and range queries agree
  double t = floor(dmul(dsub(x, g.lo[k]), k == 0 ? g.inv_hx : g.inv_h));
  int c = t < 0.0 ? 0 : (t >= (double)g.n[k] ? g.n[k] - 1 : (int)t);  // NaN -> comparisons false
  if (!(t == t)) c = 0;
  return c;
}

// Both grid kernels aggregate their atomics per warp: neighbouring points of the input usually fall into the
// same cell (lattices, meshes sampled triangle by triangle), so __match_any_sync groups the lanes of a warp by
// cell and one lane per group issues a single atomic for the whole group.
__global__ void __launch_bounds__(256) k_grid_count(const double *__restrict__ px, const double *__restrict__ py,
                                                    const double *__restrict__ pz, uint64_t P, GridDesc g,
                                                    uint32_t *__restrict__ cell_of_pt, uint32_t *__restrict__ cell_count) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  uint32_t cell = 0xffffffffu;  // lanes past the end keep to themselves
  if (i < P) {
    const double x = px[i], y = py[i], z = pz[i];
    // outside the cameras' reach: farther than max_dist from every camera, never observed (NaN stays in)
    const bool out = g.drop && (x < g.rlo[0] || x > g.rhi[0] || y < g.rlo[1] || y > g.rhi[1] || z < g.rlo[2] || z > g.rhi[2]);
    if (!out) {
      int cx = grid_coord(g, 0, x), cy = grid_coord(g, 1, y), cz = grid_coord(g, 2, z);
      cell = ((uint32_t)cz * g.n[1] + cy) * g.n[0] + cx;
    }
    cell_of_pt[i] = cell;
  }
  const unsigned peers = __match_any_sync(0xffffffffu, cell);
  if (cell != 0xffffffffu && lane == __ffs(peers) - 1) atomicAdd(&cell_count[cell], (uint32_t)__popc(peers));
}

// cursor[] starts as a copy of cell_start[], so the atomic returns the absolute position
__global__ void __launch_bounds__(256) k_grid_fill(const double *__restrict__ px, const double *__restrict__ py,
                                                   const double *__restrict__ pz, uint64_t P,
                                                   const uint32_t *__restrict__ cell_of_pt, uint32_t *__restrict__ cursor,
                                                   double *__restrict__ gx, double *__restrict__ gy,
                                                   double *__restrict__ gz, uint32_t *__restrict__ gidx) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const uint32_t cell = i < P ? cell_of_pt[i] : 0xffffffffu;
  const bool valid = cell != 0xffffffffu;  // past the end, or outside the cameras' reach
  double x = 0.0, y = 0.0, z = 0.0;
  if (valid) {
    x = px[i];
    y = py[i];
    z = pz[i];
  }
  const unsigned peers = __match_any_sync(0xffffffffu, cell);
  const int leader = __ffs(peers) - 1;
  uint32_t first = 0;
  if (valid && lane == leader) first = atomicAdd(&cursor[cell], (uint32_t)__popc(peers));
  const uint32_t pos = __shfl_sync(0xffffffffu, first, leader) + __popc(peers & ((1u << lane) - 1u));
  if (valid) {
    gx[pos] = x;
    gy[pos] = y;
    gz[pos] = z;
    gidx[pos] = (uint32_t)i;
  }
}

// min / max of point coordinates (two-stage, deterministic): out[0..2] = min, out[3..5] = max
__global__ void k_pts_bounds_partial(const double *__restrict__ px, const double *__restrict__ py,
                                     const double *__restrict__ pz, uint64_t P,
                                     double *__restrict__ partial /* 6*gridDim.x */) {
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P;
       i += (uint64_t)gridDim.x * blockDim.x) {
    double v[3] = {px[i], py[i], pz[i]};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      lo[k] = fmin(lo[k], v[k]);
      hi[k] = fmax(hi[k], v[k]);
    }
  }
  __shared__ double s[6][8];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[k] = fmin(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
      hi[k] = fmax(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
    }
    if ((threadIdx.x & 31) == 0) {
      s[k][threadIdx.x >> 5] = lo[k];
      s[3 + k][threadIdx.x >> 5] = hi[k];
    }
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double r = s[threadIdx.x][0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
      r = threadIdx.x < 3 ? fmin(r, s[threadIdx.x][w]) : fmax(r, s[threadIdx.x][w]);
    partial[6 * (uint64_t)blockIdx.x + threadIdx.x] = r;
  }
}
// one warp: lane = block partial (strided), then a shuffle tree (min and max are order-independent: the same
// result as a serial fold, 40 us sooner — this runs inside every pass of a camera shard, camera_bbox)
__global__ void k_pts_bounds_final(const double *__restrict__ partial, int nb, double *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int b = lane; b < nb; b += 32) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      lo[k] = fmin(lo[k], partial[6 * b + k]);
      hi[k] = fmax(hi[k], partial[6 * b + 3 + k]);
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[k] = fmin(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
      hi[k] = fmax(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      out[k] = lo[k];
      out[3 + k] = hi[k];
    }
  }
}

}  // namespace c2b
