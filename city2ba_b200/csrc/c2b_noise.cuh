// c2b_noise.cuh — kernel family (4): the `noise` pass (src/noise.rs:35-177) as Philox-keyed
// elementwise kernels, plus the two global statistics it needs (BAProblem::mean/std,
// src/baproblem.rs:282-304, and the element nearest the world origin, src/noise.rs:75-87) as
// deterministic two-stage tree reductions.
//
// Random stream: Philox4x32-10, key = seed, counter = (index lo, index hi, stream, slot); ONE block per
// point / observation (two per camera).  The reference draws a direction as a normalised Gaussian pair or
// triple (unit_random, src/noise.rs:35-43; (nx, ny) / |(nx, ny)|, :159-163) and a magnitude as Normal(m, s)
// from the unseedable thread_rng(): only distributions can be matched, and a normalised Gaussian pair IS a
// uniform direction on the circle, a triple a uniform point on the sphere.  So a block supplies
//     circle  (cos, sin)(2 pi w / 2^32)                                one 32-bit word
//     sphere  z = 1 - 2 (b + 1/2) / 2^32, azimuth from a               two words
//     N(0,1)  Box-Muller, u1 = (n40 + 1) 2^-40, angle from 24 bits     two words
// evaluated by table + short polynomial (cos / sin of k 2 pi / 256 with a Taylor remainder, ln by 128
// mantissa intervals and a degree-6 series): ~55 FP64 instructions per observation where two Box-Muller
// pairs through libm's log / sincos took ~160 (profiles/r01m_ncu_r01m_noise_obs.txt: FP64 pipe 47 %, 0.26 of
// the HBM peak).  Every operation is an explicit fma / mul / add in a fixed order, so a CPU restatement
// that performs the same ones on the same tables (filled on the host by c2b_init with libm) reproduces points
// and observations bit for bit (the test suite's checker does); cameras (sin / cos / pow of libm inside) to a few ulp.
#pragma once
#include "c2b_common.cuh"
#include "c2b_math.cuh"

namespace c2b {

// ST_MISMATCH: add_incorrect_correspondences (c2b_mismatch.cuh), ST_JOIN: join_landmarks (c2b_join.cuh); one block
// per observation
enum { ST_DRIFT_CAM = 1, ST_DRIFT_PT = 2, ST_NOISE_CAM = 3, ST_NOISE_PT = 4, ST_NOISE_OBS = 5, ST_MISMATCH = 6,
       ST_JOIN = 7 };

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t *out) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0;
    c1 = lo1;
    c2 = n2;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0;
  out[1] = c1;
  out[2] = c2;
  out[3] = c3;
}

__device__ double2 g_sc_tab[256];  // (cos, sin)(k 2 pi / 256)
__device__ double2 g_ln_tab[128];  // (1 / c_j, ln c_j), c_j = 1 + (2 j + 1) / 256

// the host's copy of the tables (libm), uploaded to every device by c2b_init
inline void noise_tables_host(double2 *sc, double2 *ln) {
  for (int k = 0; k < 256; ++k) {
    const double a = (double)k * (6.283185307179586 / 256.0);
    sc[k] = make_double2(cos(a), sin(a));
  }
  for (int j = 0; j < 128; ++j) {
    const double c = 1.0 + (double)(2 * j + 1) / 256.0;
    ln[j] = make_double2(1.0 / c, log(c));
  }
}

struct NoiseTabs {
  double2 sc[256];
  double2 ln[128];
};

// block-wide: the tables into shared memory (random indices: a table in constant memory would serialise)
__device__ __forceinline__ void load_noise_tabs(NoiseTabs &t) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) t.sc[i] = g_sc_tab[i];
  for (int i = threadIdx.x; i < 128; i += blockDim.x) t.ln[i] = g_ln_tab[i];
  __syncthreads();
}

__device__ __forceinline__ void noise_block(uint64_t seed, uint32_t stream, uint64_t index, uint32_t slot, uint32_t *o) {
  philox4x32_10((uint32_t)index, (uint32_t)(index >> 32), stream, slot, (uint32_t)seed, (uint32_t)(seed >> 32), o);
}

// (cos, sin) of 2 pi w / 2^32
__device__ __forceinline__ void unit2(const NoiseTabs &t, uint32_t w, double &c, double &s) {
  const uint32_t k = (w + 0x800000u) >> 24;  // nearest table angle; wraps to 0 at the top
  const double d = __dmul_rn((double)(int32_t)(w - (k << 24)), 1.4629180792671596e-09);  // 2 pi / 2^32; |d| <= pi / 256
  const double d2 = __dmul_rn(d, d);
  double ps = __fma_rn(d2, 1.0 / 120.0, -1.0 / 6.0);
  ps = __fma_rn(d2, ps, 1.0);
  const double sd = __dmul_rn(d, ps);
  double pc = __fma_rn(d2, -1.0 / 720.0, 1.0 / 24.0);
  pc = __fma_rn(d2, pc, -0.5);
  const double cd = __fma_rn(d2, pc, 1.0);
  const double2 a = t.sc[k & 255u];
  c = __fma_rn(a.x, cd, -__dmul_rn(a.y, sd));
  s = __fma_rn(a.y, cd, __dmul_rn(a.x, sd));
}

// -2 ln u, u = (n40 + 1) 2^-40 in (0, 1]; never negative
__device__ __forceinline__ double neg2ln40(const NoiseTabs &t, uint64_t n40) {
  const double u = __dmul_rn(__ull2double_rn(n40 + 1ull), 9.094947017729282e-13);  // 2^-40, exact
  const long long bits = __double_as_longlong(u);
  const int e = (int)((bits >> 52) & 0x7ff) - 1023;
  const double2 tj = t.ln[(int)((bits >> 45) & 127)];
  const double m = __longlong_as_double((bits & 0x000fffffffffffffll) | 0x3ff0000000000000ll);
  const double r = __fma_rn(m, tj.x, -1.0);
  double p = __fma_rn(r, -1.0 / 6.0, 0.2);
  p = __fma_rn(r, p, -0.25);
  p = __fma_rn(r, p, 1.0 / 3.0);
  p = __fma_rn(r, p, -0.5);
  p = __fma_rn(r, p, 1.0);
  p = __dmul_rn(r, p);
  const double ln = __dadd_rn(__fma_rn((double)e, 0.6931471805599453, tj.y), p);
  return fmax(__dmul_rn(-2.0, ln), 0.0);
}

// N(0,1) from two words: u1 from a and the top byte of b (40 bits), the angle from b's other 24 bits
__device__ __forceinline__ double normal40(const NoiseTabs &t, uint32_t a, uint32_t b) {
  const uint64_t n40 = (uint64_t)a | ((uint64_t)(b >> 24) << 32);
  double c, s;
  unit2(t, b << 8, c, s);
  return __dmul_rn(__dsqrt_rn(neg2ln40(t, n40)), c);
}

// uniform point on the unit sphere from two words
__device__ __forceinline__ V3 sphere(const NoiseTabs &t, uint32_t a, uint32_t b) {
  double c, s;
  unit2(t, a, c, s);
  const double z = __dsub_rn(1.0, __dmul_rn(__dadd_rn((double)b, 0.5), 4.656612873077393e-10));  // 2^-31
  const double q = __dsqrt_rn(fmax(__fma_rn(-z, z, 1.0), 0.0));
  return V3{__dmul_rn(q, c), __dmul_rn(q, s), z};
}

// element i of the chained sequence "camera centres, then points" (src/baproblem.rs:284-287)
__device__ __forceinline__ V3 chain_element(const double *cx, const double *cy, const double *cz,
                                            uint64_t C, const double *pts, uint64_t i) {
  if (i < C) return V3{cx[i], cy[i], cz[i]};
  const double *p = pts + 3 * (i - C);
  return V3{p[0], p[1], p[2]};
}

constexpr int ST_BLOCKS = 592;  // 4 x 148 SMs
constexpr int ST_THREADS = 256;

// MODE 0: sum of e/num ; MODE 1: sum of (e-mean)^2 ; partial[3*block + k]
template <int MODE>
__global__ void __launch_bounds__(ST_THREADS)
    k_stats_partial(const double *__restrict__ cx, const double *__restrict__ cy,
                    const double *__restrict__ cz, uint64_t C, const double *__restrict__ pts,
                    uint64_t P, double num, const double *__restrict__ mean_dev, double *__restrict__ partial) {
  // MODE 1 reads the mean the MODE 0 pass left on the device: no host round trip between the two
  const V3 mean = MODE == 1 ? V3{mean_dev[0], mean_dev[1], mean_dev[2]} : V3{0.0, 0.0, 0.0};
  double s[3] = {0, 0, 0};
  uint64_t n = C + P;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (uint64_t)gridDim.x * blockDim.x) {
    V3 e = chain_element(cx, cy, cz, C, pts, i);
    if (MODE == 0) {
      s[0] += e.x / num;
      s[1] += e.y / num;
      s[2] += e.z / num;
    } else {
      double a = e.x - mean.x, b = e.y - mean.y, c = e.z - mean.z;
      s[0] += a * a;
      s[1] += b * b;
      s[2] += c * c;
    }
  }
  __shared__ double sh[3][ST_THREADS / 32];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
    if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = s[k];
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double r = 0;
    for (int w = 0; w < ST_THREADS / 32; ++w) r += sh[threadIdx.x][w];
    partial[3 * (uint64_t)blockIdx.x + threadIdx.x] = r;
  }
}

// one warp: lane = block partial (strided, ascending), then a shuffle tree — a fixed order, so the sums are
// reproducible run to run (a single thread folding 592 partials took ~50 us of dependent loads: three such
// folds were a third of the drift pass)
__global__ void k_stats_final(const double *__restrict__ partial, int nb, double *__restrict__ out3) {
  const int lane = threadIdx.x & 31;
  double r[3] = {0.0, 0.0, 0.0};
  for (int b = lane; b < nb; b += 32) {
#pragma unroll
    for (int k = 0; k < 3; ++k) r[k] += partial[3 * b + k];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r[k] += __shfl_xor_sync(0xffffffffu, r[k], o);
  }
  if (lane < 3) out3[lane] = lane == 0 ? r[0] : (lane == 1 ? r[1] : r[2]);
}

// s[3..5] = sum of squared deviations, num = element count  ->  s[9] = |std()| (BAProblem::std, src/baproblem.rs:292-304,
// then its magnitude, src/noise.rs:127): the scale of add_noise's camera translations, left on the device
__global__ void k_bal_std(double *__restrict__ s, double num) {
  if (threadIdx.x == 0) {
    const double a = dsqrt(ddiv(s[3], num)), b = dsqrt(ddiv(s[4], num)), c = dsqrt(ddiv(s[5], num));
    s[9] = dsqrt(dadd(dadd(dmul(a, a), dmul(b, b)), dmul(c, c)));
  }
}

// nearest-to-origin element; the reference's fold keeps the LATER element on ties
// (src/noise.rs:80-86), so the reduction orders by (distance asc, index desc).
__device__ __forceinline__ bool nearer(double da, uint64_t ia, double db, uint64_t ib) {
  return da < db || (da == db && ia > ib);
}
__global__ void __launch_bounds__(ST_THREADS)
    k_nearest_partial(const double *__restrict__ cx, const double *__restrict__ cy,
                      const double *__restrict__ cz, uint64_t C, const double *__restrict__ pts,
                      uint64_t P, double *__restrict__ pd, unsigned long long *__restrict__ pi) {
  double bd = INFINITY;
  uint64_t bi = 0;
  bool have = false;
  uint64_t n = C + P;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (uint64_t)gridDim.x * blockDim.x) {
    double d = mag(chain_element(cx, cy, cz, C, pts, i));
    if (!have || nearer(d, i, bd, bi) || !(bd == bd)) {
      bd = d;
      bi = i;
      have = true;
    }
  }
  if (!have) {
    bd = INFINITY;
    bi = 0;
  }
  __shared__ double sd[ST_THREADS];
  __shared__ unsigned long long si[ST_THREADS];
  __shared__ int sv[ST_THREADS];
  sd[threadIdx.x] = bd;
  si[threadIdx.x] = bi;
  sv[threadIdx.x] = have ? 1 : 0;
  __syncthreads();
  for (int o = ST_THREADS / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      int a = threadIdx.x, b = threadIdx.x + o;
      if (sv[b] && (!sv[a] || nearer(sd[b], si[b], sd[a], si[a]))) {
        sd[a] = sd[b];
        si[a] = si[b];
        sv[a] = 1;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    pd[blockIdx.x] = sv[0] ? sd[0] : INFINITY;
    pi[blockIdx.x] = sv[0] ? si[0] : ~0ull;
  }
}
__global__ void k_nearest_final(const double *__restrict__ pd, const unsigned long long *__restrict__ pi,
                                int nb, const double *__restrict__ cx, const double *__restrict__ cy,
                                const double *__restrict__ cz, uint64_t C,
                                const double *__restrict__ pts, double *__restrict__ origin3) {
  // one warp: lane = block partial (strided), then a shuffle tree; the order (distance asc, index desc) is total,
  // so the result does not depend on how the partials are combined
  const int lane = threadIdx.x & 31;
  double bd = INFINITY;
  unsigned long long bi = ~0ull;
  for (int b = lane; b < nb; b += 32) {
    if (pi[b] == ~0ull) continue;
    if (bi == ~0ull || nearer(pd[b], pi[b], bd, bi)) {
      bd = pd[b];
      bi = pi[b];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, bd, o);
    const unsigned long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (oi != ~0ull && (bi == ~0ull || nearer(od, oi, bd, bi))) {
      bd = od;
      bi = oi;
    }
  }
  if (lane == 0) {
    V3 e = bi == ~0ull ? V3{0, 0, 0} : chain_element(cx, cy, cz, C, pts, bi);
    origin3[0] = e.x;
    origin3[1] = e.y;
    origin3[2] = e.z;
  }
}

// ---- add_drift, src/noise.rs:68-116 ------------------------------------------------------------------
constexpr int NZ_THREADS = 256;

__global__ void __launch_bounds__(NZ_THREADS)
    k_drift_cams(double *__restrict__ cams, uint64_t C, const double *__restrict__ origin, V3 dir, double strength,
                 double angle_strength, double std, uint64_t seed) {
  __shared__ NoiseTabs tabs;
  load_noise_tabs(tabs);
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C) return;
  double cam[15];
#pragma unroll
  for (int k = 0; k < 15; ++k) cam[k] = cams[15 * i + k];
  V3 c = camera_center(cam);
  V3 d{dsub(c.x, origin[0]), dsub(c.y, origin[1]), dsub(c.z, origin[2])};
  double distance = mag(d);
  double z0 = 0.0, z1 = 0.0;
  if (std != 0.0) {  // Normal(1, 0) is 1 whatever the draw
    uint32_t o[4];
    noise_block(seed, ST_DRIFT_CAM, i, 0, o);
    z0 = normal40(tabs, o[0], o[1]);  // the angle's draw first (src/noise.rs:104-107)
    z1 = normal40(tabs, o[2], o[3]);
  }
  double v1 = dadd(1.0, dmul(std, z0)), v2 = dadd(1.0, dmul(std, z1));
  double angle = dmul(dmul(angle_strength, v1), pow(distance, 1.2));
  V3 dl{dmul(dmul(dmul(dmul(dir.x, strength), v2), distance), distance),
        dmul(dmul(dmul(dmul(dir.y, strength), v2), distance), distance),
        dmul(dmul(dmul(dmul(dir.z, strength), v2), distance), distance)};
  double R[9], out[15];
  from_angle_x(angle, R);
  camera_transform(cam, R, dl, out);
#pragma unroll
  for (int k = 0; k < 15; ++k) cams[15 * i + k] = out[k];
}

__global__ void __launch_bounds__(NZ_THREADS)
    k_drift_pts(double *__restrict__ pts, uint64_t P, const double *__restrict__ origin, V3 dir, double strength,
                double std, uint64_t seed) {
  __shared__ NoiseTabs tabs;
  if (std != 0.0) load_noise_tabs(tabs);
  const double ox = origin[0], oy = origin[1], oz = origin[2];
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (uint64_t)gridDim.x * blockDim.x) {
    V3 p{pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    V3 d{dsub(p.x, ox), dsub(p.y, oy), dsub(p.z, oz)};
    double distance = mag(d);
    double z0 = 0.0;
    if (std != 0.0) {
      uint32_t o[4];
      noise_block(seed, ST_DRIFT_PT, i, 0, o);
      z0 = normal40(tabs, o[0], o[1]);
    }
    double v = dadd(1.0, dmul(std, z0));
    pts[3 * i] = dadd(p.x, dmul(dmul(dmul(dmul(dir.x, strength), v), distance), distance));
    pts[3 * i + 1] = dadd(p.y, dmul(dmul(dmul(dmul(dir.y, strength), v), distance), distance));
    pts[3 * i + 2] = dadd(p.z, dmul(dmul(dmul(dmul(dir.z, strength), v), distance), distance));
  }
}

// ---- add_noise, src/noise.rs:119-177 --------------------------------------------------------------------
// per camera: axis, angle, translation direction, magnitude (:140-141) = block 0 {sphere, N}, block 1 {sphere, N}
__global__ void __launch_bounds__(NZ_THREADS)
    k_noise_cams(double *__restrict__ cams, uint64_t C, const double *__restrict__ bal_std_dev, double translation_std,
                 double rotation_std, uint64_t seed) {
  __shared__ NoiseTabs tabs;
  load_noise_tabs(tabs);
  const double bal_std = *bal_std_dev;
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C) return;
  double cam[15];
#pragma unroll
  for (int k = 0; k < 15; ++k) cam[k] = cams[15 * i + k];
  uint32_t o0[4], o1[4];
  noise_block(seed, ST_NOISE_CAM, i, 0, o0);
  noise_block(seed, ST_NOISE_CAM, i, 1, o1);
  const V3 ax = sphere(tabs, o0[0], o0[1]);
  const double angle = dadd(0.0, dmul(rotation_std, normal40(tabs, o0[2], o0[3])));
  const V3 tr = sphere(tabs, o1[0], o1[1]);
  const double m = dadd(0.0, dmul(translation_std, normal40(tabs, o1[2], o1[3])));
  double R[9], out[15];
  from_axis_angle(ax, angle, R);
  V3 dl{dmul(dmul(tr.x, bal_std), m), dmul(dmul(tr.y, bal_std), m), dmul(dmul(tr.z, bal_std), m)};
  camera_transform(cam, R, dl, out);
#pragma unroll
  for (int k = 0; k < 15; ++k) cams[15 * i + k] = out[k];
}

// per point: direction, magnitude (:149) = one block {sphere, N}
__global__ void __launch_bounds__(NZ_THREADS)
    k_noise_pts(double *__restrict__ pts, uint64_t P, double point_std, uint64_t seed) {
  __shared__ NoiseTabs tabs;
  load_noise_tabs(tabs);
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t o[4];
    noise_block(seed, ST_NOISE_PT, i, 0, o);
    const V3 ax = sphere(tabs, o[0], o[1]);
    const double m = dadd(0.0, dmul(point_std, normal40(tabs, o[2], o[3])));
    pts[3 * i] = dadd(pts[3 * i], dmul(ax.x, m));
    pts[3 * i + 1] = dadd(pts[3 * i + 1], dmul(ax.y, m));
    pts[3 * i + 2] = dadd(pts[3 * i + 2], dmul(ax.z, m));
  }
}

// per observation: direction (nx, ny) / |(nx, ny)|, r (:159-163) = one block {circle, -, N}.  `first` = global
// index of uv[0] (the host entry streams the array through the GPU in chunks).
__global__ void __launch_bounds__(NZ_THREADS)
    k_noise_obs(double2 *__restrict__ uv, uint64_t O, uint64_t first, double observations_std, uint64_t seed) {
  __shared__ NoiseTabs tabs;
  load_noise_tabs(tabs);
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < O; i += (uint64_t)gridDim.x * blockDim.x) {
    double2 q = uv[i];
    uint32_t o[4];
    noise_block(seed, ST_NOISE_OBS, first + i, 0, o);
    double nx, ny;
    unit2(tabs, o[0], nx, ny);
    const double r = dadd(0.0, dmul(observations_std, normal40(tabs, o[2], o[3])));
    q.x = dadd(q.x, dmul(nx, r));
    q.y = dadd(q.y, dmul(ny, r));
    uv[i] = q;
  }
}

// ---- add_sin_noise, src/noise.rs:388-416 --------------------------------------------------------------
// extent of the chained sequence (BAProblem::extent, src/baproblem.rs:307-330): partial[6*block + k]
__global__ void __launch_bounds__(ST_THREADS)
    k_extent_partial(const double *__restrict__ cx, const double *__restrict__ cy,
                     const double *__restrict__ cz, uint64_t C, const double *__restrict__ pts,
                     uint64_t P, double *__restrict__ partial) {
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  uint64_t n = C + P;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (uint64_t)gridDim.x * blockDim.x) {
    V3 e = chain_element(cx, cy, cz, C, pts, i);
    // f64::min / f64::max semantics (a NaN operand is ignored), like fmin / fmax
    lo[0] = fmin(lo[0], e.x); lo[1] = fmin(lo[1], e.y); lo[2] = fmin(lo[2], e.z);
    hi[0] = fmax(hi[0], e.x); hi[1] = fmax(hi[1], e.y); hi[2] = fmax(hi[2], e.z);
  }
  __shared__ double sh[6][ST_THREADS / 32];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[k] = fmin(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
      hi[k] = fmax(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
    }
    if ((threadIdx.x & 31) == 0) {
      sh[k][threadIdx.x >> 5] = lo[k];
      sh[3 + k][threadIdx.x >> 5] = hi[k];
    }
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double r = sh[threadIdx.x][0];
    for (int w = 1; w < ST_THREADS / 32; ++w)
      r = threadIdx.x < 3 ? fmin(r, sh[threadIdx.x][w]) : fmax(r, sh[threadIdx.x][w]);
    partial[6 * (uint64_t)blockIdx.x + threadIdx.x] = r;
  }
}
// out6 = min xyz, max xyz
__global__ void k_extent_final(const double *__restrict__ partial, int nb, double *__restrict__ out6) {
  const int lane = threadIdx.x & 31;  // one warp: lane = block partial (strided), then a shuffle tree
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
      out6[k] = lo[k];
      out6[3 + k] = hi[k];
    }
  }
}

// noise(x) = sin(dot(x / dimension, dir) * frequency * pi) * strength * normalize(noise_dir)
__device__ __forceinline__ V3 sin_noise(V3 x, V3 dim, V3 dir, V3 nd, double strength, double frequency) {
  const V3 q{ddiv(x.x, dim.x), ddiv(x.y, dim.y), ddiv(x.z, dim.z)};
  const double dot = dadd(dadd(dmul(q.x, dir.x), dmul(q.y, dir.y)), dmul(q.z, dir.z));
  const double amp = dmul(sin(dmul(dmul(dot, frequency), 3.14159265358979323846)), strength);
  return V3{dmul(nd.x, amp), dmul(nd.y, amp), dmul(nd.z, amp)};
}

__global__ void k_sin_cams(double *__restrict__ cams, uint64_t C, V3 dim, V3 dir, V3 nd, double strength,
                           double frequency) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C) return;
  double cam[15], out[15];
#pragma unroll
  for (int k = 0; k < 15; ++k) cam[k] = cams[15 * i + k];
  const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};  // Basis3::one()
  camera_transform(cam, I, sin_noise(camera_center(cam), dim, dir, nd, strength, frequency), out);
#pragma unroll
  for (int k = 0; k < 15; ++k) cams[15 * i + k] = out[k];
}

__global__ void k_sin_pts(double *__restrict__ pts, uint64_t P, V3 dim, V3 dir, V3 nd, double strength,
                          double frequency) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  const V3 p{pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
  const V3 d = sin_noise(p, dim, dir, nd, strength, frequency);
  pts[3 * i] = dadd(p.x, d.x);
  pts[3 * i + 1] = dadd(p.y, d.y);
  pts[3 * i + 2] = dadd(p.z, d.z);
}

// ---- total_reprojection_error, src/baproblem.rs:265-279 (one thread per observation, two-stage sum)
__global__ void __launch_bounds__(ST_THREADS)
    k_reproj_partial(const double *__restrict__ cams, const double *__restrict__ px,
                     const double *__restrict__ py, const double *__restrict__ pz,
                     const uint64_t *__restrict__ offsets, uint64_t C,
                     const uint32_t *__restrict__ idx, const double2 *__restrict__ uv, uint64_t O,
                     double norm, double *__restrict__ partial) {
  double s = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < O;
       i += (uint64_t)gridDim.x * blockDim.x) {
    // camera of observation i: largest c with offsets[c] <= i
    uint64_t lo = 0, hi = C;
    while (hi - lo > 1) {
      uint64_t mid = (lo + hi) >> 1;
      if (offsets[mid] <= i) lo = mid; else hi = mid;
    }
    double cam[15];
#pragma unroll
    for (int k = 0; k < 15; ++k) cam[k] = __ldg(&cams[15 * lo + k]);
    uint64_t pt = idx[i];
    V3 pc = project_world(cam, V3{px[pt], py[pt], pz[pt]});
    double u, v;
    project(cam[12], cam[13], cam[14], pc, u, v);
    double du = fabs(u - uv[i].x), dv = fabs(v - uv[i].y);
    if (norm == 1.0) s += du + dv;
    else if (norm == 2.0) s += du * du + dv * dv;
    else s += pow(du, norm) + pow(dv, norm);
  }
  __shared__ double sh[ST_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double r = 0;
    for (int w = 0; w < ST_THREADS / 32; ++w) r += sh[w];
    partial[blockIdx.x] = r;
  }
}

}  // namespace c2b
