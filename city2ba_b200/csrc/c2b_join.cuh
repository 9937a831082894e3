// c2b_join.cuh — join_landmarks (src/noise.rs:323-378) on the device: n = floor(join_percent P) observations, drawn
// over all O observations, are re-pointed at one of the 10 nearest other landmarks of the landmark they see.  The
// neighbours are those of the original landmarks and the selections are distinct, so every selection is independent.
//
// The rule, restated by the test suite's checker (tests/join_ref.c) so that both agree bit for bit:
//   draws      one Philox4x32-10 block per observation o (global CSR index): key = seed, counter = (o lo, o hi,
//              ST_JOIN, 0); key_o = w0 | w1 << 32, r_o = w2 | w3 << 32.
//   selection  the min(n, O) smallest pairs (key_o, o), lexicographically: a uniform subset of exact size.
//   distance   d2(p, q) = (dx dx + dy dy) + dz dz, dx = p.x - q.x, ..., every operation rounded to nearest.
//   neighbours m = min(11, P); the list is the m smallest pairs (d2(p_q, p_k), k) over all points k (it holds q itself
//              and can hold several points at distance 0).  The pick is list[1 + mulhi64(r_o, m - 1)]: when a point of
//              lower index coincides with q, q itself can be picked (the host k-d tree's order).
//   errors     with at least one selection: P < 2 ("No neighbors?!"), or a point with a coordinate that is not finite
//              (the lowest one is named).  Nothing is changed then.
//
// Stages (ctx stream):
//   index      bounds of the f64 points and the lowest non-finite point in one pass -> 63-bit Morton codes over the
//              bounds (morton63) -> radix sort (c2b_sort.cuh) -> buckets of JN_BUCKET Morton-consecutive points as the
//              leaves of a Karras tree (k_bvh_karras), their f32 boxes rounded outward and the bottom-up refit
//              (k_bvh_refit with PointLeaf) -> the threaded pre-order layout of c2b_bvh.cuh (k_bvh_layout).  The
//              points are gathered in Morton order with their index, and each point's Morton position is kept.
//   selection  radix select of the (min(n, O))-th smallest 96-bit value (key_o << 32 | o): 12-bit digits, one
//              histogram pass over all O per digit (Philox recomputed), the host picks the digit, and stops as soon as
//              the rank falls on the whole of a digit's bucket.  Then one pass lists the selections, keyed by the
//              Morton position of the point they see, and a radix sort orders them by it.
//   queries    one thread per selection, neighbouring lanes near in space: nearest-child-first walk of the tree with a
//              per-thread stack; the m best (d2, index) pairs sorted in registers; the pick is written to idx[o] and
//              n_changed counted by warp ballot.
// Exactness of the pruning: a box's bound takes per axis the gap to the box with the same rounded subtraction, then
// the same rounded squares and sum order as d2.  Rounding is monotone, so the bound never exceeds the d2 of a point
// inside the box (the f32 box is rounded outward).  A subtree is skipped only when its bound exceeds the m-th d2
// strictly: a point at an equal distance and of lower index still enters the list.
#pragma once
#include "c2b_bvh.cuh"
#include "c2b_common.cuh"
#include "c2b_noise.cuh"
#include "c2b_sort.cuh"

namespace c2b {

constexpr int JN_THREADS = 256, JN_QUERY_THREADS = 128;
constexpr int JN_K = 11;        // the query point and its 10 neighbours (.skip(1).take(10))
constexpr int JN_BUCKET = 1;    // points per leaf (a sweep of 1, 2, 4, 8, 16 on the B200: profiles/r03f_bucket_sweep.json)
constexpr int JN_DIGIT = 12;    // bits per radix-select round (96-bit values: at most 8 rounds)
constexpr int JN_BINS = 1 << JN_DIGIT;
// A node's depth in the Karras tree is at most the number of distinct common-prefix lengths below it: 1..63 over the
// 63-bit keys and 96..127 over the leaf-index tie-break, 95 in all.  The stack holds at most one entry per level.
constexpr int JN_STACK = 96;
constexpr uint32_t JN_NO_POINT = 0xffffffffu;

inline unsigned jn_blocks(uint64_t threads, int per_block = JN_THREADS) {
  return (unsigned)((threads + per_block - 1) / per_block);
}

typedef unsigned __int128 u128;

// (key_o, r_o) of observation o
__device__ __forceinline__ void jn_draws(uint64_t seed, uint64_t o, uint64_t *key, uint64_t *r) {
  uint32_t w[4];
  noise_block(seed, ST_JOIN, o, 0, w);
  *key = (uint64_t)w[0] | (uint64_t)w[1] << 32;
  *r = (uint64_t)w[2] | (uint64_t)w[3] << 32;
}

__device__ __forceinline__ u128 jn_value(uint64_t seed, uint64_t o) {
  uint64_t key, r;
  jn_draws(seed, o, &key, &r);
  return (u128)key << 32 | (uint32_t)o;
}

__device__ __forceinline__ unsigned long long double_to_ordered(double d) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(d);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double ordered_to_double(unsigned long long u) {
  return __longlong_as_double((long long)((u >> 63) ? (u & 0x7fffffffffffffffull) : ~u));
}

__device__ __forceinline__ double jn_dist2(double3 p, double3 q) {
  const double dx = __dadd_rn(p.x, -q.x), dy = __dadd_rn(p.y, -q.y), dz = __dadd_rn(p.z, -q.z);
  return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// the lower bound of d2(q, p) over the points p of the f32 box [lo, hi]: per axis the rounded gap, 0 inside
__device__ __forceinline__ double jn_box_bound(float4 lo, float4 hi, double3 q) {
  const double gx = q.x < lo.x ? __dadd_rn((double)lo.x, -q.x) : q.x > hi.x ? __dadd_rn(q.x, -(double)hi.x) : 0.0;
  const double gy = q.y < lo.y ? __dadd_rn((double)lo.y, -q.y) : q.y > hi.y ? __dadd_rn(q.y, -(double)hi.y) : 0.0;
  const double gz = q.z < lo.z ? __dadd_rn((double)lo.z, -q.z) : q.z > hi.z ? __dadd_rn(q.z, -(double)hi.z) : 0.0;
  return __dadd_rn(__dadd_rn(__dmul_rn(gx, gx), __dmul_rn(gy, gy)), __dmul_rn(gz, gz));
}

// bounds[0..5] = ordered min xyz, max xyz over the points; *bad = the lowest point with a non-finite coordinate
__global__ void __launch_bounds__(JN_THREADS) k_jn_bounds(const double *__restrict__ pts, uint64_t P,
                                                          unsigned long long *__restrict__ bounds,
                                                          unsigned long long *__restrict__ bad) {
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  unsigned long long first_bad = ~0ull;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (uint64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double c = pts[3 * i + k];
      if (!(fabs(c) <= 1.7976931348623157e308)) first_bad = min(first_bad, (unsigned long long)i);
      lo[k] = fmin(lo[k], c);
      hi[k] = fmax(hi[k], c);
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
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) first_bad = min(first_bad, __shfl_xor_sync(0xffffffffu, first_bad, o));
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      atomicMin(&bounds[k], double_to_ordered(lo[k]));
      atomicMax(&bounds[3 + k], double_to_ordered(hi[k]));
    }
    if (first_bad != ~0ull) atomicMin(bad, first_bad);
  }
}

__global__ void __launch_bounds__(JN_THREADS) k_jn_morton(const double *__restrict__ pts, uint64_t P,
                                                          const unsigned long long *__restrict__ bounds,
                                                          uint64_t *__restrict__ keys, uint32_t *__restrict__ vals) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  float u[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const double lo = ordered_to_double(bounds[k]), ext = ordered_to_double(bounds[3 + k]) - lo;
    u[k] = ext > 0.0 ? (float)((pts[3 * i + k] - lo) / ext) : 0.0f;
  }
  keys[i] = morton63(u);
  vals[i] = (uint32_t)i;
}

// the Karras tree's leaf keys: the key of each bucket's first point
__global__ void __launch_bounds__(JN_THREADS) k_jn_leaf_keys(const uint64_t *__restrict__ keys, uint64_t n_leaves,
                                                             uint64_t *__restrict__ leaf_keys) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n_leaves) leaf_keys[s] = keys[s * JN_BUCKET];
}

// the leaf of the point tree: bucket s holds the Morton-ordered points [s B, min(s B + B, P)), gathered into spts as
// (x, y, z, index bits); pos[index] = the point's Morton position.  The f32 box is rounded outward.
struct PointLeaf {
  const double *pts;
  const uint32_t *sorted;
  uint64_t P;
  double4 *spts;
  uint32_t *pos;
  __device__ void operator()(int64_t s, float lo[3], float hi[3]) const {
    const uint64_t e = min((uint64_t)(s + 1) * JN_BUCKET, P);
    for (uint64_t j = (uint64_t)s * JN_BUCKET; j < e; ++j) {
      const uint32_t v = sorted[j];
      const double x = pts[3 * (uint64_t)v], y = pts[3 * (uint64_t)v + 1], z = pts[3 * (uint64_t)v + 2];
      spts[j] = make_double4(x, y, z, __longlong_as_double((long long)v));
      pos[v] = (uint32_t)j;
      lo[0] = fminf(lo[0], __double2float_rd(x));
      lo[1] = fminf(lo[1], __double2float_rd(y));
      lo[2] = fminf(lo[2], __double2float_rd(z));
      hi[0] = fmaxf(hi[0], __double2float_ru(x));
      hi[1] = fmaxf(hi[1], __double2float_ru(y));
      hi[2] = fmaxf(hi[2], __double2float_ru(z));
    }
  }
};

// one radix-select round: hist[d] += the values whose top `bits` bits equal pfx and whose next 12 bits are d
__global__ void __launch_bounds__(JN_THREADS) k_jn_hist(uint64_t O, uint64_t seed, int bits, u128 pfx,
                                                        uint32_t *__restrict__ hist) {
  __shared__ uint32_t h[JN_BINS];
  for (int i = threadIdx.x; i < JN_BINS; i += blockDim.x) h[i] = 0;
  __syncthreads();
  const int below = 96 - bits - JN_DIGIT;
  for (uint64_t o = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; o < O; o += (uint64_t)gridDim.x * blockDim.x) {
    const u128 v = jn_value(seed, o);
    if ((v >> (96 - bits)) == pfx) atomicAdd(&h[(uint32_t)(v >> below) & (JN_BINS - 1)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < JN_BINS; i += blockDim.x)
    if (h[i]) atomicAdd(&hist[i], h[i]);
}

// the selections (value's top `bits` bits <= pfx), in any order: key = the Morton position of the point they see,
// val = o
__global__ void __launch_bounds__(JN_THREADS) k_jn_list(uint64_t O, uint64_t seed, int bits, u128 pfx,
                                                        const uint32_t *__restrict__ idx,
                                                        const uint32_t *__restrict__ pos,
                                                        uint64_t *__restrict__ keys, uint32_t *__restrict__ vals,
                                                        unsigned long long *__restrict__ count) {
  const uint64_t o = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool s = o < O && (jn_value(seed, o) >> (96 - bits)) <= pfx;
  const unsigned m = __ballot_sync(0xffffffffu, s);
  if (!m) return;
  const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
  unsigned long long base = 0;
  if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  if (s) {
    const uint64_t at = base + __popc(m & ((1u << lane) - 1u));
    keys[at] = pos[idx[o]];
    vals[at] = (uint32_t)o;
  }
}

// (d, k) < (bd, bk) lexicographically
__device__ __forceinline__ bool jn_less(double d, uint32_t k, double bd, uint32_t bk) {
  return d < bd || (d == bd && k < bk);
}

// one thread per selection, in Morton order of the point it sees: the m nearest (d2, index) pairs, the pick into
// idx[o]; *n_changed += the selections whose pick is not the point they saw
__global__ void __launch_bounds__(JN_QUERY_THREADS)
    k_jn_query(const float4 *__restrict__ nodes, const double4 *__restrict__ spts, uint64_t P,
               const uint64_t *__restrict__ sel_pos, const uint32_t *__restrict__ sel_obs, uint64_t n_sel,
               uint64_t seed, uint32_t *__restrict__ idx, unsigned long long *__restrict__ n_changed) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool changed = false;
  if (s < n_sel) {
    const uint32_t o = sel_obs[s];
    const double4 qp = spts[sel_pos[s]];
    const double3 q = make_double3(qp.x, qp.y, qp.z);
    const uint32_t qi = (uint32_t)__double_as_longlong(qp.w);
    double bd[JN_K];
    uint32_t bk[JN_K];
#pragma unroll
    for (int j = 0; j < JN_K; ++j) {
      bd[j] = INFINITY;
      bk[j] = JN_NO_POINT;  // above every point index (P < 2^32 - 1): real pairs always enter before it
    }
    uint2 stack[JN_STACK];  // (node, f32 bound rounded down)
    int sp = 0;
    uint32_t node = 0;
    for (;;) {
      const float4 b = nodes[2 * node + 1];
      const int w = __float_as_int(b.w);
      if (w >= 0) {
        const uint64_t e = min((uint64_t)(w + 1) * JN_BUCKET, P);
        for (uint64_t j = (uint64_t)w * JN_BUCKET; j < e; ++j) {
          const double4 p = spts[j];
          const double d = jn_dist2(make_double3(p.x, p.y, p.z), q);
          const uint32_t k = (uint32_t)__double_as_longlong(p.w);
          if (jn_less(d, k, bd[JN_K - 1], bk[JN_K - 1])) {
            bool placed = false;
#pragma unroll
            for (int t = JN_K - 1; t >= 1; --t) {
              if (!placed && jn_less(d, k, bd[t - 1], bk[t - 1])) {
                bd[t] = bd[t - 1];
                bk[t] = bk[t - 1];
              } else if (!placed) {
                bd[t] = d;
                bk[t] = k;
                placed = true;
              }
            }
            if (!placed) {
              bd[0] = d;
              bk[0] = k;
            }
          }
        }
      } else {
        const uint32_t c0 = node + 1, c1 = (uint32_t)(-w - 1);
        const double b0 = jn_box_bound(nodes[2 * c0], nodes[2 * c0 + 1], q);
        const double b1 = jn_box_bound(nodes[2 * c1], nodes[2 * c1 + 1], q);
        const bool first0 = b0 <= b1;
        const uint32_t near = first0 ? c0 : c1, far = first0 ? c1 : c0;
        const double bn = first0 ? b0 : b1, bf = first0 ? b1 : b0;
        if (!(bn > bd[JN_K - 1])) {
          if (!(bf > bd[JN_K - 1])) stack[sp++] = make_uint2(far, __float_as_uint(__double2float_rd(bf)));
          node = near;
          continue;
        }
      }
      // the next stacked subtree whose bound does not exceed the m-th distance (a rounded-down bound above it
      // means the exact one is above it too)
      bool found = false;
      while (sp > 0) {
        const uint2 t = stack[--sp];
        if (!((double)__uint_as_float(t.y) > bd[JN_K - 1])) {
          node = t.x;
          found = true;
          break;
        }
      }
      if (!found) break;
    }
    uint64_t key, r;
    jn_draws(seed, o, &key, &r);
    const uint64_t m = P < JN_K ? P : JN_K;
    const uint64_t at = 1 + __umul64hi(r, m - 1);
    uint32_t pick = bk[1];
#pragma unroll
    for (int j = 2; j < JN_K; ++j)
      if (at == (uint64_t)j) pick = bk[j];
    idx[o] = pick;
    changed = pick != qi;
  }
  const unsigned m = __ballot_sync(0xffffffffu, changed);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(n_changed, (unsigned long long)__popc(m));
}

// scratch of the pass: sort keys / values (points, then selections), the tree and its boxes, the points in Morton
// order and their positions, the select histogram, flags and counters
struct JoinBufs {
  DevBuf keys[2], vals[2], hist, leaf_keys, left, right, first, last, par_i, par_l, visit, leaf_box, int_box, nodes,
      spts, pos, sel_hist, small;
  DevBuf scan_tmp[3];
};

// n = floor(join_percent P), 0 for a negative or NaN join_percent; then min(n, O)
inline uint64_t join_count(double join_percent, uint64_t P, uint64_t O) {
  const double nf = join_percent * (double)P;
  const uint64_t n = nf >= 18446744073709551616.0 ? ~0ull : nf >= 1.0 ? (uint64_t)nf : 0;
  return n < O ? n : O;
}

enum { JN_OK = 0, JN_NO_NEIGHBORS = 1, JN_NOT_FINITE = 2 };

// The pass over device points (pts: P AoS f64) and point indices (idx: O entries, all < P), enqueued on the ctx
// stream.  On return *err is JN_OK and idx holds the result, or *err names the input error (*bad_point: the lowest
// non-finite point) and idx is unchanged.
inline int join_pass(c2b_ctx *ctx, JoinBufs &b, const double *pts, uint64_t P, uint32_t *idx, uint64_t O,
                     double join_percent, uint64_t seed, uint64_t *n_selected, uint64_t *n_changed, int *err,
                     uint64_t *bad_point) {
  cudaStream_t st = ctx->stream;
  const uint64_t k = join_count(join_percent, P, O);
  *n_selected = *n_changed = 0;
  *err = JN_OK;
  if (k == 0) return C2B_OK;
  if (P < 2) {
    *err = JN_NO_NEIGHBORS;
    return C2B_OK;
  }
  C2B_TRY(ctx->h_small.ensure(256));
  C2B_TRY(b.small.ensure(128));
  // ordered bounds (min xyz, max xyz), the lowest non-finite point, selections listed, selections changed
  unsigned long long *bounds = b.small.as<unsigned long long>(), *bad = bounds + 6, *count = bounds + 7;
  const unsigned long long init[9] = {~0ull, ~0ull, ~0ull, 0ull, 0ull, 0ull, ~0ull, 0ull, 0ull};
  // ---- index
  C2B_CUDA(cudaMemcpyAsync(bounds, init, sizeof init, cudaMemcpyHostToDevice, st));
  k_jn_bounds<<<std::min<unsigned>(jn_blocks(P), 4u * ctx->sm_count), JN_THREADS, 0, st>>>(pts, P, bounds, bad);
  C2B_KERNEL_CHECK();
  // the pairs of the point sort, then of the selection sort: k = min(floor(join_percent P), O) exceeds P when
  // join_percent > 1 and O > P
  const uint64_t n_pairs = std::max(P, k);
  for (int i = 0; i < 2; ++i) {
    C2B_TRY(b.keys[i].ensure(n_pairs * 8));
    C2B_TRY(b.vals[i].ensure(n_pairs * 4));
  }
  uint64_t *keys[2] = {b.keys[0].as<uint64_t>(), b.keys[1].as<uint64_t>()};
  uint32_t *vals[2] = {b.vals[0].as<uint32_t>(), b.vals[1].as<uint32_t>()};
  k_jn_morton<<<jn_blocks(P), JN_THREADS, 0, st>>>(pts, P, bounds, keys[0], vals[0]);
  C2B_KERNEL_CHECK();
  int res = 0;
  C2B_TRY(radix_sort_pairs(st, keys, vals, P, 63, b.hist, b.scan_tmp, &res));
  const uint64_t nl = (P + JN_BUCKET - 1) / JN_BUCKET, ni = nl - 1;
  C2B_TRY(b.leaf_keys.ensure(nl * 8));
  C2B_TRY(b.leaf_box.ensure(nl * 24));
  C2B_TRY(b.par_l.ensure(nl * 4));
  C2B_TRY(b.nodes.ensure((2 * nl - 1) * 32));
  C2B_TRY(b.spts.ensure(P * 32));
  C2B_TRY(b.pos.ensure(P * 4));
  if (ni) {
    C2B_TRY(b.left.ensure(ni * 4));
    C2B_TRY(b.right.ensure(ni * 4));
    C2B_TRY(b.first.ensure(ni * 4));
    C2B_TRY(b.last.ensure(ni * 4));
    C2B_TRY(b.par_i.ensure(ni * 4));
    C2B_TRY(b.int_box.ensure(ni * 24));
    C2B_TRY(b.visit.ensure(ni * 4));
    C2B_CUDA(cudaMemsetAsync(b.visit.p, 0, ni * 4, st));
    k_jn_leaf_keys<<<jn_blocks(nl), JN_THREADS, 0, st>>>(keys[res], nl, b.leaf_keys.as<uint64_t>());
    C2B_KERNEL_CHECK();
    k_bvh_karras<<<jn_blocks(ni), JN_THREADS, 0, st>>>(b.leaf_keys.as<uint64_t>(), (int64_t)nl, b.left.as<uint32_t>(),
                                                       b.right.as<uint32_t>(), b.first.as<uint32_t>(),
                                                       b.last.as<uint32_t>(), b.par_i.as<uint32_t>(),
                                                       b.par_l.as<uint32_t>());
    C2B_KERNEL_CHECK();
  }
  k_bvh_refit<<<jn_blocks(nl), JN_THREADS, 0, st>>>(
      PointLeaf{pts, vals[res], P, b.spts.as<double4>(), b.pos.as<uint32_t>()}, (int64_t)nl, b.left.as<uint32_t>(),
      b.right.as<uint32_t>(), b.par_i.as<uint32_t>(), b.par_l.as<uint32_t>(), b.leaf_box.as<float>(),
      b.int_box.as<float>(), b.visit.as<uint32_t>());
  C2B_KERNEL_CHECK();
  k_bvh_layout<<<jn_blocks(2 * nl - 1), JN_THREADS, 0, st>>>(
      (int64_t)nl, b.left.as<uint32_t>(), b.right.as<uint32_t>(), b.first.as<uint32_t>(), b.last.as<uint32_t>(),
      b.par_i.as<uint32_t>(), b.par_l.as<uint32_t>(), b.leaf_box.as<float>(), b.int_box.as<float>(),
      b.nodes.as<float4>());
  C2B_KERNEL_CHECK();
  // ---- selection: the k-th smallest value, digit by digit (the first round's copy also brings the non-finite flag)
  int bits = 0;
  u128 pfx = 0;
  if (k < O) {
    C2B_TRY(b.sel_hist.ensure(JN_BINS * 4));
    uint32_t *hh = ctx->h_small.as<uint32_t>();
    std::vector<uint32_t> hist(JN_BINS);
    const unsigned nb = std::min<unsigned>(jn_blocks(O), 8u * ctx->sm_count);
    uint64_t need = k;
    while (bits < 96) {
      C2B_CUDA(cudaMemsetAsync(b.sel_hist.p, 0, JN_BINS * 4, st));
      k_jn_hist<<<nb, JN_THREADS, 0, st>>>(O, seed, bits, pfx, b.sel_hist.as<uint32_t>());
      C2B_KERNEL_CHECK();
      C2B_CUDA(cudaMemcpyAsync(hist.data(), b.sel_hist.p, JN_BINS * 4, cudaMemcpyDeviceToHost, st));
      if (bits == 0) C2B_CUDA(cudaMemcpyAsync(hh, bad, 8, cudaMemcpyDeviceToHost, st));
      C2B_CUDA(cudaStreamSynchronize(st));
      if (bits == 0 && *reinterpret_cast<unsigned long long *>(hh) != ~0ull) break;
      uint32_t d = 0;
      while (d < JN_BINS - 1 && need > hist[d]) need -= hist[d++];
      pfx = pfx << JN_DIGIT | d;
      bits += JN_DIGIT;
      if (need == hist[d]) break;  // the whole bucket is selected
    }
  }
  unsigned long long *h = ctx->h_small.as<unsigned long long>();
  if (k == O || bits == 0) {
    C2B_CUDA(cudaMemcpyAsync(h, bad, 8, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaStreamSynchronize(st));
  }
  if (h[0] != ~0ull) {
    *err = JN_NOT_FINITE;
    *bad_point = h[0];
    return C2B_OK;
  }
  // ---- selections, in Morton order of their point, and the queries
  k_jn_list<<<jn_blocks(O), JN_THREADS, 0, st>>>(O, seed, bits, pfx, idx, b.pos.as<uint32_t>(), keys[0], vals[0], count);
  C2B_KERNEL_CHECK();
  int pos_bits = 0;
  while (pos_bits < 32 && (P - 1) >> pos_bits) ++pos_bits;
  C2B_TRY(radix_sort_pairs(st, keys, vals, k, pos_bits, b.hist, b.scan_tmp, &res));
  k_jn_query<<<jn_blocks(k, JN_QUERY_THREADS), JN_QUERY_THREADS, 0, st>>>(
      b.nodes.as<float4>(), b.spts.as<double4>(), P, keys[res], vals[res], k, seed, idx, count + 1);
  C2B_KERNEL_CHECK();
  C2B_CUDA(cudaMemcpyAsync(h, count, 16, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  if (h[0] != k) return set_error(C2B_ERR_CUDA, "join_landmarks: %llu selections listed, %llu expected", h[0],
                                  (unsigned long long)k);
  *n_selected = k;
  *n_changed = h[1];
  return C2B_OK;
}

}  // namespace c2b
