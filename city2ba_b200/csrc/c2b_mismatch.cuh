// c2b_mismatch.cuh — add_incorrect_correspondences (src/noise.rs:180-226) on the device: within every camera of more
// than one observation, each observation i is selected with probability mismatch_chance and trades its point index
// with a partner j of the same camera drawn with weight w_j = maxd - |uv_i - uv_j| (maxd = the largest of those
// distances; w_i = maxd, as the reference is written).  (u, v) never move, so every (i, j) depends on (u, v) and the
// draws only; the transpositions are then applied per camera in ascending i.
//
// The rule, restated by the test suite's checker so that both agree bit for bit:
//   draws     one Philox4x32-10 block per observation: key = seed, counter = (o lo, o hi, ST_MISMATCH, 0), o the
//             global CSR index.  u = ((w0 | w1 << 32) >> 11) 2^-53; selected iff u <= mismatch_chance (NaN: never).
//             r = w2 | w3 << 32.
//   distance  d_j = sqrt(dx dx + dy dy), dx = u_i - u_j, dy = v_i - v_j, every operation rounded to nearest, no
//             contraction.  maxd = sqrt(max_j dx dx + dy dy) (sqrt is monotone, so this is max_j d_j).
//   errors    any distance not finite: NegativeWeight; otherwise maxd == 0: AllWeightsZero (Rng::weighted's order).
//   weights   q_j = floor((maxd - d_j) / maxd * 2^32) in u64 (q_i = 2^32), T = sum q_j (exact: O < 2^32).
//   pick      t = mulhi64(r, T) in [0, T); j = the smallest index whose inclusive prefix sum of q exceeds t.
// Integer sums are associative, so any evaluation order gives the same j.
//
// Passes (ctx stream): count selections per camera (one warp per camera) -> exclusive scan -> list the selected
// observations with their camera, in CSR order -> one thread per selection computes its j (a warp holds 32
// consecutive selections: lanes of one camera read the same (u, v) in step, a long camera spreads over many warps)
// -> one thread per camera applies its transpositions in ascending i, unless an error was flagged.  The error flag
// is atomicMin over (o << 1 | kind), so the reported observation is the lowest offending one, the one the sequential
// host forms stop at.
#pragma once
#include "c2b_common.cuh"
#include "c2b_noise.cuh"
#include "c2b_sort.cuh"

namespace c2b {

constexpr int MM_THREADS = 256;
enum { MM_ALL_WEIGHTS_ZERO = 0, MM_NEGATIVE_WEIGHT = 1 };
constexpr unsigned long long MM_NO_ERROR = ~0ull;

inline unsigned mm_blocks(uint64_t threads) { return (unsigned)((threads + MM_THREADS - 1) / MM_THREADS); }

// whether observation o is selected (words 0-1 of its block; words 2-3 are the pick's, k_mm_pick)
__device__ __forceinline__ bool mm_selected(uint64_t seed, uint64_t o, double chance) {
  uint32_t w[4];
  noise_block(seed, ST_MISMATCH, o, 0, w);
  const double u = __dmul_rn((double)((((uint64_t)w[1] << 32) | w[0]) >> 11), 0x1p-53);
  return u <= chance;
}

__device__ __forceinline__ double mm_dist2(double2 p, double2 q) {
  const double dx = __dadd_rn(p.x, -q.x), dy = __dadd_rn(p.y, -q.y);
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
}

// q = floor((maxd - d) / maxd * 2^32), in [0, 2^32]
__device__ __forceinline__ uint64_t mm_weight(double2 p, double2 q, double maxd) {
  const double d = __dsqrt_rn(mm_dist2(p, q));
  return __double2ull_rz(__dmul_rn(__ddiv_rn(__dadd_rn(maxd, -d), maxd), 4294967296.0));
}

// one warp per camera: cnt[c] = selected observations of camera c (0 when it has at most one)
__global__ void __launch_bounds__(MM_THREADS) k_mm_count(const uint64_t *__restrict__ off, uint64_t C, double chance,
                                                         uint64_t seed, uint32_t *__restrict__ cnt) {
  const uint64_t c = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C) return;
  const uint64_t b = off[c], e = off[c + 1];
  uint32_t n = 0;
  if (e - b > 1)
    for (uint64_t o = b + lane; o < e; o += 32) n += mm_selected(seed, o, chance);
  n = __reduce_add_sync(0xffffffffu, n);
  if (lane == 0) cnt[c] = n;
}

// one warp per camera: the selected observations (o, c) from sel[base[c]] on, in CSR order
__global__ void __launch_bounds__(MM_THREADS) k_mm_list(const uint64_t *__restrict__ off, uint64_t C, double chance,
                                                        uint64_t seed, const uint32_t *__restrict__ base,
                                                        uint2 *__restrict__ sel) {
  const uint64_t c = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C) return;
  const uint64_t b = off[c], e = off[c + 1];
  if (e - b <= 1) return;
  uint32_t pos = base[c];
  for (uint64_t o0 = b; o0 < e; o0 += 32) {
    const uint64_t o = o0 + lane;
    const bool s = o < e && mm_selected(seed, o, chance);
    const unsigned m = __ballot_sync(0xffffffffu, s);
    if (s) sel[pos + __popc(m & ((1u << lane) - 1u))] = make_uint2((uint32_t)o, (uint32_t)c);
    pos += __popc(m);
  }
}

// one thread per selection: its partner j (global CSR index) into pick[s], or the lowest error into *err
__global__ void __launch_bounds__(MM_THREADS)
    k_mm_pick(const uint64_t *__restrict__ off, const double2 *__restrict__ uv, const uint2 *__restrict__ sel,
              uint64_t n_sel, uint64_t seed, uint32_t *__restrict__ pick, unsigned long long *__restrict__ err,
              unsigned long long *__restrict__ n_swapped) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool swapped = false;
  if (s < n_sel) {
    const uint2 e = sel[s];
    const uint64_t a = off[e.y];
    const uint32_t n = (uint32_t)(off[e.y + 1] - a), i = (uint32_t)(e.x - a);  // camera slice, i within it
    const double2 *cu = uv + a;
    const double2 p = cu[i];
    double m2 = 0.0;
    bool finite = true;
    for (uint32_t k = 0; k < n; ++k) {
      const double s2 = mm_dist2(p, cu[k]);
      finite &= s2 <= 1.7976931348623157e308;  // false for NaN and inf
      m2 = fmax(m2, s2);
    }
    if (!finite) {
      atomicMin(err, (unsigned long long)e.x << 1 | MM_NEGATIVE_WEIGHT);
    } else if (m2 == 0.0) {
      atomicMin(err, (unsigned long long)e.x << 1 | MM_ALL_WEIGHTS_ZERO);
    } else {
      const double maxd = __dsqrt_rn(m2);
      uint32_t w[4];
      noise_block(seed, ST_MISMATCH, e.x, 0, w);
      // walk 0 sums T (no limit); walk 1 stops at the first prefix above t = mulhi64(r, T).  Q_{n-1} = T > t, so
      // when no earlier prefix exceeds t, j is the last observation.  (One loop walked twice: a single call site of
      // the square root's slow path.)
      uint64_t t = ~0ull;
      uint32_t j = 0;
      for (int walk = 0; walk < 2; ++walk) {
        uint64_t acc = 0;
        for (j = 0; j < n; ++j) {
          acc += mm_weight(p, cu[j], maxd);
          if (acc > t) break;
        }
        t = __umul64hi((uint64_t)w[2] | (uint64_t)w[3] << 32, acc);
      }
      pick[s] = (uint32_t)a + j;
      swapped = j != i;
    }
  }
  const unsigned m = __ballot_sync(0xffffffffu, swapped);
  if ((threadIdx.x & 31) == 0 && m) atomicAdd(n_swapped, (unsigned long long)__popc(m));
}

// one thread per camera: its transpositions in ascending i, only when no selection failed
__global__ void __launch_bounds__(MM_THREADS)
    k_mm_apply(const uint32_t *__restrict__ cnt, const uint32_t *__restrict__ base, uint64_t C,
               const uint2 *__restrict__ sel, const uint32_t *__restrict__ pick,
               const unsigned long long *__restrict__ err, uint32_t *__restrict__ idx) {
  const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C || *err != MM_NO_ERROR) return;
  const uint32_t k0 = base[c], k1 = k0 + cnt[c];
  for (uint32_t k = k0; k < k1; ++k) {
    const uint32_t i = sel[k].x, j = pick[k];
    const uint32_t t = idx[i];
    idx[i] = idx[j];
    idx[j] = t;
  }
}

// scratch of the pass: per-camera counts and bases, the selection list and picks, the flag and counters
struct MismatchBufs {
  DevBuf *cnt, *sel, *small;
};

// The pass over the device CSR (off: C + 1 offsets, validated; idx / uv: offsets[C] entries), enqueued on the ctx
// stream with two host synchronisations.  On return *err is MM_NO_ERROR and idx holds the result, or *err is the
// lowest failing (o << 1 | kind) and idx is unchanged.
inline int mismatch_pass(c2b_ctx *ctx, const MismatchBufs &bufs, const uint64_t *off, uint64_t C, uint32_t *idx,
                         const double2 *uv, double chance, uint64_t seed, uint64_t *n_selected, uint64_t *n_swapped,
                         unsigned long long *err) {
  cudaStream_t st = ctx->stream;
  C2B_TRY(bufs.cnt->ensure((2 * C + 1) * 4));
  C2B_TRY(bufs.small->ensure(32));
  C2B_TRY(ctx->h_small.ensure(256));
  uint32_t *cnt = bufs.cnt->as<uint32_t>(), *base = cnt + C;
  unsigned long long *d_err = bufs.small->as<unsigned long long>(), *d_swapped = d_err + 1;
  uint32_t *d_nsel = reinterpret_cast<uint32_t *>(d_err + 2);
  unsigned long long *h = ctx->h_small.as<unsigned long long>();
  C2B_CUDA(cudaMemsetAsync(d_err, 0xff, 8, st));
  C2B_CUDA(cudaMemsetAsync(d_swapped, 0, 16, st));
  if (C) {
    k_mm_count<<<mm_blocks(C * 32), MM_THREADS, 0, st>>>(off, C, chance, seed, cnt);
    C2B_KERNEL_CHECK();
    C2B_TRY(exclusive_scan_u32(st, cnt, base, C, d_nsel, ctx->scan_tmp));
  }
  C2B_CUDA(cudaMemcpyAsync(h, d_nsel, 4, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  const uint64_t ns = *reinterpret_cast<uint32_t *>(h);
  if (ns) {
    C2B_TRY(bufs.sel->ensure(ns * 12));
    uint2 *sel = bufs.sel->as<uint2>();
    uint32_t *pick = reinterpret_cast<uint32_t *>(sel + ns);
    k_mm_list<<<mm_blocks(C * 32), MM_THREADS, 0, st>>>(off, C, chance, seed, base, sel);
    C2B_KERNEL_CHECK();
    k_mm_pick<<<mm_blocks(ns), MM_THREADS, 0, st>>>(off, uv, sel, ns, seed, pick, d_err, d_swapped);
    C2B_KERNEL_CHECK();
    k_mm_apply<<<mm_blocks(C), MM_THREADS, 0, st>>>(cnt, base, C, sel, pick, d_err, idx);
    C2B_KERNEL_CHECK();
  }
  C2B_CUDA(cudaMemcpyAsync(h, d_err, 16, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  *err = h[0];
  *n_selected = ns;
  *n_swapped = h[1];
  return C2B_OK;
}

}  // namespace c2b
