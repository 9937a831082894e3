// c2b_graph_cull.cuh — BAProblem::cull (src/baproblem.rs:538-549) on the device: largest_connected_component
// (:456-534, with its observation filter at :523 as written) followed by remove_singletons (:426-453), applied
// until the camera and point counts stop changing.  Not to be confused with the camera x point visibility test
// of c2b_cull.cuh: the kernels here are k_lcc_* (components) and k_prune_* (flags, compaction).
//
// One application on (C cameras, P points, camera-major CSR of O observations):
//   1. components of the bipartite graph over entities 0..C-1 (cameras) and C..C+P-1 (points): lock-free
//      union-find, one warp per camera over its CSR slice, min-hooking by atomicCAS on the larger root and path
//      halving in find (ECL-CC style).  Roots are only ever hooked under smaller roots, so after one compression
//      pass every entity holds the smallest entity of its component: the host mirrors' label.
//   2. component sizes (warp-aggregated histogram) and L = the largest component, lowest label on a tie
//      (one u64 atomicMax over (size << 32) | ~label).
//   3. per camera c in L: the observations (c, p) with label[p] == L — the reference's sets[x.0] at :523, the point
//      index used as an entity index without the camera offset — count for the camera and, by atomics, for the
//      point.  A camera survives with > 3 such observations, a point with > 1.  An observation survives if its
//      camera, its own flag and its point do.
//   4. one ballot word per 32 observations / cameras / points, k_word_popc + exclusive_scan_u32 (the visibility
//      pass's compaction scheme, c2b_compact.cuh / c2b_sort.cuh), position = word prefix + popc(lower bits):
//      stable compaction of camera records, points, remapped point indices, (u, v) and the new CSR offsets.
// One host synchronisation per application reads (C', P', O') and decides whether the loop stops.
// Bounds: C + P < 2^32 (u32 entity ids and labels), O < 2^32 (u32 word prefixes).
#pragma once
#include "c2b_common.cuh"
#include "c2b_compact.cuh"
#include "c2b_sort.cuh"

namespace c2b {

constexpr int PR_THREADS = 256;
constexpr int PR_WARPS = PR_THREADS / 32;

// ---- components -------------------------------------------------------------------------------------------
// parent[x] <= x always holds (hooks go from the larger root to the smaller), so the walk ends at a root.
// Path halving (hooking phase only): every visited entity is pointed at its grandparent.  Such a store can only set a
// non-root's parent to another ancestor on the same upward chain, and roots are changed by atomicCAS only, so no hook
// is lost.  The stored value need not be final there: the label pass resolves every entity to its root.
__device__ __forceinline__ uint32_t lcc_find(volatile uint32_t *parent, uint32_t x) {
  while (true) {
    const uint32_t p = parent[x];
    if (p == x) return x;
    const uint32_t g = parent[p];
    if (g == p) return p;
    parent[x] = g;
    x = g;
  }
}

// hook the components of roots (possibly stale) u and v: the larger root goes under the smaller one
__device__ __forceinline__ void lcc_unite(uint32_t *parent, uint32_t u, uint32_t v) {
  while (u != v) {
    if (u > v) {
      const uint32_t t = u;
      u = v;
      v = t;
    }
    const uint32_t old = atomicCAS(parent + v, v, u);
    if (old == v) return;
    v = lcc_find(parent, old);  // v had been hooked meanwhile: continue from its new root
    u = lcc_find(parent, u);
  }
}

__global__ void k_lcc_init(uint32_t *__restrict__ parent, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) parent[i] = (uint32_t)i;
}

// one warp per camera: unite camera c with entity C + p of each of its observations
__global__ void __launch_bounds__(PR_THREADS) k_lcc_hook(const uint64_t *__restrict__ off, const uint32_t *__restrict__ idx,
                                                         uint64_t C, uint32_t *parent) {
  const uint64_t c = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C) return;
  const uint64_t b = off[c], e = off[c + 1];
  uint32_t cr = lcc_find(parent, (uint32_t)c);
  for (uint64_t j = b + lane; j < e; j += 32) {
    const uint32_t v = lcc_find(parent, (uint32_t)(C + idx[j]));
    cr = lcc_find(parent, cr);
    lcc_unite(parent, cr, v);
  }
}

// the root of x without writing anything (no hooks happen any more when it is used)
__device__ __forceinline__ uint32_t lcc_root(const volatile uint32_t *parent, uint32_t x) {
  uint32_t r = parent[x];
  while (true) {
    const uint32_t p = parent[r];
    if (p == r) return r;
    r = p;
  }
}

// compression (parent[i] = root = smallest entity of i's component) and the component sizes, one atomic per
// group of lanes of a warp that share a root.  The walk is read-only, so the one store to parent[i] is thread i's
// own root: a halving store by another thread could otherwise land after it and leave parent[i] at a non-root
// ancestor.  Other threads' stores meanwhile only put roots into the chain, so every walk still ends at the root.
__global__ void __launch_bounds__(PR_THREADS) k_lcc_label(uint32_t *parent, uint64_t n, uint32_t *__restrict__ size) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((i & ~31ull) >= n) return;
  uint32_t r = 0xffffffffu;
  if (i < n) {
    r = lcc_root(parent, (uint32_t)i);
    parent[i] = r;
  }
  const unsigned peers = __match_any_sync(0xffffffffu, r);
  if (i < n && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(size + r, (uint32_t)__popc(peers));
}

// *best = max over roots of (size << 32) | (0xffffffff - label): the largest component, the lowest label on a tie
__global__ void __launch_bounds__(PR_THREADS) k_lcc_pick(const uint32_t *__restrict__ size, uint64_t n,
                                                         unsigned long long *__restrict__ best) {
  unsigned long long m = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t s = size[i];
    if (s) m = max(m, ((unsigned long long)s << 32) | (unsigned long long)(0xffffffffu - (uint32_t)i));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(best, m);
}

__device__ __forceinline__ uint32_t lcc_label_of(const unsigned long long *best) {
  return 0xffffffffu - (uint32_t)(*best & 0xffffffffull);
}

// ---- flags -------------------------------------------------------------------------------------------------
// one warp per camera: the observations that survive the component filter (camera in L, label[p] == L), counted
// per camera (cam_cnt) and per point (pt_cnt, atomics)
__global__ void __launch_bounds__(PR_THREADS)
    k_prune_count(const uint64_t *__restrict__ off, const uint32_t *__restrict__ idx, uint64_t C,
                  const uint32_t *__restrict__ label, const unsigned long long *__restrict__ best,
                  uint32_t *__restrict__ cam_cnt, uint32_t *__restrict__ pt_cnt) {
  const uint64_t c = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C) return;
  const uint32_t L = lcc_label_of(best);
  uint32_t n = 0;
  if (label[c] == L) {
    const uint64_t b = off[c], e = off[c + 1];
    for (uint64_t j = b + lane; j < e; j += 32) {
      const uint32_t p = idx[j];
      if (label[p] == L) {  // src/baproblem.rs:523: sets[point index], no camera offset
        atomicAdd(pt_cnt + p, 1u);
        ++n;
      }
    }
  }
  n = __reduce_add_sync(0xffffffffu, n);
  if (lane == 0) cam_cnt[c] = n;
}

// one warp per surviving camera, over the 32-aligned words its CSR slice touches: bit j of the observation words
// = observation j survives.  Words shared with a neighbouring camera are merged by atomicOr (zeroed before).
__global__ void __launch_bounds__(PR_THREADS)
    k_prune_obs_words(const uint64_t *__restrict__ off, const uint32_t *__restrict__ idx, uint64_t C,
                      const uint32_t *__restrict__ label, const unsigned long long *__restrict__ best,
                      const uint32_t *__restrict__ cam_cnt, const uint32_t *__restrict__ pt_cnt,
                      uint32_t *__restrict__ words) {
  const uint64_t c = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= C || cam_cnt[c] <= 3) return;
  const uint32_t L = lcc_label_of(best);
  const uint64_t b = off[c], e = off[c + 1];
  for (uint64_t base = b & ~31ull; base < e; base += 32) {
    const uint64_t j = base + lane;
    bool keep = false;
    if (j >= b && j < e) {
      const uint32_t p = idx[j];
      keep = label[p] == L && pt_cnt[p] > 1;
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (lane == 0 && m) atomicOr(words + (base >> 5), m);
  }
}

// bit i of words = cnt[i] > threshold (cameras: > 3 observations, points: > 1)
__global__ void __launch_bounds__(PR_THREADS) k_prune_flag_words(const uint32_t *__restrict__ cnt, uint64_t n,
                                                                 uint32_t threshold, uint32_t *__restrict__ words) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if ((i & ~31ull) >= n) return;
  const unsigned m = __ballot_sync(0xffffffffu, i < n && cnt[i] > threshold);
  if ((threadIdx.x & 31) == 0) words[i >> 5] = m;
}

// ---- compaction --------------------------------------------------------------------------------------------
__device__ __forceinline__ bool prune_bit(const uint32_t *words, uint64_t i) { return (words[i >> 5] >> (i & 31)) & 1u; }
// new index of item i = surviving items before it
__device__ __forceinline__ uint32_t prune_rank(const uint32_t *words, const uint32_t *prefix, uint64_t i) {
  return prefix[i >> 5] + __popc(words[i >> 5] & ((1u << (i & 31)) - 1u));
}

__global__ void __launch_bounds__(PR_THREADS)
    k_prune_write_obs(const uint32_t *__restrict__ idx, const double2 *__restrict__ uv, uint64_t O,
                      const uint32_t *__restrict__ obs_words, const uint32_t *__restrict__ obs_prefix,
                      const uint32_t *__restrict__ pt_words, const uint32_t *__restrict__ pt_prefix,
                      uint32_t *__restrict__ out_idx, double2 *__restrict__ out_uv) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= O || !prune_bit(obs_words, i)) return;
  const uint32_t pos = prune_rank(obs_words, obs_prefix, i);
  out_idx[pos] = prune_rank(pt_words, pt_prefix, idx[i]);
  out_uv[pos] = uv[i];
}

// one thread per double of the camera records; the thread of a surviving camera's first double also writes its
// CSR offset (surviving observations of the cameras before it), thread 0 the closing offset
__global__ void __launch_bounds__(PR_THREADS)
    k_prune_write_cams(const double *__restrict__ cams, const uint64_t *__restrict__ off, uint64_t C,
                       const uint32_t *__restrict__ cam_words, const uint32_t *__restrict__ cam_prefix,
                       const uint32_t *__restrict__ obs_words, const uint32_t *__restrict__ obs_prefix,
                       const uint32_t *__restrict__ totals, double *__restrict__ out_cams,
                       uint64_t *__restrict__ out_off) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e == 0) out_off[totals[0]] = totals[2];
  if (e >= 15 * C) return;
  const uint64_t c = e / 15, k = e - 15 * c;
  if (!prune_bit(cam_words, c)) return;
  const uint64_t pos = prune_rank(cam_words, cam_prefix, c);
  out_cams[15 * pos + k] = cams[e];
  if (k == 0) out_off[pos] = prune_rank(obs_words, obs_prefix, off[c]);
}

__global__ void __launch_bounds__(PR_THREADS)
    k_prune_write_pts(const double *__restrict__ pts, uint64_t P, const uint32_t *__restrict__ pt_words,
                      const uint32_t *__restrict__ pt_prefix, double *__restrict__ out_pts) {
  const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= 3 * P) return;
  const uint64_t p = e / 3, k = e - 3 * p;
  if (!prune_bit(pt_words, p)) return;
  out_pts[3 * (uint64_t)prune_rank(pt_words, pt_prefix, p) + k] = pts[e];
}

// input check of c2b_cull_problem: bit 0 = offsets[0] != 0 or a decreasing offset, bit 1 = point index >= P
__global__ void __launch_bounds__(PR_THREADS) k_prune_validate(const uint64_t *__restrict__ off, uint64_t C,
                                                               const uint32_t *__restrict__ idx, uint64_t O, uint64_t P,
                                                               uint32_t *__restrict__ flag) {
  uint32_t f = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < C || i < O; i += (uint64_t)gridDim.x * blockDim.x) {
    if (i < C && off[i + 1] < off[i]) f |= 1u;
    if (i < O && idx[i] >= P) f |= 2u;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && off[0] != 0) f |= 1u;
  f = __reduce_or_sync(0xffffffffu, f);
  if ((threadIdx.x & 31) == 0 && f) atomicOr(flag, f);
}

// ---- driver ------------------------------------------------------------------------------------------------
// the arrays of one problem on the device: camera records (15 f64), points (3 f64), CSR offsets (u64), point
// indices (u32), (u, v)
struct PruneSet {
  DevBuf *cams, *pts, *off, *idx, *uv;
};

inline unsigned prune_blocks(uint64_t n) { return (unsigned)((n + PR_THREADS - 1) / PR_THREADS); }

// One application of LCC + remove_singletons from set `in` to set `out` (C > 0; out's buffers hold the input's
// sizes).  Leaves (C', P', O') in totals[0..2] on the device.
inline int prune_apply(c2b_ctx *ctx, const PruneSet &in, const PruneSet &out, uint64_t C, uint64_t P, uint64_t O,
                       uint32_t *totals) {
  cudaStream_t st = ctx->stream;
  const uint64_t n = C + P;
  const uint64_t wo = (O + 31) / 32, wc = (C + 31) / 32, wp = (P + 31) / 32;
  C2B_TRY(ctx->pr_parent.ensure(n * 4));
  C2B_TRY(ctx->pr_size.ensure(n * 4));
  C2B_TRY(ctx->pr_cam_cnt.ensure(C * 4));
  C2B_TRY(ctx->pr_pt_cnt.ensure(std::max<uint64_t>(P, 1) * 4));
  C2B_TRY(ctx->pr_words.ensure((wo + wc + wp + 1) * 4));
  C2B_TRY(ctx->pr_prefix.ensure((wo + wc + wp + 1) * 4));
  uint32_t *parent = ctx->pr_parent.as<uint32_t>(), *size = ctx->pr_size.as<uint32_t>();
  uint32_t *cam_cnt = ctx->pr_cam_cnt.as<uint32_t>(), *pt_cnt = ctx->pr_pt_cnt.as<uint32_t>();
  uint32_t *w_obs = ctx->pr_words.as<uint32_t>(), *w_cam = w_obs + wo, *w_pt = w_cam + wc;
  uint32_t *x_obs = ctx->pr_prefix.as<uint32_t>(), *x_cam = x_obs + wo, *x_pt = x_cam + wc;
  unsigned long long *best = ctx->pr_small.as<unsigned long long>();
  const uint64_t *off = in.off->as<uint64_t>();
  const uint32_t *idx = in.idx->as<uint32_t>();

  C2B_CUDA(cudaMemsetAsync(best, 0, 8, st));
  C2B_CUDA(cudaMemsetAsync(size, 0, n * 4, st));
  if (P) C2B_CUDA(cudaMemsetAsync(pt_cnt, 0, P * 4, st));
  if (wo) C2B_CUDA(cudaMemsetAsync(w_obs, 0, wo * 4, st));
  // components, sizes, L
  k_lcc_init<<<prune_blocks(n), PR_THREADS, 0, st>>>(parent, n);
  C2B_KERNEL_CHECK();
  if (O) {
    k_lcc_hook<<<prune_blocks(C * 32), PR_THREADS, 0, st>>>(off, idx, C, parent);
    C2B_KERNEL_CHECK();
  }
  k_lcc_label<<<prune_blocks(n), PR_THREADS, 0, st>>>(parent, n, size);
  C2B_KERNEL_CHECK();
  k_lcc_pick<<<(unsigned)std::min<uint64_t>(prune_blocks(n), (uint64_t)ctx->sm_count * 8), PR_THREADS, 0, st>>>(size, n,
                                                                                                               best);
  C2B_KERNEL_CHECK();
  // flags
  k_prune_count<<<prune_blocks(C * 32), PR_THREADS, 0, st>>>(off, idx, C, parent, best, cam_cnt, pt_cnt);
  C2B_KERNEL_CHECK();
  if (O) {
    k_prune_obs_words<<<prune_blocks(C * 32), PR_THREADS, 0, st>>>(off, idx, C, parent, best, cam_cnt, pt_cnt, w_obs);
    C2B_KERNEL_CHECK();
  }
  k_prune_flag_words<<<prune_blocks(C), PR_THREADS, 0, st>>>(cam_cnt, C, 3u, w_cam);
  C2B_KERNEL_CHECK();
  if (P) {
    k_prune_flag_words<<<prune_blocks(P), PR_THREADS, 0, st>>>(pt_cnt, P, 1u, w_pt);
    C2B_KERNEL_CHECK();
  }
  // ranks: popcount per word, exclusive scan, totals = (C', P', O')
  const uint64_t w_all = wo + wc + wp;
  k_word_popc<<<prune_blocks(w_all), PR_THREADS, 0, st>>>(w_obs, w_all, x_obs);
  C2B_KERNEL_CHECK();
  C2B_TRY(exclusive_scan_u32(st, x_cam, x_cam, wc, totals + 0, ctx->scan_tmp));
  C2B_TRY(exclusive_scan_u32(st, x_pt, x_pt, wp, totals + 1, ctx->scan_tmp));
  C2B_TRY(exclusive_scan_u32(st, x_obs, x_obs, wo, totals + 2, ctx->scan_tmp));
  // gathers
  if (O) {
    k_prune_write_obs<<<prune_blocks(O), PR_THREADS, 0, st>>>(idx, in.uv->as<double2>(), O, w_obs, x_obs, w_pt, x_pt,
                                                             out.idx->as<uint32_t>(), out.uv->as<double2>());
    C2B_KERNEL_CHECK();
  }
  k_prune_write_cams<<<prune_blocks(15 * C), PR_THREADS, 0, st>>>(in.cams->as<double>(), off, C, w_cam, x_cam, w_obs,
                                                                 x_obs, totals, out.cams->as<double>(),
                                                                 out.off->as<uint64_t>());
  C2B_KERNEL_CHECK();
  if (P) {
    k_prune_write_pts<<<prune_blocks(3 * P), PR_THREADS, 0, st>>>(in.pts->as<double>(), P, w_pt, x_pt,
                                                                 out.pts->as<double>());
    C2B_KERNEL_CHECK();
  }
  return C2B_OK;
}

// BAProblem::cull's loop:  culled = f(orig); prev = counts(orig); while counts(culled) != prev: prev =
// counts(culled); culled = f(culled).  sets[*cur] holds the input; on return sets[*cur] holds the result and
// (*C, *P, *O) its sizes.  The buffers of the other set are grown here to the input's sizes (sizes only shrink).
inline int prune_fixed_point(c2b_ctx *ctx, PruneSet sets[2], int *cur, uint64_t *C, uint64_t *P, uint64_t *O,
                             uint32_t *iterations) {
  cudaStream_t st = ctx->stream;
  const PruneSet &o = sets[*cur ^ 1];
  C2B_TRY(o.cams->ensure(std::max<uint64_t>(*C, 1) * 120));
  C2B_TRY(o.pts->ensure(std::max<uint64_t>(*P, 1) * 24));
  C2B_TRY(o.off->ensure((*C + 1) * 8));
  C2B_TRY(o.idx->ensure(std::max<uint64_t>(*O, 1) * 4));
  C2B_TRY(o.uv->ensure(std::max<uint64_t>(*O, 1) * 16));
  C2B_TRY(ctx->pr_small.ensure(64));
  C2B_TRY(ctx->h_small.ensure(256));
  uint32_t *totals = ctx->pr_small.as<uint32_t>() + 4;  // after the 8-byte component key
  uint32_t *h = ctx->h_small.as<uint32_t>();
  uint64_t prev_c, prev_p;
  *iterations = 0;
  do {
    prev_c = *C;
    prev_p = *P;
    ++*iterations;
    if (*C == 0) {
      // largest_connected_component returns the problem as it is (no cameras: no observations), and
      // remove_singletons keeps no point (none is observed).  offsets[0] of the current set is already 0.
      *P = 0;
      *O = 0;
    } else {
      C2B_TRY(prune_apply(ctx, sets[*cur], sets[*cur ^ 1], *C, *P, *O, totals));
      C2B_CUDA(cudaMemcpyAsync(h, totals, 12, cudaMemcpyDeviceToHost, st));
      C2B_CUDA(cudaStreamSynchronize(st));
      *C = h[0];
      *P = h[1];
      *O = h[2];
      *cur ^= 1;
    }
  } while (*C != prev_c || *P != prev_p);
  return C2B_OK;
}

}  // namespace c2b
