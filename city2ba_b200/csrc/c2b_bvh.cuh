// c2b_bvh.cuh — GPU LBVH build (replaces Embree's rtcCommitScene, src/bin/city2ba.rs:521).
//
// Pipeline: triangle bounds -> 63-bit Morton code of the centroid -> radix sort -> Karras 2012
// radix tree (one thread per internal node) -> bottom-up AABB refit -> threaded pre-order
// layout: node i's first child is i+1 and every node carries an ESCAPE index (the next node in
// pre-order outside its subtree), so traversal needs no stack.
//
// HBM layout (SoA float4, 32 B per node, 48 B per triangle):
//   nodes[2*i+0] = {lo.x, lo.y, lo.z, as_float(escape)}
//   nodes[2*i+1] = {hi.x, hi.y, hi.z, as_float(leaf ? triangle slot : -1)}
//   tris[3*s+k]  = {v_k.x, v_k.y, v_k.z, 0}   (s = leaf order = Morton order)
#pragma once
#include "c2b_common.cuh"
#include "c2b_sort.cuh"

namespace c2b {

__device__ __forceinline__ uint32_t float_to_ordered(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_float(uint32_t u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// bounds[0..2] = min xyz, bounds[3..5] = max xyz (ordered-uint encoding) over triangle vertices
__global__ void k_bvh_bounds(const float *__restrict__ xyz, const uint32_t *__restrict__ tri,
                             uint64_t nt, uint32_t *__restrict__ bounds) {
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nt;
       t += (uint64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      uint64_t v = tri[3 * t + j];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        float c = xyz[3 * v + k];
        lo[k] = fminf(lo[k], c);
        hi[k] = fmaxf(hi[k], c);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
      hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
    }
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      atomicMin(&bounds[k], float_to_ordered(lo[k]));
      atomicMax(&bounds[3 + k], float_to_ordered(hi[k]));
    }
  }
}

__device__ __forceinline__ uint64_t expand21(uint64_t v) {
  v &= 0x1fffffull;
  v = (v | (v << 32)) & 0x1f00000000ffffull;
  v = (v | (v << 16)) & 0x1f0000ff0000ffull;
  v = (v | (v << 8)) & 0x100f00f00f00f00full;
  v = (v | (v << 4)) & 0x10c30c30c30c30c3ull;
  v = (v | (v << 2)) & 0x1249249249249249ull;
  return v;
}

__global__ void k_bvh_morton(const float *__restrict__ xyz, const uint32_t *__restrict__ tri,
                             uint64_t nt, const uint32_t *__restrict__ bounds,
                             uint64_t *__restrict__ keys, uint32_t *__restrict__ vals) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nt) return;
  float c[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float a = xyz[3 * (uint64_t)tri[3 * t] + k], b = xyz[3 * (uint64_t)tri[3 * t + 1] + k],
          d = xyz[3 * (uint64_t)tri[3 * t + 2] + k];
    float lo = fminf(a, fminf(b, d)), hi = fmaxf(a, fmaxf(b, d));
    c[k] = 0.5f * lo + 0.5f * hi;
  }
  uint64_t q[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float lo = ordered_to_float(bounds[k]), hi = ordered_to_float(bounds[3 + k]);
    float ext = hi - lo;
    float u = ext > 0.0f ? (c[k] - lo) / ext : 0.0f;
    u = fminf(fmaxf(u, 0.0f), 1.0f);
    uint64_t v = (uint64_t)(u * 2097151.0f);
    q[k] = v > 2097151ull ? 2097151ull : v;
  }
  keys[t] = (expand21(q[0]) << 2) | (expand21(q[1]) << 1) | expand21(q[2]);
  vals[t] = (uint32_t)t;
}

// common-prefix length of sorted keys i and j (index tie-break), -1 when j is out of range
__device__ __forceinline__ int lbvh_delta(const uint64_t *__restrict__ keys, int64_t n, int64_t i,
                                          int64_t j) {
  if (j < 0 || j >= n) return -1;
  uint64_t a = keys[i], b = keys[j];
  if (a == b) return 64 + __clzll((unsigned long long)((uint64_t)i ^ (uint64_t)j));
  return __clzll((unsigned long long)(a ^ b));
}

// child encoding: internal node k -> k ; leaf k -> k | LEAF_BIT
constexpr uint32_t LEAF_BIT = 0x80000000u;

__global__ void k_bvh_karras(const uint64_t *__restrict__ keys, int64_t n,
                             uint32_t *__restrict__ left, uint32_t *__restrict__ right,
                             uint32_t *__restrict__ first, uint32_t *__restrict__ last,
                             uint32_t *__restrict__ parent_internal,
                             uint32_t *__restrict__ parent_leaf) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  int d = (lbvh_delta(keys, n, i, i + 1) - lbvh_delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
  int dmin = lbvh_delta(keys, n, i, i - d);
  int64_t lmax = 2;
  while (lbvh_delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
  int64_t l = 0;
  for (int64_t t = lmax >> 1; t >= 1; t >>= 1)
    if (lbvh_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
  int64_t j = i + l * d;
  int dnode = lbvh_delta(keys, n, i, j);
  int64_t s = 0;
  for (int64_t t = (l + 1) >> 1;; t = (t + 1) >> 1) {
    if (lbvh_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    if (t <= 1) break;
  }
  int64_t gamma = i + s * d + (d < 0 ? -1 : 0);
  int64_t lo = i < j ? i : j, hi = i < j ? j : i;
  uint32_t lc = (lo == gamma) ? ((uint32_t)gamma | LEAF_BIT) : (uint32_t)gamma;
  uint32_t rc = (hi == gamma + 1) ? ((uint32_t)(gamma + 1) | LEAF_BIT) : (uint32_t)(gamma + 1);
  left[i] = lc;
  right[i] = rc;
  first[i] = (uint32_t)lo;
  last[i] = (uint32_t)hi;
  if (lc & LEAF_BIT)
    parent_leaf[gamma] = (uint32_t)i;
  else
    parent_internal[gamma] = (uint32_t)i;
  if (rc & LEAF_BIT)
    parent_leaf[gamma + 1] = (uint32_t)i;
  else
    parent_internal[gamma + 1] = (uint32_t)i;
  if (i == 0) parent_internal[0] = 0xffffffffu;
}

// leaves: gather the triangle into its Morton slot, compute its box, then climb; the second
// thread to arrive at an internal node merges the two child boxes (boxes are re-read from global
// memory after a __threadfence, so they are complete).
__global__ void k_bvh_refit(const float *__restrict__ xyz, const uint32_t *__restrict__ tri,
                            const uint32_t *__restrict__ sorted_tri, int64_t n,
                            const uint32_t *__restrict__ left, const uint32_t *__restrict__ right,
                            const uint32_t *__restrict__ parent_internal,
                            const uint32_t *__restrict__ parent_leaf, float4 *__restrict__ tris_out,
                            float *leaf_box /*6n*/, float *int_box /*6(n-1)*/,
                            uint32_t *__restrict__ visit) {
  int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  uint64_t t = sorted_tri[s];
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    uint64_t v = tri[3 * t + j];
    float x = xyz[3 * v], y = xyz[3 * v + 1], z = xyz[3 * v + 2];
    tris_out[3 * s + j] = make_float4(x, y, z, 0.0f);
    lo[0] = fminf(lo[0], x);
    lo[1] = fminf(lo[1], y);
    lo[2] = fminf(lo[2], z);
    hi[0] = fmaxf(hi[0], x);
    hi[1] = fmaxf(hi[1], y);
    hi[2] = fmaxf(hi[2], z);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    leaf_box[6 * s + k] = lo[k];
    leaf_box[6 * s + 3 + k] = hi[k];
  }
  if (n == 1) return;
  uint32_t p = parent_leaf[s];
  while (p != 0xffffffffu) {
    __threadfence();
    if (atomicAdd(&visit[p], 1u) == 0u) return;  // first arrival: the sibling will finish
    __threadfence();
    uint32_t lc = left[p], rc = right[p];
    const volatile float *bl = (lc & LEAF_BIT) ? leaf_box + 6 * (uint64_t)(lc & ~LEAF_BIT)
                                               : int_box + 6 * (uint64_t)lc;
    const volatile float *br = (rc & LEAF_BIT) ? leaf_box + 6 * (uint64_t)(rc & ~LEAF_BIT)
                                               : int_box + 6 * (uint64_t)rc;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      int_box[6 * (uint64_t)p + k] = fminf(bl[k], br[k]);
      int_box[6 * (uint64_t)p + 3 + k] = fmaxf(bl[3 + k], br[3 + k]);
    }
    p = parent_internal[p];
  }
}

// pre-order index of a node covering leaves [f, ...]: 2f - k + d, where d = depth and k = number
// of right-child steps on the path from the root (see DESIGN.md); subtree of an internal node
// covering [f,l] has 2(l-f+1)-1 nodes.
__global__ void k_bvh_layout(int64_t n, const uint32_t *__restrict__ left,
                             const uint32_t *__restrict__ right, const uint32_t *__restrict__ first,
                             const uint32_t *__restrict__ last,
                             const uint32_t *__restrict__ parent_internal,
                             const uint32_t *__restrict__ parent_leaf,
                             const float *__restrict__ leaf_box, const float *__restrict__ int_box,
                             float4 *__restrict__ nodes) {
  int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = 2 * n - 1;
  if (id >= total) return;
  bool leaf = id >= n - 1;
  int64_t k_self = leaf ? id - (n - 1) : id;  // leaf slot or internal index
  uint32_t f = leaf ? (uint32_t)k_self : first[k_self];
  uint32_t l = leaf ? (uint32_t)k_self : last[k_self];
  uint32_t depth = 0, rights = 0;
  uint32_t child_code = leaf ? ((uint32_t)k_self | LEAF_BIT) : (uint32_t)k_self;
  uint32_t p = (n == 1) ? 0xffffffffu : (leaf ? parent_leaf[k_self] : parent_internal[k_self]);
  while (p != 0xffffffffu) {
    ++depth;
    if (right[p] == child_code) ++rights;
    child_code = p;
    p = parent_internal[p];
  }
  uint64_t pre = 2ull * f - rights + depth;
  uint64_t size = 2ull * (l - f + 1) - 1;
  const float *b = leaf ? leaf_box + 6 * (uint64_t)k_self : int_box + 6 * (uint64_t)k_self;
  int esc = (int)(pre + size);
  // second w field: leaf -> triangle slot (>= 0); internal -> -(pre-order index of the RIGHT child) - 1
  // (<= -3; the left child is pre + 1), which lane = node traversals need to push both children
  int leaf_slot = (int)k_self;
  if (!leaf) {
    const uint32_t lc = left[k_self];
    const uint32_t split = (lc & LEAF_BIT) ? (lc & ~LEAF_BIT) : last[lc];
    leaf_slot = -(int)(pre + 2ull * (split - f + 1)) - 1;
  }
  nodes[2 * pre] = make_float4(b[0], b[1], b[2], __int_as_float(esc));
  nodes[2 * pre + 1] = make_float4(b[3], b[4], b[5], __int_as_float(leaf_slot));
}

struct BvhScratch {
  DevBuf xyz, tri, bounds, keys[2], vals[2], hist, left, right, first, last, par_i, par_l, leaf_box,
      int_box, visit;
  DevBuf scan_tmp[3];
};

// h_tri holds only valid (non-degenerate, in-range) triples.
inline int bvh_build(c2b_ctx *ctx, c2b_scene *sc, const float *h_xyz, uint64_t nv,
                     const uint32_t *h_tri, uint64_t nt) {
  cudaStream_t st = ctx->stream;
  sc->n_tris = nt;
  sc->n_nodes = nt ? 2 * nt - 1 : 0;
  if (nt == 0) return C2B_OK;
  if (nt >= 0x7fffffffull / 2) return set_error(C2B_ERR_INVALID, "too many triangles (%llu)", (unsigned long long)nt);
  BvhScratch s;
  C2B_TRY(s.xyz.ensure(nv * 12));
  C2B_TRY(s.tri.ensure(nt * 12));
  C2B_CUDA(cudaMemcpyAsync(s.xyz.p, h_xyz, nv * 12, cudaMemcpyHostToDevice, st));
  C2B_CUDA(cudaMemcpyAsync(s.tri.p, h_tri, nt * 12, cudaMemcpyHostToDevice, st));
  C2B_TRY(s.bounds.ensure(24));
  uint32_t init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
  C2B_CUDA(cudaMemcpyAsync(s.bounds.p, init, 24, cudaMemcpyHostToDevice, st));
  int nb = (int)((nt + 255) / 256);
  int nb_red = nb < 4 * ctx->sm_count ? nb : 4 * ctx->sm_count;
  k_bvh_bounds<<<nb_red, 256, 0, st>>>(s.xyz.as<float>(), s.tri.as<uint32_t>(), nt,
                                       s.bounds.as<uint32_t>());
  C2B_KERNEL_CHECK();
  for (int b = 0; b < 2; ++b) {
    C2B_TRY(s.keys[b].ensure(nt * 8));
    C2B_TRY(s.vals[b].ensure(nt * 4));
  }
  k_bvh_morton<<<nb, 256, 0, st>>>(s.xyz.as<float>(), s.tri.as<uint32_t>(), nt,
                                   s.bounds.as<uint32_t>(), s.keys[0].as<uint64_t>(),
                                   s.vals[0].as<uint32_t>());
  C2B_KERNEL_CHECK();
  uint64_t *keys[2] = {s.keys[0].as<uint64_t>(), s.keys[1].as<uint64_t>()};
  uint32_t *vals[2] = {s.vals[0].as<uint32_t>(), s.vals[1].as<uint32_t>()};
  int res = 0;
  C2B_TRY(radix_sort_pairs(st, keys, vals, nt, 63, s.hist, s.scan_tmp, &res));
  C2B_TRY(sc->tris.ensure(nt * 48));
  C2B_TRY(sc->nodes.ensure(sc->n_nodes * 32));
  C2B_TRY(s.leaf_box.ensure(nt * 24));
  uint64_t ni = nt - 1;
  if (ni) {
    C2B_TRY(s.left.ensure(ni * 4));
    C2B_TRY(s.right.ensure(ni * 4));
    C2B_TRY(s.first.ensure(ni * 4));
    C2B_TRY(s.last.ensure(ni * 4));
    C2B_TRY(s.par_i.ensure(ni * 4));
    C2B_TRY(s.int_box.ensure(ni * 24));
    C2B_TRY(s.visit.ensure(ni * 4));
    C2B_CUDA(cudaMemsetAsync(s.visit.p, 0, ni * 4, st));
    C2B_TRY(s.par_l.ensure(nt * 4));
    k_bvh_karras<<<(int)((ni + 255) / 256), 256, 0, st>>>(
        keys[res], (int64_t)nt, s.left.as<uint32_t>(), s.right.as<uint32_t>(),
        s.first.as<uint32_t>(), s.last.as<uint32_t>(), s.par_i.as<uint32_t>(),
        s.par_l.as<uint32_t>());
    C2B_KERNEL_CHECK();
  }
  k_bvh_refit<<<nb, 256, 0, st>>>(s.xyz.as<float>(), s.tri.as<uint32_t>(), vals[res], (int64_t)nt,
                                  s.left.as<uint32_t>(), s.right.as<uint32_t>(),
                                  s.par_i.as<uint32_t>(), s.par_l.as<uint32_t>(),
                                  sc->tris.as<float4>(), s.leaf_box.as<float>(),
                                  s.int_box.as<float>(), s.visit.as<uint32_t>());
  C2B_KERNEL_CHECK();
  k_bvh_layout<<<(int)((sc->n_nodes + 255) / 256), 256, 0, st>>>(
      (int64_t)nt, s.left.as<uint32_t>(), s.right.as<uint32_t>(), s.first.as<uint32_t>(),
      s.last.as<uint32_t>(), s.par_i.as<uint32_t>(), s.par_l.as<uint32_t>(),
      s.leaf_box.as<float>(), s.int_box.as<float>(), sc->nodes.as<float4>());
  C2B_KERNEL_CHECK();
  uint32_t hb[6];
  C2B_CUDA(cudaMemcpyAsync(hb, s.bounds.p, 24, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  for (int k = 0; k < 3; ++k) {
    uint32_t a = hb[k], b = hb[3 + k];
    uint32_t ua = (a & 0x80000000u) ? (a & 0x7fffffffu) : ~a;
    uint32_t ub = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b;
    memcpy(&sc->lo[k], &ua, 4);
    memcpy(&sc->hi[k], &ub, 4);
  }
  return C2B_OK;
}

}  // namespace c2b
