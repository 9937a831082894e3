// c2b_common.cuh — context, error plumbing, grow-only device buffers.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>
#if defined(__linux__)
#include <sys/syscall.h>
#include <unistd.h>
#endif

#include "../../include/city2ba_cuda.h"

namespace c2b {

// thread-local last error (c2b_last_error)
inline std::string &last_error_ref() {
  static thread_local std::string s;
  return s;
}
inline int set_error(int code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  last_error_ref() = buf;
  return code;
}

#define C2B_CUDA(call)                                                                        \
  do {                                                                                        \
    cudaError_t _e = (call);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      return c2b::set_error(_e == cudaErrorMemoryAllocation ? C2B_ERR_OOM : C2B_ERR_CUDA,     \
                            "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
    }                                                                                         \
  } while (0)

#define C2B_TRY(call)        \
  do {                       \
    int _s = (call);         \
    if (_s != C2B_OK) return _s; \
  } while (0)

// every kernel launch in the library is followed by this macro: it also counts launches
// (c2b_kernel_launches, used by bench.py's gpu_launches)
inline std::atomic<uint64_t> &launch_counter() {
  static std::atomic<uint64_t> n{0};
  return n;
}
#define C2B_KERNEL_CHECK()           \
  do {                               \
    ++c2b::launch_counter();         \
    C2B_CUDA(cudaGetLastError());    \
  } while (0)

// grow-only device buffer, freed by its destructor: its owner makes the buffer's device current first
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(DevBuf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, (size_t)0)) {}
  DevBuf &operator=(DevBuf &&o) noexcept {
    if (this != &o) {
      release();
      p = std::exchange(o.p, nullptr);
      cap = std::exchange(o.cap, (size_t)0);
    }
    return *this;
  }
  ~DevBuf() { release(); }
  int ensure(size_t bytes) {
    if (bytes <= cap) return C2B_OK;
    release();
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      e = cudaMalloc(&p, bytes);
      want = bytes;
    }
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      p = nullptr;
      return set_error(C2B_ERR_OOM, "cudaMalloc(%zu bytes) failed: %s", bytes,
                       cudaGetErrorString(e));
    }
    cap = want;
    return C2B_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T *as() const {
    return reinterpret_cast<T *>(p);
  }
};

// grow-only pinned host buffer
// Pinned host buffers are allocated on the NUMA node the GPU hangs off (c2b_init reads it from sysfs):
// with one process per GPU on a two-socket host, result slabs that land on the other socket cross the
// inter-socket link on their way out of every GPU at once.  Done by setting the calling thread's memory
// policy to MPOL_PREFERRED(node) around the allocation only; C2B_NUMA_LOCAL=0 switches it off.
struct NumaPreferred {
  bool active = false;
  explicit NumaPreferred(int node) {
#if defined(__linux__)
    if (node < 0 || node >= 1024) return;
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    active = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, 1025ul) == 0;
#else
    (void)node;
#endif
  }
  ~NumaPreferred() {
#if defined(__linux__)
    if (active) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
#endif
  }
};

struct PinBuf {
  void *p = nullptr;
  size_t cap = 0;
  int node = -1;  // NUMA node of the GPU these buffers feed (-1: unknown / off)
  bool portable = false;  // every device of the process may DMA into it (the one host CSR of c2b_visibility_graph_multi)
  PinBuf() = default;
  PinBuf(PinBuf &&o) noexcept
      : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, (size_t)0)), node(o.node), portable(o.portable) {}
  PinBuf &operator=(PinBuf &&o) noexcept {
    if (this != &o) {
      release();
      p = std::exchange(o.p, nullptr);
      cap = std::exchange(o.cap, (size_t)0);
      node = o.node;
      portable = o.portable;
    }
    return *this;
  }
  ~PinBuf() { release(); }
  int ensure(size_t bytes) {
    if (bytes <= cap) return C2B_OK;
    release();
    // pinning costs ~0.5 s per GB on this pool's hosts (profiles/r02b_alloc_probe.txt): large buffers get
    // little slack, small ones a quarter
    size_t want = bytes + (bytes > (64u << 20) ? bytes / 32 : bytes / 4) + 256;
    NumaPreferred local(node);
    cudaError_t e = cudaHostAlloc(&p, want, portable ? cudaHostAllocPortable : cudaHostAllocDefault);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      p = nullptr;
      return set_error(C2B_ERR_OOM, "cudaHostAlloc(%zu bytes) failed: %s", want,
                       cudaGetErrorString(e));
    }
    cap = want;
    return C2B_OK;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T *as() const {
    return reinterpret_cast<T *>(p);
  }
};

// An owned event or stream: create() makes it (a C2B_* status), the destructor or release() destroys it, with the
// owner's device current.  Converts to the raw handle for the runtime calls.
template <class H, cudaError_t (*make)(H *, unsigned), cudaError_t (*destroy)(H)>
class CudaHandle {
 public:
  CudaHandle() = default;
  CudaHandle(CudaHandle &&o) noexcept : h_(std::exchange(o.h_, nullptr)) {}
  CudaHandle &operator=(CudaHandle &&o) noexcept {
    if (this != &o) {
      release();
      h_ = std::exchange(o.h_, nullptr);
    }
    return *this;
  }
  ~CudaHandle() { release(); }
  int create(unsigned flags = 0) {
    release();
    C2B_CUDA(make(&h_, flags));
    return C2B_OK;
  }
  void release() {
    if (h_) destroy(h_);
    h_ = nullptr;
  }
  operator H() const { return h_; }

 private:
  H h_ = nullptr;
};
using Event = CudaHandle<cudaEvent_t, cudaEventCreateWithFlags, cudaEventDestroy>;
using Stream = CudaHandle<cudaStream_t, cudaStreamCreateWithFlags, cudaStreamDestroy>;

static_assert(!std::is_copy_constructible<DevBuf>::value && !std::is_copy_constructible<PinBuf>::value &&
                  !std::is_copy_constructible<Event>::value && !std::is_copy_constructible<Stream>::value,
              "owners of device resources are move-only");

struct CtxExtra;  // per-context state of c2b_api.cu (tunables, caches, BAL buffers)

enum StageEvent {
  EV_START = 0,
  EV_H2D,
  EV_PREP,
  EV_CULL,
  EV_SORT,
  EV_TRAVERSE,
  EV_COMPACT,
  EV_D2H,
  EV_COUNT
};

}  // namespace c2b

struct c2b_scene {
  int device = 0;  // the scene may outlive the ctx that built it; keep the ordinal, not the ctx
  uint64_t n_tris = 0;   // after dropping degenerate index triples
  uint64_t n_nodes = 0;  // 2*n_tris - 1 (0 when empty)
  float lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
  c2b::DevBuf nodes;  // float4[2*n_nodes]: {lo.xyz, escape}, {hi.xyz, leaf tri slot or -1}
  c2b::DevBuf tris;   // float4[3*n_tris]: v0, v1, v2 in leaf (Morton) order
};

// Owns everything it lists; ~c2b_ctx (c2b_api.cu, where CtxExtra is complete) runs with `device` current.  The
// streams come first so that they are destroyed last.
struct c2b_ctx {
  int device = 0;
  int sm_count = 148;
  c2b::Stream stream;
  c2b::Stream copy_stream;
  c2b::Stream aux_stream;  // leaf lists beside the plan (visibility_grid_fused)
  std::unique_ptr<c2b::CtxExtra> extra;
  c2b::Event ev[c2b::EV_COUNT];

  // resident problem
  uint64_t C = 0, P = 0;
  c2b::DevBuf cams_all;      // host-buffer call: all of the call's cameras (its batches are slices of it)
  c2b::DevBuf cams;          // double[15*C] as given
  c2b::DevBuf cam_center;    // double[3*C]  SoA: x[C], y[C], z[C]
  c2b::DevBuf pts;           // double[3*P]  SoA: x[P], y[P], z[P] (streamed by the cull kernels)
  c2b::DevBuf pts_aos;       // double[3*P]  as given (24 B records for the per-candidate gathers)
  c2b::DevBuf stage;         // staging for H2D of AoS inputs
  c2b::PinBuf pin_in;        // pinned staging for pageable callers

  // grid over points
  c2b::DevBuf cell_of_pt, cell_start, cell_cursor, grid_x, grid_y, grid_z, grid_idx;

  // candidate pool + sort
  c2b::DevBuf pool_key, pool_uv, cam_count, counters;
  c2b::DevBuf sort_keys[2], sort_vals[2], sort_hist;
  c2b::DevBuf scan_tmp[3];
  uint64_t pool_capacity = 0;

  // traversal + compaction
  c2b::DevBuf vis_words, word_prefix;
  // device CSR, double-buffered so that the D2H copy of one camera batch overlaps the next batch
  c2b::DevBuf out_offsets[2], out_idx[2], out_uv[2];
  int out_sel = 0;
  uint64_t out_C = 0, out_O = 0;
  c2b::Event ev_fork, ev_join;
  c2b::Event ev_ready[2], ev_copied[2];
  c2b::DevBuf misc;  // small scratch (reductions)
  c2b::DevBuf tri_list, tri_count;  // per-camera leaf lists for list-driven traversal
  // fused grid schedule: per-camera plan (row points -> scratch slice), visible counts, CSR offsets
  c2b::DevBuf ev_off, vis_count, seg_off, scratch_idx, plan_rows, plan_row_count;
  int numa_node = -1;  // of the device, from sysfs (-1: unknown)

  // noise passes on host arrays: grow-only device copies kept between calls
  c2b::DevBuf nz_cams, nz_centers, nz_pts, nz_uv, nz_scratch;
  float noise_ms[3] = {0, 0, 0};  // last noise call: upload, statistics + kernels, download

  // LCC + remove_singletons (c2b_graph_cull.cuh): the host entry's two problem sets (the resident entry uses set 1
  // of cameras / points beside the resident arrays), union-find labels, component sizes, counts, ballot words
  c2b::DevBuf pr_cams[2], pr_pts[2], pr_off[2], pr_idx[2], pr_uv[2];
  c2b::DevBuf pr_parent, pr_size, pr_cam_cnt, pr_pt_cnt, pr_words, pr_prefix, pr_small;

  // host results
  c2b::PinBuf h_offsets, h_idx, h_uv, h_small;

  ~c2b_ctx();
};
