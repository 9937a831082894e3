// c2b_api.cu — the extern "C" boundary of libcity2ba_cuda.so (include/city2ba_cuda.h) and the
// host-side orchestration of the kernels: upload -> (grid build) -> cull -> radix sort ->
// warp-cooperative BVH traversal -> compaction -> download.
#include <algorithm>
#include <charconv>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#if defined(__linux__)
#include <cerrno>
#include <fcntl.h>
#include <unistd.h>
#include <sys/mman.h>
#include <sys/stat.h>
#endif

#include "c2b_bal.cuh"
#include "c2b_bal_read.cuh"
#include "c2b_bvh.cuh"
#include "c2b_common.cuh"
#include "c2b_compact.cuh"
#include "c2b_cull.cuh"
#include "c2b_fused.cuh"
#include "c2b_graph_cull.cuh"
#include "c2b_internal.h"
#include "c2b_math.cuh"
#include "c2b_mismatch.cuh"
#include "c2b_noise.cuh"
#include "c2b_sample.cuh"
#include "c2b_sort.cuh"
#include "c2b_traverse.cuh"

using namespace c2b;

namespace {

// internal status of the resident pipeline: the camera batch holds more than 2^32 pairs / candidates.
// c2b_visibility_graph halves the batch and retries; the public resident entry reports C2B_ERR_INVALID.
constexpr int ERR_TOO_LARGE = -100;

inline int bit_length(uint64_t v) {
  int b = 0;
  while (v) {
    ++b;
    v >>= 1;
  }
  return b;
}

// smallest double T with sqrt_rn(T) >= max_dist, so that  m2 < T  <=>  sqrt_rn(m2) < max_dist
// (sqrt_rn is monotone non-decreasing).  NaN / non-positive max_dist admit nothing.
double exact_sq_threshold(double max_dist) {
  if (!(max_dist > 0.0)) return 0.0;  // m2 < 0 is never true (and NaN compares false)
  if (std::isinf(max_dist)) return INFINITY;
  double x = max_dist * max_dist;
  if (std::isinf(x)) x = 1.7976931348623157e308;
  while (x > 0.0 && std::sqrt(x) >= max_dist) x = std::nextafter(x, 0.0);
  while (std::sqrt(x) < max_dist) {
    double nx = std::nextafter(x, INFINITY);
    if (std::isinf(nx)) return nx;
    x = nx;
  }
  return x;
}

// Small read-backs (counters) go through a kernel that stores into mapped pinned host memory, not
// through cudaMemcpy: a memcpy would queue behind the bulk result transfer on the D2H copy engine
// and stall the next camera batch.
__global__ void k_copy_words(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst, int n) {
  if ((int)threadIdx.x < n) dst[threadIdx.x] = src[threadIdx.x];
}

__global__ void k_iota_u32(uint32_t *v, uint64_t n) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = (uint32_t)i;
}

inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

struct GridCache {
  bool valid = false;
  double max_dist = 0;
  uint64_t points_version = 0;
  GridDesc desc;
  uint64_t n_cells = 0;
  // hinted: the cells cover only what the cameras of that call could reach (their centres' box grown by
  // max_dist), because cells of side max_dist/4 over the bounding box of ALL points would have exceeded the
  // cell budget (outliers); such a grid serves a later call only if its cameras stay inside the hint
  bool hinted = false;
  double hint_lo[3] = {0, 0, 0}, hint_hi[3] = {0, 0, 0};
};

// Measurement / test hooks (include/city2ba_cuda.h, c2b_tune).  Defaults are the product's behaviour; the
// environment variables of the same names in upper case with a C2B_ prefix are read ONCE, in c2b_init.
struct Tunables {
  int parts_log2 = -1;             // tickets per camera = 2^k; -1 = automatic
  int trilist_cap = 128;           // entries of a camera's leaf list before it counts as overflowed
  uint64_t max_pairs = 0xffffffffull;  // 32-bit scratch offsets: pairs inside max_dist per resident pass
  int hoist_max = 64;              // leaf lists up to this length get per-camera triangle records (<= FU_HOIST)
  int packet_bvh = 1;              // list overflow: 1 = lane = node packet traversal, 0 = per-ray stackless walk
  int trilist_warp = -1;           // leaf lists by one warp per camera (1) / one thread (0); -1 = by camera count
  int batches = 0;                 // camera batches of the host-buffer call; 0 = automatic
  double grid_cell_factor = 0.25;  // point-grid cell side / max_dist
  int stage_threads = 4;           // host threads staging a pageable input through the pinned ring; 0 = let the
                                   // driver copy from pageable memory itself
  int cold_staged = 1;             // first host-buffer call on a ctx returns its CSR in unpinned memory filled
                                   // through a pinned ring (0: pin the result arrays at once, as later calls do)
  int optimistic = 1;              // launch a pass's kernels without waiting for the plan's totals when the
                                   // previous pass on this ctx left sizes to go by (one host sync instead of three)
  uint64_t bal_chunk_bytes = 1ull << 25;  // BAL writer: bytes per chunk (device buffer, pinned ring slot)
};

// Pageable host memory backed by transparent huge pages (mmap + MADV_HUGEPAGE): what the FIRST host-buffer call
// on a ctx returns its CSR in.  Pinning 1.1 GB takes 0.55-1.3 s on this pool's hosts
// (profiles/r02b_alloc_probe.txt, r02l_cold_probe.json) — far longer than computing and transferring the result —
// so a one-shot caller gets an unpinned array filled through a small pinned ring by host threads (Drainer);
// a second call on the same ctx is no one-shot any more and switches to pinned arrays.
struct PageBuf {
  void *p = nullptr;
  size_t cap = 0;
  PageBuf() = default;
  PageBuf(PageBuf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, (size_t)0)) {}
  PageBuf &operator=(PageBuf &&o) noexcept {
    if (this != &o) {
      release();
      p = std::exchange(o.p, nullptr);
      cap = std::exchange(o.cap, (size_t)0);
    }
    return *this;
  }
  ~PageBuf() { release(); }
  int ensure_fresh(size_t bytes) {  // contents are not kept
    if (bytes <= cap) return C2B_OK;
    release();
    const size_t want = (bytes + bytes / 16 + (2u << 20)) & ~(size_t)((2u << 20) - 1);
#if defined(__linux__)
    void *q = mmap(nullptr, want, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (q == MAP_FAILED) return set_error(C2B_ERR_OOM, "mmap(%zu bytes) failed", want);
    (void)madvise(q, want, MADV_HUGEPAGE);
#else
    void *q = malloc(want);
    if (!q) return set_error(C2B_ERR_OOM, "malloc(%zu bytes) failed", want);
#endif
    p = q;
    cap = want;
    return C2B_OK;
  }
  void release() {
#if defined(__linux__)
    if (p) munmap(p, cap);
#else
    free(p);
#endif
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T *as() const {
    return reinterpret_cast<T *>(p);
  }
};
static_assert(!std::is_copy_constructible<PageBuf>::value, "PageBuf is move-only");

// Device -> pageable host memory through a pinned ring: `threads` host threads, each with its own stream and two
// 2 MB ring slots, take 2 MB chunks off a queue: DMA into a slot, then memcpy the slot to its destination (the
// first touch of the destination's pages happens there, in parallel).  submit() never blocks the caller.
class Drainer {
 public:
  static constexpr size_t CH = 2u << 20;  // pinning the ring itself costs ~1 ms per MB: keep it small
  int start(int device, int threads, char *ring) {
    n_ = threads;
    for (int t = 0; t < n_; ++t)
      workers_.emplace_back([this, device, t, ring]() { loop(device, ring + (size_t)t * 2 * CH); });
    return C2B_OK;
  }
  // bytes from dev_src (valid once `ready` has fired on its stream) to host_dst; `batch` tags the chunks
  void submit(const void *dev_src, void *host_dst, size_t bytes, cudaEvent_t ready, int batch) {
    std::lock_guard<std::mutex> lk(mu_);
    if ((size_t)batch >= dma_left_.size()) dma_left_.resize((size_t)batch + 1, 0);
    for (size_t off = 0; off < bytes; off += CH) {
      q_.push_back(Chunk{static_cast<const char *>(dev_src) + off, static_cast<char *>(host_dst) + off,
                         std::min(CH, bytes - off), ready, batch});
      ++dma_left_[(size_t)batch];
      ++left_;
    }
    cv_.notify_all();
  }
  // every chunk of `batch` has left the device (its device buffers may be overwritten)
  void wait_dma(int batch) {
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] { return (size_t)batch >= dma_left_.size() || dma_left_[(size_t)batch] == 0 || err_ != cudaSuccess; });
  }
  // everything submitted so far has landed in host memory
  void wait_all() {
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] { return left_ == 0 || err_ != cudaSuccess; });
  }
  // everything submitted has landed in host memory; joins the threads
  cudaError_t finish() {
    {
      std::unique_lock<std::mutex> lk(mu_);
      cv_done_.wait(lk, [&] { return left_ == 0 || err_ != cudaSuccess; });
      quit_ = true;
    }
    cv_.notify_all();
    for (auto &w : workers_) w.join();
    workers_.clear();
    return err_;
  }
  ~Drainer() {
    if (!workers_.empty()) (void)finish();
  }

 private:
  struct Chunk {
    const char *src;
    char *dst;
    size_t n;
    cudaEvent_t ready;
    int batch;
  };
  void loop(int device, char *slots) {
    cudaError_t e = cudaSetDevice(device);
    Stream st;  // destroyed on this thread, with `device` current
    if (e == cudaSuccess && st.create(cudaStreamNonBlocking) != C2B_OK) e = cudaGetLastError();
    for (int turn = 0;; ++turn) {
      Chunk c;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return !q_.empty() || quit_ || err_ != cudaSuccess; });
        if (q_.empty() || err_ != cudaSuccess) break;
        c = q_.front();
        q_.pop_front();
      }
      char *slot = slots + (size_t)(turn & 1) * CH;
      if (e == cudaSuccess) e = cudaStreamWaitEvent(st, c.ready, 0);
      if (e == cudaSuccess) e = cudaMemcpyAsync(slot, c.src, c.n, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (e != cudaSuccess) err_ = e;
        --dma_left_[(size_t)c.batch];
      }
      cv_done_.notify_all();
      if (e == cudaSuccess) memcpy(c.dst, slot, c.n);
      {
        std::lock_guard<std::mutex> lk(mu_);
        --left_;
      }
      cv_done_.notify_all();
      if (e != cudaSuccess) break;
    }
    cv_done_.notify_all();
  }
  int n_ = 0;
  std::vector<std::thread> workers_;
  std::mutex mu_;
  std::condition_variable cv_, cv_done_;
  std::deque<Chunk> q_;
  std::vector<size_t> dma_left_;
  size_t left_ = 0;
  bool quit_ = false;
  cudaError_t err_ = cudaSuccess;
};

// what the previous host-buffer call cost per camera: decides whether the next one is bound by the result
// transfer or by the kernels (camera batch policy of c2b_visibility_graph)
struct CallHist {
  bool valid = false;
  double ms_compute_per_cam = 0, d2h_bytes_per_cam = 0;
};

// what the previous resident pass (grid schedule) found: lets the next one launch its kernels without waiting
// for the plan's totals (the kernels check every assumption and flag a misfit)
struct PassMemo {
  bool valid = false, any_overflow = false, big = false;
};

}  // namespace

struct c2b::CtxExtra {
  Tunables tun;
  CallHist hist;
  PassMemo memo;
  bool grid_locked = false;  // inside c2b_visibility_graph: the grid was built for all of the call's cameras
  PageBuf pg_idx, pg_uv;     // first host-buffer call: unpinned result arrays (see PageBuf)
  PinBuf pin_out;            // and the ring they are filled through
  // BAL writer (c2b_bal.cuh): window lengths / offsets, two chunk buffers, camera 9-vectors, pinned chunk ring
  DevBuf bal_scan, bal_out[2], bal_vecs;
  PinBuf bal_ring;
  // BAL reader (c2b_bal_read.cuh): per-observation camera, per-camera counts, slow-token records of two chunks,
  // error offsets / token counter
  DevBuf bal_cam, bal_cnt, bal_slow[2], bal_small;
  // add_incorrect_correspondences (c2b_mismatch.cuh): per-camera counts / bases, selections + picks, flag / counters
  DevBuf mm_cnt, mm_sel, mm_small;
  GridCache grid;
  uint64_t points_version = 0;
  double pts_bounds[6] = {0, 0, 0, 0, 0, 0};
  bool have_points = false, have_cameras = false, have_result = false;
  // the last pass was the host-buffer c2b_visibility_graph (only its last batch stays).  have_result is already false
  // then; this only picks the message with which c2b_cull_problem_resident refuses
  bool host_call_last = false;
  uint64_t res_candidates = 0;
};

c2b_ctx::~c2b_ctx() = default;

static bool tune(Tunables &t, const char *name, double v) {
  const std::string n(name);
  if (n == "parts_log2") t.parts_log2 = v < 0 ? -1 : std::min((int)v, 2);
  else if (n == "trilist_cap") t.trilist_cap = std::max(1, (int)v);
  else if (n == "max_pairs") t.max_pairs = std::min<uint64_t>(0xffffffffull, v < 0 ? 0 : (uint64_t)v);
  else if (n == "hoist_max") t.hoist_max = std::min(std::max(0, (int)v), 64);
  else if (n == "packet_bvh") t.packet_bvh = v != 0;
  else if (n == "trilist_warp") t.trilist_warp = v < 0 ? -1 : (v != 0);
  else if (n == "batches") t.batches = std::max(0, (int)v);
  else if (n == "grid_cell_factor") t.grid_cell_factor = v > 0 ? v : 0.25;
  else if (n == "stage_threads") t.stage_threads = std::min(std::max(0, (int)v), 16);
  else if (n == "optimistic") t.optimistic = v != 0;
  else if (n == "cold_staged") t.cold_staged = v != 0;
  else if (n == "bal_chunk_bytes") t.bal_chunk_bytes = (uint64_t)(v >= 4096.0 ? std::min(v, 1073741824.0) : 4096.0) & ~7ull;
  else return false;
  return true;
}

static float scene_abs_max(const c2b_scene *scene) {
  float m = 0.0f;
  if (scene)
    for (int k = 0; k < 3; ++k) m = std::max(m, std::max(std::fabs(scene->lo[k]), std::fabs(scene->hi[k])));
  if (!std::isfinite(m)) m = 3.0e38f;
  return m;
}


extern "C" {

const char *c2b_last_error(void) { return last_error_ref().c_str(); }
int c2b_abi_version(void) { return C2B_ABI_VERSION; }
uint64_t c2b_kernel_launches(void) { return launch_counter(); }

int c2b_init(int device, c2b_ctx **out) {
  if (!out) return set_error(C2B_ERR_INVALID, "c2b_init: out is null");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    (void)cudaGetLastError();
    return set_error(C2B_ERR_NO_DEVICE, "no CUDA device visible (%s); this library has no CPU fallback",
                     e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  }
  if (device < 0 || device >= n) return set_error(C2B_ERR_INVALID, "device %d out of range [0,%d)", device, n);
  C2B_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  C2B_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return set_error(C2B_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only",
                     device, prop.major, prop.minor);
  // freed with everything built so far by any early return below (the device is current)
  std::unique_ptr<c2b_ctx> ctx(new (std::nothrow) c2b_ctx());
  if (!ctx) return set_error(C2B_ERR_OOM, "out of host memory");
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  C2B_TRY(ctx->stream.create(cudaStreamNonBlocking));
  for (int i = 0; i < EV_COUNT; ++i) C2B_TRY(ctx->ev[i].create());
  C2B_TRY(ctx->copy_stream.create(cudaStreamNonBlocking));
  C2B_TRY(ctx->aux_stream.create(cudaStreamNonBlocking));
  C2B_TRY(ctx->ev_fork.create(cudaEventDisableTiming));
  C2B_TRY(ctx->ev_join.create(cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) {
    C2B_TRY(ctx->ev_ready[i].create(cudaEventDisableTiming));
    C2B_TRY(ctx->ev_copied[i].create(cudaEventDisableTiming));
  }
  // NUMA node of the device (sysfs), for the pinned staging / result buffers (see PinBuf)
  {
    int node = -1;
    const char *off = getenv("C2B_NUMA_LOCAL");
    char bus[32] = {0};
    if (!(off && atoi(off) == 0) && cudaDeviceGetPCIBusId(bus, sizeof bus, device) == cudaSuccess) {
      for (char *c = bus; *c; ++c) *c = (char)tolower((unsigned char)*c);
      const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
      if (FILE *f = fopen(path.c_str(), "r")) {
        if (fscanf(f, "%d", &node) != 1) node = -1;
        fclose(f);
      }
    }
    (void)cudaGetLastError();
    ctx->numa_node = node;
    for (PinBuf *b : {&ctx->pin_in, &ctx->h_offsets, &ctx->h_idx, &ctx->h_uv, &ctx->h_small}) b->node = node;
  }
  {  // tables of the noise draws (c2b_noise.cuh), one copy per device
    static double2 sc[256], ln[128];
    static std::once_flag once;
    std::call_once(once, [] { noise_tables_host(sc, ln); });
    C2B_CUDA(cudaMemcpyToSymbol(g_sc_tab, sc, sizeof sc));
    C2B_CUDA(cudaMemcpyToSymbol(g_ln_tab, ln, sizeof ln));
  }
  ctx->extra = std::make_unique<CtxExtra>();
  {
    struct { const char *env, *name; } hooks[] = {
        {"C2B_PARTS_LOG2", "parts_log2"}, {"C2B_TRILIST_CAP", "trilist_cap"}, {"C2B_MAX_PAIRS", "max_pairs"},
        {"C2B_HOIST_MAX", "hoist_max"}, {"C2B_PACKET_BVH", "packet_bvh"}, {"C2B_TRILIST_WARP", "trilist_warp"},
        {"C2B_BATCHES", "batches"}, {"C2B_GRID_CELL_FACTOR", "grid_cell_factor"},
        {"C2B_STAGE_THREADS", "stage_threads"}, {"C2B_OPTIMISTIC", "optimistic"}, {"C2B_COLD_STAGED", "cold_staged"},
        {"C2B_BAL_CHUNK_BYTES", "bal_chunk_bytes"}};
    for (auto &h : hooks)
      if (const char *e = getenv(h.env)) (void)tune(ctx->extra->tun, h.name, atof(e));
  }
  *out = ctx.release();
  return C2B_OK;
}

int c2b_tune(c2b_ctx *ctx, const char *name, double value) {
  if (!ctx || !name) return set_error(C2B_ERR_INVALID, "c2b_tune: null argument");
  if (!strcmp(name, "reset")) {
    ctx->extra->tun = Tunables();
    return C2B_OK;
  }
  if (!tune(ctx->extra->tun, name, value)) return set_error(C2B_ERR_INVALID, "c2b_tune: unknown hook '%s'", name);
  return C2B_OK;
}

void c2b_shutdown(c2b_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
  delete ctx;
}

// ---- scene -------------------------------------------------------------------------------------
int c2b_scene_create(c2b_ctx *ctx, const float *xyz, uint64_t nv, const uint32_t *tri, uint64_t nt,
                     c2b_scene **out) {
  if (!ctx || !out) return set_error(C2B_ERR_INVALID, "c2b_scene_create: null ctx/out");
  *out = nullptr;
  if ((nv && !xyz) || (nt && !tri)) return set_error(C2B_ERR_INVALID, "c2b_scene_create: null mesh arrays");
  C2B_CUDA(cudaSetDevice(ctx->device));
  std::vector<uint32_t> keep;
  keep.reserve(3 * nt);
  for (uint64_t i = 0; i < nt; ++i) {
    uint32_t a = tri[3 * i], b = tri[3 * i + 1], c = tri[3 * i + 2];
    if (a >= nv || b >= nv || c >= nv)
      return set_error(C2B_ERR_INVALID, "triangle %llu references vertex >= %llu",
                       (unsigned long long)i, (unsigned long long)nv);
    if (a == b || b == c || a == c) continue;  // zero-area (tobj `l` records): can never be hit
    keep.push_back(a);
    keep.push_back(b);
    keep.push_back(c);
  }
  c2b_scene *sc = new (std::nothrow) c2b_scene();
  if (!sc) return set_error(C2B_ERR_OOM, "out of host memory");
  sc->device = ctx->device;
  int rc = bvh_build(ctx, sc, xyz, nv, keep.data(), keep.size() / 3);
  if (rc != C2B_OK) {
    delete sc;  // ctx->device is current
    return rc;
  }
  *out = sc;
  return C2B_OK;
}

int c2b_scene_bounds(const c2b_scene *scene, float lower[3], float upper[3]) {
  if (!scene || !lower || !upper) return set_error(C2B_ERR_INVALID, "c2b_scene_bounds: null argument");
  for (int k = 0; k < 3; ++k) {
    lower[k] = scene->lo[k];
    upper[k] = scene->hi[k];
  }
  return C2B_OK;
}
uint64_t c2b_scene_num_triangles(const c2b_scene *scene) { return scene ? scene->n_tris : 0; }
uint64_t c2b_scene_num_nodes(const c2b_scene *scene) { return scene ? scene->n_nodes : 0; }
void c2b_scene_destroy(c2b_scene *scene) {
  if (!scene) return;
  cudaSetDevice(scene->device);
  delete scene;
}

// ---- ray-level entries ------------------------------------------------------------------------------
int c2b_occluded(c2b_ctx *ctx, const c2b_scene *scene, c2b_ray48 *rays, uint64_t n) {
  if (!ctx || !scene || (n && !rays)) return set_error(C2B_ERR_INVALID, "c2b_occluded: null argument");
  if (n == 0 || scene->n_nodes == 0) return C2B_OK;
  C2B_CUDA(cudaSetDevice(ctx->device));
  C2B_TRY(ctx->stage.ensure(n * sizeof(c2b_ray48)));
  C2B_TRY(ctx->counters.ensure(32));
  float absmax = 0.0f;
  for (int k = 0; k < 3; ++k) absmax = std::max(absmax, std::max(std::fabs(scene->lo[k]), std::fabs(scene->hi[k])));
  C2B_CUDA(cudaMemcpyAsync(ctx->stage.p, rays, n * sizeof(c2b_ray48), cudaMemcpyHostToDevice, ctx->stream));
  k_occluded_rays<false><<<blocks_for(n, 256), 256, 0, ctx->stream>>>(
      scene->nodes.as<float4>(), scene->tris.as<float4>(), (int)scene->n_nodes,
      ctx->stage.as<c2b_ray48>(), n, absmax, ctx->counters.as<unsigned long long>());
  C2B_KERNEL_CHECK();
  C2B_CUDA(cudaMemcpyAsync(rays, ctx->stage.p, n * sizeof(c2b_ray48), cudaMemcpyDeviceToHost, ctx->stream));
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));
  return C2B_OK;
}

int c2b_intersect(c2b_ctx *ctx, const c2b_scene *scene, c2b_ray48 *rays, uint64_t n) {
  if (!ctx || !scene || (n && !rays)) return set_error(C2B_ERR_INVALID, "c2b_intersect: null argument");
  if (n == 0) return C2B_OK;
  if (scene->n_nodes == 0) {
    for (uint64_t i = 0; i < n; ++i) rays[i].flags = 0;
    return C2B_OK;
  }
  C2B_CUDA(cudaSetDevice(ctx->device));
  C2B_TRY(ctx->stage.ensure(n * sizeof(c2b_ray48)));
  C2B_CUDA(cudaMemcpyAsync(ctx->stage.p, rays, n * sizeof(c2b_ray48), cudaMemcpyHostToDevice, ctx->stream));
  k_intersect_rays<<<blocks_for(n, 256), 256, 0, ctx->stream>>>(scene->nodes.as<float4>(), scene->tris.as<float4>(),
                                                                (int)scene->n_nodes, ctx->stage.as<c2b_ray48>(), n,
                                                                scene_abs_max(scene));
  C2B_KERNEL_CHECK();
  C2B_CUDA(cudaMemcpyAsync(rays, ctx->stage.p, n * sizeof(c2b_ray48), cudaMemcpyDeviceToHost, ctx->stream));
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));
  return C2B_OK;
}

int c2b_intersect1(c2b_ctx *ctx, const c2b_scene *scene, const float org[3], const float dir[3],
                   int *hit, float *tfar) {
  if (!ctx || !scene || !org || !dir || !hit || !tfar)
    return set_error(C2B_ERR_INVALID, "c2b_intersect1: null argument");
  c2b_ray48 r;
  memset(&r, 0, sizeof r);
  r.org_x = org[0];
  r.org_y = org[1];
  r.org_z = org[2];
  r.dir_x = dir[0];
  r.dir_y = dir[1];
  r.dir_z = dir[2];
  r.tfar = INFINITY;  // Ray::new(org, dir): tnear 0, tfar +inf
  C2B_TRY(c2b_intersect(ctx, scene, &r, 1));
  *hit = r.flags != 0;
  *tfar = r.flags ? r.tfar : INFINITY;
  return C2B_OK;
}

// ---- uploads ------------------------------------------------------------------------------------------
void c2b_vis_options_default(c2b_vis_options *opt) {
  if (!opt) return;
  opt->cull_mode = C2B_CULL_GRID;
  opt->occlusion = C2B_OCC_MESH;
  opt->endpoint_guard_rel = 0;
  opt->count_traversal = 0;
  opt->block_length = 20.0;
  opt->block_inset = 1.0;
  opt->predicate = C2B_PRED_WATERTIGHT;
  opt->reserved = 0;
}

// Host -> device copy of a caller's array on ctx->stream.  A pinned (or registered) source goes to the copy
// engine as it is.  A PAGEABLE one — what `points.as_ptr()` of a Rust Vec or a numpy array is — would be
// staged by the driver through its own bounce buffer on one thread; instead `stage_threads` host threads
// copy 2 MB chunks into the ctx's pinned ring (two slots per thread) and queue each chunk's DMA as soon as
// it is staged, so the host-side memcpy runs at several cores' bandwidth and overlaps the PCIe transfer.
int copy_in(c2b_ctx *ctx, void *d, const void *h, size_t bytes, cudaMemcpyKind kind) {
  cudaStream_t st = ctx->stream;
  if (bytes == 0) return C2B_OK;
  const int T = ctx->extra->tun.stage_threads;
  constexpr size_t CH = 2u << 20;  // pinning the ring itself costs ~1 ms per MB: keep it small
  bool pageable = false;
  if (kind == cudaMemcpyHostToDevice && T > 0 && bytes >= (64u << 10)) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, h) == cudaSuccess)
      pageable = at.type == cudaMemoryTypeUnregistered;
    else
      (void)cudaGetLastError();
  }
  if (!pageable) {
    C2B_CUDA(cudaMemcpyAsync(d, h, bytes, kind, st));
    return C2B_OK;
  }
  if (bytes < 4 * CH) {
    // a small pageable array (a camera range): one hop through the ring on this thread.  Left to the driver,
    // pageable copies issued for several GPUs at once queue behind one another — 12 ms for 1.5 MB per GPU at
    // N = 8 (profiles/r02k_bench_cfg4_8gpu.json: e2e_pageable)
    C2B_CUDA(cudaStreamSynchronize(st));  // the ring may still feed an earlier copy
    C2B_TRY(ctx->pin_in.ensure(std::max<size_t>(bytes, 8 * CH)));
    memcpy(ctx->pin_in.p, h, bytes);
    C2B_CUDA(cudaMemcpyAsync(d, ctx->pin_in.p, bytes, cudaMemcpyHostToDevice, st));
    return C2B_OK;
  }
  const size_t n_chunks = (bytes + CH - 1) / CH;
  const int nt = (int)std::min<size_t>((size_t)T, n_chunks);
  // the ring may still feed the previous call's DMA
  C2B_CUDA(cudaStreamSynchronize(st));
  C2B_TRY(ctx->pin_in.ensure(std::max<size_t>((size_t)nt * 2 * CH, 8 * CH)));
  std::vector<cudaError_t> err((size_t)nt, cudaSuccess);
  std::vector<std::thread> workers;
  const int device = ctx->device;
  char *ring = ctx->pin_in.as<char>();
  for (int t = 0; t < nt; ++t)
    workers.emplace_back([=, &err]() {
      cudaError_t e = cudaSetDevice(device);
      Event ev[2];  // destroyed on this thread, with `device` current
      for (int k = 0; k < 2 && e == cudaSuccess; ++k)
        if (ev[k].create(cudaEventDisableTiming) != C2B_OK) e = cudaGetLastError();
      size_t turn = 0;
      for (size_t c = (size_t)t; c < n_chunks && e == cudaSuccess; c += (size_t)nt, ++turn) {
        const int slot = (int)(turn & 1);
        char *pin = ring + ((size_t)t * 2 + slot) * CH;
        const size_t off = c * CH, n = std::min(CH, bytes - off);
        if (turn >= 2) e = cudaEventSynchronize(ev[slot]);  // the slot's previous DMA has drained
        if (e != cudaSuccess) break;
        memcpy(pin, static_cast<const char *>(h) + off, n);
        e = cudaMemcpyAsync(static_cast<char *>(d) + off, pin, n, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaEventRecord(ev[slot], st);
      }
      for (int k = 0; k < 2; ++k)
        if (ev[k] && e == cudaSuccess) e = cudaEventSynchronize(ev[k]);
      err[(size_t)t] = e;
    });
  for (auto &w : workers) w.join();
  for (cudaError_t e : err)
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      return set_error(C2B_ERR_CUDA, "staged host-to-device copy failed: %s", cudaGetErrorString(e));
    }
  return C2B_OK;
}

int c2b_internal_copy_in(c2b_ctx *ctx, void *d, const void *h, size_t bytes) {
  return copy_in(ctx, d, h, bytes, cudaMemcpyHostToDevice);
}

// The AoS point array of the ctx, with room for `capacity` points, for callers that fill it on the device
// themselves (an NCCL all-gather of per-GPU shards, c2b_multi.cu); followed by c2b_points_commit.
int c2b_points_device_buffer(c2b_ctx *ctx, uint64_t capacity, double **d_out) {
  if (!ctx || !d_out) return set_error(C2B_ERR_INVALID, "c2b_points_device_buffer: null argument");
  C2B_CUDA(cudaSetDevice(ctx->device));
  C2B_TRY(ctx->pts_aos.ensure(std::max<uint64_t>(capacity, 1) * 24));
  *d_out = ctx->pts_aos.as<double>();
  return C2B_OK;
}

// pts_aos[0, P) is (being) written on ctx->stream: derive the SoA copy and the coordinate bounds
int c2b_points_commit(c2b_ctx *ctx, uint64_t P) {
  if (!ctx) return set_error(C2B_ERR_INVALID, "c2b_points_commit: null ctx");
  if (P * 24 > ctx->pts_aos.cap) return set_error(C2B_ERR_INVALID, "c2b_points_commit: %llu points exceed the buffer", (unsigned long long)P);
  if (P >= 0xffffffffull) return set_error(C2B_ERR_INVALID, "too many points (%llu)", (unsigned long long)P);
  CtxExtra *x = ctx->extra.get();
  C2B_CUDA(cudaSetDevice(ctx->device));
  ctx->P = P;
  x->points_version++;
  x->grid.valid = false;
  x->have_points = true;
  x->have_result = false;
  x->host_call_last = false;
  if (P == 0) return C2B_OK;
  C2B_TRY(ctx->pts.ensure(P * 24));
  double *px = ctx->pts.as<double>(), *py = px + P, *pz = py + P;
  k_aos_to_soa3<<<blocks_for(P, 256), 256, 0, ctx->stream>>>(ctx->pts_aos.as<double>(), P, px, py, pz);
  C2B_KERNEL_CHECK();
  // coordinate bounds (grid extent); tiny D2H happens lazily when a grid is built
  int nb = (int)std::min<uint64_t>(blocks_for(P, 256), (uint64_t)4 * ctx->sm_count);
  C2B_TRY(ctx->misc.ensure((size_t)nb * 48 + 64));
  double *partial = ctx->misc.as<double>() + 8;
  k_pts_bounds_partial<<<nb, 256, 0, ctx->stream>>>(px, py, pz, P, partial);
  C2B_KERNEL_CHECK();
  k_pts_bounds_final<<<1, 32, 0, ctx->stream>>>(partial, nb, ctx->misc.as<double>());
  C2B_KERNEL_CHECK();
  C2B_CUDA(cudaMemcpyAsync(x->pts_bounds, ctx->misc.p, 48, cudaMemcpyDeviceToHost, ctx->stream));
  return C2B_OK;
}

static int upload_points_impl(c2b_ctx *ctx, const double *pts, uint64_t P, cudaMemcpyKind kind) {
  if (!ctx || (P && !pts)) return set_error(C2B_ERR_INVALID, "c2b_upload_points: null argument");
  if (P >= 0xffffffffull) return set_error(C2B_ERR_INVALID, "too many points (%llu)", (unsigned long long)P);
  double *d = nullptr;
  C2B_TRY(c2b_points_device_buffer(ctx, P, &d));
  if (P) C2B_TRY(copy_in(ctx, d, pts, P * 24, kind));
  return c2b_points_commit(ctx, P);
}

int c2b_upload_points(c2b_ctx *ctx, const double *pts, uint64_t P) {
  return upload_points_impl(ctx, pts, P, cudaMemcpyHostToDevice);
}

int c2b_upload_points_device(c2b_ctx *ctx, const double *d_pts, uint64_t P) {
  return upload_points_impl(ctx, d_pts, P, cudaMemcpyDeviceToDevice);
}

int c2b_drop_point_grid(c2b_ctx *ctx) {
  if (!ctx) return set_error(C2B_ERR_INVALID, "c2b_drop_point_grid: null ctx");
  ctx->extra->grid.valid = false;
  return C2B_OK;
}

int c2b_upload_cameras(c2b_ctx *ctx, const double *cams, uint64_t C) {
  if (!ctx || (C && !cams)) return set_error(C2B_ERR_INVALID, "c2b_upload_cameras: null argument");
  if (C >= 0xffffffffull) return set_error(C2B_ERR_INVALID, "too many cameras (%llu)", (unsigned long long)C);
  CtxExtra *x = ctx->extra.get();
  C2B_CUDA(cudaSetDevice(ctx->device));
  ctx->C = C;
  x->have_cameras = true;
  x->have_result = false;
  x->host_call_last = false;
  if (C == 0) return C2B_OK;
  C2B_TRY(ctx->cams.ensure(C * 120));
  C2B_TRY(ctx->cam_center.ensure(C * 24));
  C2B_TRY(copy_in(ctx, ctx->cams.p, cams, C * 120, cudaMemcpyHostToDevice));
  double *cx = ctx->cam_center.as<double>();
  k_cam_prep<<<blocks_for(C, 128), 128, 0, ctx->stream>>>(ctx->cams.as<double>(), C, cx, cx + C, cx + 2 * C);
  C2B_KERNEL_CHECK();
  return C2B_OK;
}

// cameras [first, first + count) of the call's device copy (ctx->cams_all) become the resident cameras:
// what c2b_upload_cameras does for a batch, without touching host memory again
static int select_cameras(c2b_ctx *ctx, uint64_t first, uint64_t count) {
  CtxExtra *x = ctx->extra.get();
  ctx->C = count;
  x->have_cameras = true;
  x->have_result = false;
  if (count == 0) return C2B_OK;
  C2B_TRY(ctx->cams.ensure(count * 120));
  C2B_TRY(ctx->cam_center.ensure(count * 24));
  C2B_CUDA(cudaMemcpyAsync(ctx->cams.p, ctx->cams_all.as<double>() + 15 * first, count * 120, cudaMemcpyDeviceToDevice,
                           ctx->stream));
  double *cx = ctx->cam_center.as<double>();
  k_cam_prep<<<blocks_for(count, 128), 128, 0, ctx->stream>>>(ctx->cams.as<double>(), count, cx, cx + count, cx + 2 * count);
  C2B_KERNEL_CHECK();
  return C2B_OK;
}

// ---- the pipeline ---------------------------------------------------------------------------------------
// the 128-byte counter block -> host, synchronising the compute stream
static int read_counters(c2b_ctx *ctx, unsigned long long *h_cnt) {
  C2B_TRY(ctx->h_small.ensure(256));
  k_copy_words<<<1, 32, 0, ctx->stream>>>(ctx->counters.as<uint32_t>(), ctx->h_small.as<uint32_t>(), 32);
  C2B_KERNEL_CHECK();
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));
  memcpy(h_cnt, ctx->h_small.p, 128);
  return C2B_OK;
}

// bounding box of the resident cameras' centres (tiny two-stage reduction; synchronises the stream)
static int camera_bbox(c2b_ctx *ctx, double lo[3], double hi[3]) {
  const uint64_t C = ctx->C;
  const double *cx = ctx->cam_center.as<double>();
  int nb = (int)std::min<uint64_t>(std::max<uint64_t>(blocks_for(C, 256), 1), (uint64_t)ctx->sm_count);
  C2B_TRY(ctx->misc.ensure((size_t)nb * 48 + 64));
  double *partial = ctx->misc.as<double>() + 8;
  k_pts_bounds_partial<<<nb, 256, 0, ctx->stream>>>(cx, cx + C, cx + 2 * C, C, partial);
  C2B_KERNEL_CHECK();
  k_pts_bounds_final<<<1, 32, 0, ctx->stream>>>(partial, nb, ctx->misc.as<double>());
  C2B_KERNEL_CHECK();
  double b[6];
  C2B_CUDA(cudaMemcpyAsync(b, ctx->misc.p, 48, cudaMemcpyDeviceToHost, ctx->stream));
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int k = 0; k < 3; ++k) {
    lo[k] = b[k];
    hi[k] = b[3 + k];
  }
  return C2B_OK;
}

// what the cameras can reach: their centres' box grown by max_dist (and a little)
static void reach_box(const double clo[3], const double chi[3], double max_dist, double lo[3], double hi[3]) {
  for (int k = 0; k < 3; ++k) {
    const double pad = max_dist + 1e-6 * (std::fabs(max_dist) + std::fabs(clo[k]) + std::fabs(chi[k]));
    lo[k] = clo[k] - pad;
    hi[k] = chi[k] + pad;
  }
}

static int build_grid(c2b_ctx *ctx, CtxExtra *x, double max_dist) {
  cudaStream_t st = ctx->stream;
  const uint64_t P = ctx->P;
  C2B_CUDA(cudaStreamSynchronize(st));  // pts_bounds has landed
  GridDesc g;
  double h = max_dist * x->tun.grid_cell_factor;
  double ext[3];
  for (int k = 0; k < 3; ++k) {
    g.min_c[k] = x->pts_bounds[k];
    g.max_c[k] = x->pts_bounds[3 + k];
    ext[k] = g.max_c[k] - g.min_c[k];
    if (!(ext[k] >= 0.0) || std::isinf(ext[k])) ext[k] = 0.0;  // NaN / inf coordinates: one cell
    g.lo[k] = std::isfinite(g.min_c[k]) ? g.min_c[k] : 0.0;
  }
  if (!(h > 0.0) || !std::isfinite(h)) h = 1.0;
  const double max_cells = 4194304.0;  // 2^22
  auto cells_at = [&](double hh) {
    double total = 1.0;
    for (int k = 0; k < 3; ++k) total *= std::min(std::floor(ext[k] / hh) + 1.0, 1e9);
    return total;
  };
  x->grid.hinted = false;
  g.drop = 0;
  for (int k = 0; k < 3; ++k) g.rlo[k] = g.rhi[k] = 0.0;
  bool odd_bounds = false;  // an infinite coordinate would collapse its axis to one cell
  for (int k = 0; k < 3; ++k) odd_bounds = odd_bounds || !std::isfinite(g.min_c[k]) || !std::isfinite(g.max_c[k]);
  if (ctx->C) {
    // No point farther than max_dist from every camera can be observed, so only the cameras' REACH (their
    // centres' box grown by max_dist) has to be binned.  When the reach is clearly smaller than the data —
    // a camera shard of a multi-GPU run, or a few far-away outlier vertices of an OBJ scene that would stretch
    // every cell — the cells cover the reach only and points outside it are left out of the grid altogether
    // (k_grid_count); a GPU that owns 1/8 of the cameras then bins about 1/8 of the points.
    double clo[3], chi[3], rlo[3], rhi[3];
    C2B_TRY(camera_bbox(ctx, clo, chi));
    reach_box(clo, chi, max_dist, rlo, rhi);
    bool usable = true;
    for (int k = 0; k < 3; ++k) usable = usable && std::isfinite(rlo[k]) && std::isfinite(rhi[k]) && rlo[k] <= rhi[k];
    double frac = 1.0;  // share of the data's box the reach covers
    if (usable)
      for (int k = 0; k < 3; ++k) {
        const double a = std::fmax(g.min_c[k], rlo[k]), b = std::fmin(g.max_c[k], rhi[k]);
        if (ext[k] > 0.0) frac *= a <= b ? std::fmin((b - a) / ext[k], 1.0) : 0.0;
      }
    if (usable && (cells_at(h) > max_cells || odd_bounds || frac < 0.7)) {
      for (int k = 0; k < 3; ++k) {
        // the reach intersected with the data bounds (which may be infinite); empty: one cell at the reach's edge
        const double a = std::fmax(g.min_c[k], rlo[k]), b = std::fmin(g.max_c[k], rhi[k]);
        g.lo[k] = a <= b ? a : rlo[k];
        ext[k] = a <= b ? b - a : 0.0;
        g.min_c[k] = g.lo[k];  // what is IN the grid: rows of edge cells end here (camera_row)
        g.max_c[k] = a <= b ? b : g.lo[k];
        g.rlo[k] = rlo[k];
        g.rhi[k] = rhi[k];
        x->grid.hint_lo[k] = rlo[k];
        x->grid.hint_hi[k] = rhi[k];
      }
      g.drop = 1;
      x->grid.hinted = true;
    }
  }
  for (;;) {
    double total = 1.0;
    for (int k = 0; k < 3; ++k) {
      double nk = std::floor(ext[k] / h) + 1.0;
      if (nk > 1e9) nk = 1e9;
      g.n[k] = (int)nk;
      total *= nk;
    }
    if (total <= max_cells) break;
    h *= 1.5;
  }
  g.inv_h = 1.0 / h;
  uint64_t n_cells = (uint64_t)g.n[0] * g.n[1] * g.n[2];
  C2B_TRY(ctx->cell_of_pt.ensure(P * 4));
  C2B_TRY(ctx->cell_start.ensure((n_cells + 1) * 4));
  C2B_TRY(ctx->cell_cursor.ensure((n_cells + 1) * 4));
  C2B_TRY(ctx->grid_x.ensure(P * 8));
  C2B_TRY(ctx->grid_y.ensure(P * 8));
  C2B_TRY(ctx->grid_z.ensure(P * 8));
  C2B_TRY(ctx->grid_idx.ensure(P * 4));
  C2B_CUDA(cudaMemsetAsync(ctx->cell_start.p, 0, (n_cells + 1) * 4, st));
  const double *px = ctx->pts.as<double>(), *py = px + P, *pz = py + P;
  k_grid_count<<<blocks_for(P, 256), 256, 0, st>>>(px, py, pz, P, g, ctx->cell_of_pt.as<uint32_t>(),
                                                   ctx->cell_start.as<uint32_t>());
  C2B_KERNEL_CHECK();
  C2B_TRY(exclusive_scan_u32(st, ctx->cell_start.as<uint32_t>(), ctx->cell_start.as<uint32_t>(),
                             n_cells + 1, nullptr, ctx->scan_tmp));
  C2B_CUDA(cudaMemcpyAsync(ctx->cell_cursor.p, ctx->cell_start.p, (n_cells + 1) * 4, cudaMemcpyDeviceToDevice, st));
  k_grid_fill<<<blocks_for(P, 256), 256, 0, st>>>(
      px, py, pz, P, ctx->cell_of_pt.as<uint32_t>(), ctx->cell_cursor.as<uint32_t>(), ctx->grid_x.as<double>(),
      ctx->grid_y.as<double>(), ctx->grid_z.as<double>(), ctx->grid_idx.as<uint32_t>());
  C2B_KERNEL_CHECK();
  x->grid.valid = true;
  x->grid.max_dist = max_dist;
  x->grid.points_version = x->points_version;
  x->grid.desc = g;
  x->grid.n_cells = n_cells;
  return C2B_OK;
}

// the point grid for the resident cameras: the cached one if it still serves them, else a new one
static int ensure_grid(c2b_ctx *ctx, CtxExtra *x, double max_dist) {
  if (!(ctx->C && ctx->P)) return C2B_OK;
  bool valid = x->grid.valid && x->grid.max_dist == max_dist && x->grid.points_version == x->points_version;
  // built for some cameras' reach: still good if the current ones stay inside it (a host-buffer call builds it
  // once for ALL its cameras and locks it for the call's batches)
  if (valid && x->grid.hinted && !x->grid_locked) {
    double clo[3], chi[3], rlo[3], rhi[3];
    C2B_TRY(camera_bbox(ctx, clo, chi));
    reach_box(clo, chi, max_dist, rlo, rhi);
    for (int k = 0; k < 3; ++k) valid = valid && rlo[k] >= x->grid.hint_lo[k] && rhi[k] <= x->grid.hint_hi[k];
  }
  if (!valid) C2B_TRY(build_grid(ctx, x, max_dist));
  return C2B_OK;
}

namespace {

void fill_stats(c2b_ctx *ctx, c2b_obs *stats, uint64_t C, uint64_t n_cand, uint64_t pairs_eval,
                uint64_t nodes, uint64_t tris) {
  if (!stats) return;
  memset(stats, 0, sizeof *stats);
  stats->n_cameras = C;
  stats->n_obs = ctx->out_O;
  stats->n_candidates = n_cand;
  stats->pairs_evaluated = pairs_eval;
  stats->nodes_visited = nodes;
  stats->tris_tested = tris;
  auto ms = [&](int a, int b) {
    float t = 0;
    cudaEventElapsedTime(&t, ctx->ev[a], ctx->ev[b]);
    return t;
  };
  stats->ms_prep = ms(EV_H2D, EV_PREP);
  stats->ms_cull = ms(EV_PREP, EV_CULL);
  stats->ms_sort = ms(EV_CULL, EV_SORT);
  stats->ms_traverse = ms(EV_SORT, EV_TRAVERSE);
  stats->ms_compact = ms(EV_TRAVERSE, EV_COMPACT);
  stats->ms_total = ms(EV_START, EV_D2H);
}

// ---- grid schedule: plan -> fused cull + occlusion -> per-camera sort + write (c2b_fused.cuh) ------
// Stage timers: ms_cull = plan + scan (+ per-camera leaf lists), ms_traverse = the fused kernel,
// ms_compact = visible-count scan + sort/write; ms_sort stays 0 (there is no global sort).
int visibility_grid_fused(c2b_ctx *ctx, CtxExtra *x, const c2b_scene *scene, double max_dist,
                          const c2b_vis_options &opt, int pbits, int cbits, c2b_obs *stats) {
  cudaStream_t st = ctx->stream;
  const uint64_t C = ctx->C, P = ctx->P;
  const int sel = ctx->out_sel;
  C2B_TRY(ensure_grid(ctx, x, max_dist));
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_PREP], st));

  C2B_TRY(ctx->counters.ensure(128));
  C2B_TRY(ctx->out_offsets[sel].ensure((C + 1) * 8));
  C2B_CUDA(cudaMemsetAsync(ctx->counters.p, 0, 128, st));
  uint64_t n_cand = 0, pairs_eval = 0, total_obs = 0, nodes = 0, tris_t = 0;
  if (!(C && P)) {
    C2B_CUDA(cudaMemsetAsync(ctx->out_offsets[sel].p, 0, (C + 1) * 8, st));
    for (int e : {EV_CULL, EV_SORT, EV_TRAVERSE, EV_COMPACT, EV_D2H}) C2B_CUDA(cudaEventRecord(ctx->ev[e], st));
    C2B_CUDA(cudaStreamSynchronize(st));
    ctx->out_C = C;
    ctx->out_O = 0;
    x->have_result = true;
    x->res_candidates = 0;
    fill_stats(ctx, stats, C, 0, 0, 0, 0);
    return C2B_OK;
  }

  // Tickets per camera: with fewer cameras than persistent warps a camera's rows are split over 2 or 4
  // tickets (a ticket repeats the per-camera set-up, so it only pays on warps that would otherwise idle).
  int parts_log2 = 0;
  {
    const uint64_t warps = (uint64_t)ctx->sm_count * FU_RESIDENT_WARPS;
    if (2 * C <= warps) parts_log2 = 1;
    if (4 * C <= warps) parts_log2 = 2;
    if (x->tun.parts_log2 >= 0) parts_log2 = x->tun.parts_log2;  // test hook
  }
  const uint64_t slots = C << parts_log2;
  C2B_TRY(ctx->ev_off.ensure((slots + 1) * 4));
  C2B_TRY(ctx->vis_count.ensure((slots + 1) * 4));
  C2B_TRY(ctx->seg_off.ensure((slots + 1) * 4));
  const double *cxp = ctx->cam_center.as<double>();
  const bool mesh = opt.occlusion == C2B_OCC_MESH && scene && scene->n_nodes > 0;
  FusedArgs fa;
  memset(&fa, 0, sizeof fa);
  fa.cams = ctx->cams.as<double>();
  fa.cen_x = cxp;
  fa.cen_y = cxp + C;
  fa.cen_z = cxp + 2 * C;
  fa.C = C;
  fa.gx = ctx->grid_x.as<double>();
  fa.gy = ctx->grid_y.as<double>();
  fa.gz = ctx->grid_z.as<double>();
  fa.gidx = ctx->grid_idx.as<uint32_t>();
  fa.cell_start = ctx->cell_start.as<uint32_t>();
  fa.g = x->grid.desc;
  fa.max_dist = max_dist;
  fa.t_star = exact_sq_threshold(max_dist);
  fa.scene_absmax = scene_abs_max(scene);
  fa.endpoint_guard_rel = opt.endpoint_guard_rel;
  fa.block_length = opt.block_length;
  fa.block_inset = opt.block_inset;
  fa.parts_log2 = parts_log2;
  C2B_TRY(ctx->plan_rows.ensure(C * FU_ROWS * sizeof(uint2)));
  C2B_TRY(ctx->plan_row_count.ensure(C * 4));
  fa.rows = ctx->plan_rows.as<uint2>();
  fa.row_count = ctx->plan_row_count.as<uint32_t>();
  fa.ev_count = ctx->ev_off.as<uint32_t>();
  fa.vis_count = ctx->vis_count.as<uint32_t>();
  fa.counters = ctx->counters.as<unsigned long long>();

  uint32_t *d_total = ctx->counters.as<uint32_t>() + 12;  // bytes 48..51 of the counter block
  uint32_t *d_max = ctx->counters.as<uint32_t>() + 13;    // bytes 52..55
  unsigned long long h_cnt[16];

  // Per-camera leaf lists (cameras + BVH only) and the plan (cameras + point grid only) are independent and
  // each too small to fill the GPU (one thread or warp per camera, latency-bound): the lists run on a
  // second stream beside the plan and its scan, and the main stream joins before the counters are read.
  cudaStream_t ax = ctx->aux_stream;
  if (mesh) {
    const uint32_t trilist_cap = (uint32_t)x->tun.trilist_cap;
    C2B_TRY(ctx->tri_list.ensure((size_t)C * trilist_cap * 4));
    C2B_TRY(ctx->tri_count.ensure(C * 4));
    float rmax = (float)max_dist;
    if ((double)rmax < max_dist) rmax = std::nextafter(rmax, INFINITY);
    rmax = rmax * (1.0f + 4e-6f);
    fa.nodes = scene->nodes.as<float4>();
    fa.tris = scene->tris.as<float4>();
    fa.n_nodes = (int)scene->n_nodes;
    fa.tri_list = ctx->tri_list.as<uint32_t>();
    fa.tri_count = ctx->tri_count.as<uint32_t>();
    fa.tri_cap = trilist_cap;
    fa.hoist_max = (uint32_t)std::min(x->tun.hoist_max, FU_HOIST);
    fa.packet_bvh = x->tun.packet_bvh;
    const bool tl_warp = x->tun.trilist_warp >= 0 ? x->tun.trilist_warp != 0 : C < 32768;
    C2B_CUDA(cudaEventRecord(ctx->ev_fork, st));  // after the counter reset and the camera upload
    C2B_CUDA(cudaStreamWaitEvent(ax, ctx->ev_fork, 0));
    if (tl_warp)
      k_cam_trilist_warp<<<blocks_for(C, TL_WARPS), TL_WARPS * 32, 0, ax>>>(
          fa.nodes, fa.n_nodes, fa.cen_x, fa.cen_y, fa.cen_z, C, rmax, fa.scene_absmax, trilist_cap,
          ctx->tri_list.as<uint32_t>(), ctx->tri_count.as<uint32_t>(), fa.counters + 0);
    else
      k_cam_trilist<<<blocks_for(C, 128), 128, 0, ax>>>(fa.nodes, fa.n_nodes, fa.cen_x, fa.cen_y, fa.cen_z, C, rmax,
                                                       fa.scene_absmax, trilist_cap, ctx->tri_list.as<uint32_t>(),
                                                       ctx->tri_count.as<uint32_t>(), fa.counters + 0);
    C2B_KERNEL_CHECK();
    C2B_CUDA(cudaEventRecord(ctx->ev_join, ax));
  }
  // plan: row points per camera -> scratch slices
  k_cam_plan<<<blocks_for(C + 1, 128), 128, 0, st>>>(fa);
  C2B_KERNEL_CHECK();
  C2B_TRY(exclusive_scan_u32(st, fa.ev_count, fa.ev_count, slots + 1, nullptr, ctx->scan_tmp));
  if (mesh) C2B_CUDA(cudaStreamWaitEvent(st, ctx->ev_join, 0));
  // Sizes of the scratch / output arrays and the kernel variant depend on the plan's totals.  The first pass
  // waits for them; later passes go by what the previous pass left (grow-only buffers, the remembered variant),
  // launch everything back to back, and check at the one final sync that it all fitted.
  const uint64_t max_pairs = x->tun.max_pairs;  // 32-bit scratch offsets (lower: test hook)
  const bool mt = mesh && opt.predicate == C2B_PRED_MT;
  const bool optimistic = x->tun.optimistic && x->memo.valid && !opt.count_traversal && ctx->scratch_idx.cap >= 4 &&
                          ctx->out_idx[sel].cap >= 4 && ctx->out_uv[sel].cap >= 16;
  bool any_overflow = x->memo.any_overflow;
  if (!optimistic) {
    C2B_TRY(read_counters(ctx, h_cnt));
    pairs_eval = h_cnt[1];
    any_overflow = h_cnt[0] != 0;  // cameras whose leaf list exceeded the cap
    if (pairs_eval >= max_pairs)
      return set_error(ERR_TOO_LARGE, "more than 2^32 camera-point pairs inside max_dist in one call; shard the cameras");
    C2B_TRY(ctx->scratch_idx.ensure(std::max<uint64_t>(pairs_eval, 1) * 4));
  }
  fa.scratch_idx = ctx->scratch_idx.as<uint32_t>();
  fa.scratch_cap = ctx->scratch_idx.cap / 4;
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_CULL], st));
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_SORT], st));

  // fused cull + occlusion
  C2B_CUDA(cudaMemsetAsync(ctx->vis_count.p, 0, (slots + 1) * 4, st));
  {
    // persistent warps draw cameras from a ticket; more CTAs than can be resident is harmless
    const unsigned nb = (unsigned)std::min<uint64_t>(blocks_for(slots, FU_WARPS), (uint64_t)ctx->sm_count * 8), nt = FU_WARPS * 32;
    const bool cnt = opt.count_traversal != 0;
    // The template's third argument counts CTAs of EIGHT warps per SM (fu_min_ctas translates for four-warp CTAs).
    // Eight-warp CTAs, r01m kernels at cfg4: 4 CTAs/SM at 64 registers 2.68 ms; 3 at 80 2.69 ms; 5 at 48 2.74 ms.
    // Four-warp CTAs, r02y kernels: 7 CTAs/SM at 72 registers 2.31 ms against 2.38 ms for 4 x 8 warps at 64.
    if (mt) {
      // candidates only; k_filter_candidates_mt decides occlusion below
      k_visibility_fused<FU_OCC_NONE, false, 3, false><<<nb, nt, 0, st>>>(fa);
    } else if (mesh) {
      if (cnt)
        k_visibility_fused<FU_OCC_MESH, true, 3, true><<<nb, nt, 0, st>>>(fa);
      else if (any_overflow)
        k_visibility_fused<FU_OCC_MESH, false, 4, true><<<nb, nt, 0, st>>>(fa);
      else
        k_visibility_fused<FU_OCC_MESH, false, 4, false><<<nb, nt, 0, st>>>(fa);
    } else if (opt.occlusion == C2B_OCC_ANALYTIC) {
      k_visibility_fused<FU_OCC_ANALYTIC, false, 2, false><<<nb, nt, 0, st>>>(fa);
    } else {
      k_visibility_fused<FU_OCC_NONE, false, 3, false><<<nb, nt, 0, st>>>(fa);
    }
    C2B_KERNEL_CHECK();
    if (mt) {
      FilterArgs f{fa.nodes, fa.tris, fa.n_nodes, fa.scene_absmax, fa.cen_x, fa.cen_y, fa.cen_z, ctx->pts_aos.as<double>(),
                   slots, parts_log2, opt.endpoint_guard_rel, fa.ev_count, fa.scratch_idx, fa.vis_count, fa.counters};
      k_filter_candidates_mt<<<blocks_for(slots, 8), 256, 0, st>>>(f);
      C2B_KERNEL_CHECK();
    }
  }
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_TRAVERSE], st));

  // visible counts -> CSR offsets
  C2B_TRY(exclusive_scan_u32(st, fa.vis_count, ctx->seg_off.as<uint32_t>(), slots + 1, d_total, ctx->scan_tmp));
  k_max_cam<<<(unsigned)std::min<uint64_t>(blocks_for(C, 256), 1024), 256, 0, st>>>(ctx->seg_off.as<uint32_t>(), C, parts_log2, d_max);
  C2B_KERNEL_CHECK();
  uint32_t total32 = 0, max32 = 0;
  auto read_totals = [&]() -> int {
    C2B_TRY(read_counters(ctx, h_cnt));
    if (h_cnt[5]) return set_error(C2B_ERR_CUDA, "internal: a camera's scratch slice overflowed");
    memcpy(&total32, reinterpret_cast<const char *>(h_cnt) + 48, 4);
    memcpy(&max32, reinterpret_cast<const char *>(h_cnt) + 52, 4);
    total_obs = total32;
    n_cand = h_cnt[4];
    nodes = h_cnt[2];
    tris_t = h_cnt[3];
    return C2B_OK;
  };
  auto sort_write_args = [&]() {
    return SortWriteArgs{fa.ev_count, ctx->seg_off.as<uint32_t>(), C, fa.scratch_idx, fa.cams, ctx->pts_aos.as<double>(),
                         ctx->out_offsets[sel].as<uint64_t>(), ctx->out_idx[sel].as<uint32_t>(), ctx->out_uv[sel].as<double2>(),
                         std::max(pbits, 1), parts_log2,
                         std::min<uint64_t>(ctx->out_idx[sel].cap / 4, ctx->out_uv[sel].cap / 16), fa.counters + 12};
  };
  const unsigned swb = (unsigned)blocks_for(C, SW_WARPS), swt = SW_WARPS * 32;
  if (optimistic) {
    // sort + write straight away into the arrays as they are; the one sync of the pass comes after it
    const SortWriteArgs sw = sort_write_args();
    if (parts_log2 > 0)
      k_sort_write<6, true><<<swb, swt, 0, st>>>(sw);
    else
      k_sort_write<8, false><<<swb, swt, 0, st>>>(sw);
    C2B_KERNEL_CHECK();
    if (x->memo.big) {
      k_sort_write_block<<<(unsigned)C, 256, 0, st>>>(sw);
      C2B_KERNEL_CHECK();
    }
    C2B_TRY(read_totals());
    pairs_eval = h_cnt[1];
    const bool fits = h_cnt[12] == 0 && pairs_eval <= fa.scratch_cap && pairs_eval < max_pairs &&
                      (max32 <= SW_WARP_MAX || (x->memo.big && max32 <= SW_BLOCK_MAX));
    if (!fits) {
      // this pass is larger than what the previous one left behind: size everything exactly and repeat it
      x->memo.valid = false;
      if (pairs_eval >= max_pairs)
        return set_error(ERR_TOO_LARGE, "more than 2^32 camera-point pairs inside max_dist in one call; shard the cameras");
      return visibility_grid_fused(ctx, x, scene, max_dist, opt, pbits, cbits, stats);
    }
    x->memo.any_overflow = h_cnt[0] != 0;
    x->memo.big = max32 > SW_WARP_MAX;
  } else {
    C2B_TRY(read_totals());
    x->memo.valid = true;
    x->memo.any_overflow = any_overflow;
    x->memo.big = max32 > SW_WARP_MAX;
    if (total_obs) {
      C2B_TRY(ctx->out_idx[sel].ensure(total_obs * 4));
      C2B_TRY(ctx->out_uv[sel].ensure(total_obs * 16));
      const SortWriteArgs sw = sort_write_args();
      if (max32 <= SW_BLOCK_MAX) {
        // registers capped for 8 CTAs/SM (measured at cfg4: 0.81 ms; 6 CTAs/SM 0.91 ms, 4 CTAs/SM 1.12 ms)
        if (parts_log2 > 0)
          k_sort_write<6, true><<<swb, swt, 0, st>>>(sw);
        else
          k_sort_write<8, false><<<swb, swt, 0, st>>>(sw);
        C2B_KERNEL_CHECK();
        if (max32 > SW_WARP_MAX) {
          k_sort_write_block<<<(unsigned)C, 256, 0, st>>>(sw);
          C2B_KERNEL_CHECK();
        }
      } else {
        // a camera sees more points than the shared-memory sort holds: radix-sort all visible keys
        C2B_TRY(ctx->sort_keys[0].ensure(total_obs * 8));
        C2B_TRY(ctx->sort_keys[1].ensure(total_obs * 8));
        C2B_TRY(ctx->sort_vals[0].ensure(total_obs * 4));
        C2B_TRY(ctx->sort_vals[1].ensure(total_obs * 4));
        k_expand_keys<<<blocks_for(C, 8), 256, 0, st>>>(sw, pbits, ctx->sort_keys[0].as<uint64_t>());
        C2B_KERNEL_CHECK();
        uint64_t *keys[2] = {ctx->sort_keys[0].as<uint64_t>(), ctx->sort_keys[1].as<uint64_t>()};
        uint32_t *vals[2] = {ctx->sort_vals[0].as<uint32_t>(), ctx->sort_vals[1].as<uint32_t>()};
        int res = 0;
        C2B_TRY(radix_sort_pairs(st, keys, vals, total_obs, pbits + cbits, ctx->sort_hist, ctx->scan_tmp, &res));
        k_write_sorted<<<blocks_for(total_obs, 256), 256, 0, st>>>(
            keys[res], total_obs, pbits, fa.cams, ctx->pts_aos.as<double>(), ctx->out_idx[sel].as<uint32_t>(),
            ctx->out_uv[sel].as<double2>());
        C2B_KERNEL_CHECK();
        k_widen_cam_offsets<<<blocks_for(C + 1, 256), 256, 0, st>>>(ctx->seg_off.as<uint32_t>(), C + 1, parts_log2,
                                                                   ctx->out_offsets[sel].as<uint64_t>());
        C2B_KERNEL_CHECK();
      }
    } else {
      C2B_CUDA(cudaMemsetAsync(ctx->out_offsets[sel].p, 0, (C + 1) * 8, st));
    }
  }
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_COMPACT], st));
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_D2H], st));
  C2B_CUDA(cudaStreamSynchronize(st));
  ctx->out_C = C;
  ctx->out_O = total_obs;
  x->have_result = true;
  x->res_candidates = n_cand;
  fill_stats(ctx, stats, C, n_cand, pairs_eval, nodes, tris_t);
  return C2B_OK;
}

}  // namespace

static int visibility_resident_impl(c2b_ctx *ctx, const c2b_scene *scene, double max_dist,
                                    const c2b_vis_options *opt_in, c2b_obs *stats);

int c2b_visibility_graph_resident(c2b_ctx *ctx, const c2b_scene *scene, double max_dist,
                                  const c2b_vis_options *opt_in, c2b_obs *stats) {
  const int rc = visibility_resident_impl(ctx, scene, max_dist, opt_in, stats);
  if (ctx) ctx->extra->host_call_last = false;
  return rc == ERR_TOO_LARGE ? C2B_ERR_INVALID : rc;
}

static int visibility_resident_impl(c2b_ctx *ctx, const c2b_scene *scene, double max_dist,
                                    const c2b_vis_options *opt_in, c2b_obs *stats) {
  if (!ctx) return set_error(C2B_ERR_INVALID, "c2b_visibility_graph_resident: null ctx");
  CtxExtra *x = ctx->extra.get();
  if (!x->have_points || !x->have_cameras)
    return set_error(C2B_ERR_INVALID, "upload cameras and points first");
  c2b_vis_options opt;
  if (opt_in)
    opt = *opt_in;
  else
    c2b_vis_options_default(&opt);
  if (opt.occlusion == C2B_OCC_MESH && !scene)
    return set_error(C2B_ERR_INVALID, "C2B_OCC_MESH needs a scene");
  if (opt.cull_mode != C2B_CULL_GRID && opt.cull_mode != C2B_CULL_EXHAUSTIVE)
    return set_error(C2B_ERR_INVALID, "unknown cull_mode %d", opt.cull_mode);
  if (opt.occlusion < C2B_OCC_MESH || opt.occlusion > C2B_OCC_ANALYTIC)
    return set_error(C2B_ERR_INVALID, "unknown occlusion %d", opt.occlusion);
  if (opt.predicate != C2B_PRED_WATERTIGHT && opt.predicate != C2B_PRED_MT)
    return set_error(C2B_ERR_INVALID, "unknown predicate %d", opt.predicate);
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const uint64_t C = ctx->C, P = ctx->P;
  x->have_result = false;

  C2B_CUDA(cudaEventRecord(ctx->ev[EV_START], st));
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_H2D], st));

  const int pbits = std::max(1, bit_length(P ? P - 1 : 0));
  const int cbits = std::max(1, bit_length(C ? C - 1 : 0));
  if (pbits + cbits > 63) return set_error(C2B_ERR_INVALID, "camera x point index space exceeds 63 bits");
  if (opt.cull_mode == C2B_CULL_GRID) return visibility_grid_fused(ctx, x, scene, max_dist, opt, pbits, cbits, stats);

  // ---- exhaustive schedule: every pair -> pool -> radix sort -> ordered traversal -> stream compaction --
  C2B_TRY(ctx->counters.ensure(128));
  C2B_TRY(ctx->cam_count.ensure((C + 1) * 4));
  C2B_TRY(ctx->out_offsets[ctx->out_sel].ensure((C + 1) * 8));
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_PREP], st));

  uint64_t n_cand = 0, pairs_eval = 0, pool_n = 0;
  if (C && P) {
    CullArgs a;
    a.cams = ctx->cams.as<double>();
    a.cen_x = ctx->cam_center.as<double>();
    a.cen_y = a.cen_x + C;
    a.cen_z = a.cen_y + C;
    a.C = C;
    a.P = P;
    a.t_star = exact_sq_threshold(max_dist);
    a.t_cons = a.t_star * (1.0 + 4e-15);
    if (a.t_star > 0.0 && a.t_cons == a.t_star) a.t_cons = std::nextafter(a.t_star, INFINITY);
    a.pbits = pbits;
    a.cam_count = ctx->cam_count.as<uint32_t>();
    a.counters = ctx->counters.as<unsigned long long>();
    a.px = ctx->pts.as<double>();
    a.py = a.px + P;
    a.pz = a.py + P;
    if (ctx->pool_capacity == 0) {
      long double pairs = (long double)C * (long double)P;
      uint64_t guess = std::max<uint64_t>(1u << 20, 96 * C);
      if ((long double)guess > pairs) guess = (uint64_t)pairs;
      ctx->pool_capacity = std::max<uint64_t>(guess, 1024);
    }
    for (int attempt = 0;; ++attempt) {
      // the pool's key array doubles as buffer 0 of the radix sort
      C2B_TRY(ctx->sort_keys[0].ensure(ctx->pool_capacity * 8));
      C2B_TRY(ctx->pool_uv.ensure(ctx->pool_capacity * 16));
      a.pool_key = ctx->sort_keys[0].as<uint64_t>();
      a.pool_uv = ctx->pool_uv.as<double2>();
      a.pool_capacity = ctx->pool_capacity;
      C2B_CUDA(cudaMemsetAsync(ctx->counters.p, 0, 64, st));
      C2B_CUDA(cudaMemsetAsync(ctx->cam_count.p, 0, (C + 1) * 4, st));
      dim3 grid(blocks_for(P, CB_THREADS * CB_PPT), blocks_for(C, CB_TC));
      if (grid.y > 65535u) return set_error(C2B_ERR_INVALID, "too many cameras for one exhaustive launch");
      k_cull_exhaustive<<<grid, CB_THREADS, 0, st>>>(a);
      C2B_KERNEL_CHECK();
      unsigned long long h_cnt[16];
      C2B_TRY(read_counters(ctx, h_cnt));
      pool_n = h_cnt[0];
      n_cand = h_cnt[0];
      pairs_eval = C * P;
      if (pool_n <= ctx->pool_capacity) break;
      if (attempt >= 2) return set_error(C2B_ERR_CUDA, "candidate pool overflow persisted");
      ctx->pool_capacity = pool_n + pool_n / 16 + 1024;  // exact count is known now: re-run once
    }
    if (pool_n >= 0xffffffffull)
      return set_error(ERR_TOO_LARGE, "more than 2^32 candidates in one call; shard the cameras");
  } else {
    C2B_CUDA(cudaMemsetAsync(ctx->counters.p, 0, 64, st));
    C2B_CUDA(cudaMemsetAsync(ctx->cam_count.p, 0, (C + 1) * 4, st));
  }
  C2B_CUDA(cudaEventRecord(ctx->ev[EV_CULL], st));

  const double *cxp = ctx->cam_center.as<double>();
  const double *pxp = ctx->pts.as<double>();
  const float scene_absmax = scene_abs_max(scene);

  // occlusion of `n` sorted candidate keys -> one ballot word per 32 keys
  auto run_occlusion = [&](const uint64_t *keys_in, uint64_t n, uint64_t n_words) -> int {
    if (!n) return C2B_OK;
    if (opt.occlusion == C2B_OCC_MESH && scene->n_nodes > 0) {
      TraverseArgs t;
      t.nodes = scene->nodes.as<float4>();
      t.tris = scene->tris.as<float4>();
      t.n_nodes = (int)scene->n_nodes;
      t.keys = keys_in;
      t.n_cand = n;
      t.scene_absmax = scene_absmax;
      t.pbits = pbits;
      t.cen_x = cxp;
      t.cen_y = cxp + C;
      t.cen_z = cxp + 2 * C;
      t.p_aos = ctx->pts_aos.as<double>();
      t.endpoint_guard_rel = opt.endpoint_guard_rel;
      t.vis_words = ctx->vis_words.as<uint32_t>();
      t.counters = ctx->counters.as<unsigned long long>();
      if (opt.predicate == C2B_PRED_MT)
        k_traverse<false, true><<<blocks_for(n_words, 8), 256, 0, st>>>(t);
      else if (opt.count_traversal)
        k_traverse<true><<<blocks_for(n_words, 8), 256, 0, st>>>(t);
      else
        k_traverse<false><<<blocks_for(n_words, 8), 256, 0, st>>>(t);
    } else if (opt.occlusion == C2B_OCC_ANALYTIC) {
      k_analytic_occlusion<<<blocks_for(n_words * 32, 256), 256, 0, st>>>(
          keys_in, n, pbits, cxp, cxp + C, cxp + 2 * C, pxp, pxp + P, pxp + 2 * P, opt.block_length,
          opt.block_inset, ctx->vis_words.as<uint32_t>());
    } else {
      k_words_all_visible<<<blocks_for(n_words * 32, 256), 256, 0, st>>>(keys_in, ctx->vis_words.as<uint32_t>(), n);
    }
    C2B_KERNEL_CHECK();
    return C2B_OK;
  };

  uint32_t *d_total = ctx->counters.as<uint32_t>() + 12;  // bytes 48..51 of the counter block
  uint64_t total_obs = 0;
  unsigned long long h_fin[16] = {0};
  {
    C2B_TRY(exclusive_scan_u32(st, ctx->cam_count.as<uint32_t>(), ctx->cam_count.as<uint32_t>(), C + 1,
                               nullptr, ctx->scan_tmp));
    int res = 0;
    uint64_t *keys[2] = {nullptr, nullptr};
    uint32_t *vals[2] = {nullptr, nullptr};
    if (n_cand) {
      C2B_TRY(ctx->sort_keys[1].ensure(n_cand * 8));
      C2B_TRY(ctx->sort_vals[0].ensure(n_cand * 4));
      C2B_TRY(ctx->sort_vals[1].ensure(n_cand * 4));
      keys[0] = ctx->sort_keys[0].as<uint64_t>();
      keys[1] = ctx->sort_keys[1].as<uint64_t>();
      vals[0] = ctx->sort_vals[0].as<uint32_t>();
      vals[1] = ctx->sort_vals[1].as<uint32_t>();
      k_iota_u32<<<blocks_for(n_cand, 256), 256, 0, st>>>(vals[0], n_cand);
      C2B_KERNEL_CHECK();
      C2B_TRY(radix_sort_pairs(st, keys, vals, n_cand, pbits + cbits, ctx->sort_hist, ctx->scan_tmp, &res));
    }
    C2B_CUDA(cudaEventRecord(ctx->ev[EV_SORT], st));

    const uint64_t n_words = (n_cand + 31) / 32;
    C2B_TRY(ctx->vis_words.ensure((n_words + 1) * 4));
    C2B_TRY(ctx->word_prefix.ensure((n_words + 1) * 4));
    C2B_TRY(run_occlusion(keys[res], n_cand, n_words));
    C2B_CUDA(cudaEventRecord(ctx->ev[EV_TRAVERSE], st));

    C2B_CUDA(cudaMemsetAsync(d_total, 0, 8, st));
    if (n_cand) {
      C2B_TRY(ctx->out_idx[ctx->out_sel].ensure(n_cand * 4));
      C2B_TRY(ctx->out_uv[ctx->out_sel].ensure(n_cand * 16));
      k_word_popc<<<blocks_for(n_words, 256), 256, 0, st>>>(ctx->vis_words.as<uint32_t>(), n_words,
                                                            ctx->word_prefix.as<uint32_t>());
      C2B_KERNEL_CHECK();
      C2B_TRY(exclusive_scan_u32(st, ctx->word_prefix.as<uint32_t>(), ctx->word_prefix.as<uint32_t>(),
                                 n_words, d_total, ctx->scan_tmp));
      k_compact_write<<<blocks_for(n_cand, 256), 256, 0, st>>>(
          ctx->vis_words.as<uint32_t>(), ctx->word_prefix.as<uint32_t>(), keys[res], vals[res],
          ctx->pool_uv.as<double2>(), n_cand, pbits, ctx->out_idx[ctx->out_sel].as<uint32_t>(),
          ctx->out_uv[ctx->out_sel].as<double2>());
      C2B_KERNEL_CHECK();
    }
    k_csr_offsets<<<blocks_for(C + 1, 256), 256, 0, st>>>(
        ctx->cam_count.as<uint32_t>(), C, ctx->vis_words.as<uint32_t>(), ctx->word_prefix.as<uint32_t>(),
        n_cand, d_total, ctx->out_offsets[ctx->out_sel].as<uint64_t>());
    C2B_KERNEL_CHECK();
    C2B_CUDA(cudaEventRecord(ctx->ev[EV_COMPACT], st));
    C2B_CUDA(cudaEventRecord(ctx->ev[EV_D2H], st));
    C2B_TRY(read_counters(ctx, h_fin));
    uint32_t total32;
    memcpy(&total32, reinterpret_cast<const char *>(h_fin) + 48, 4);
    total_obs = total32;
  }
  ctx->out_C = C;
  ctx->out_O = total_obs;
  x->have_result = true;
  x->res_candidates = n_cand;
  fill_stats(ctx, stats, C, n_cand, pairs_eval, h_fin[2], h_fin[3]);
  return C2B_OK;
}

int c2b_download_obs(c2b_ctx *ctx, c2b_obs *out) {
  if (!ctx || !out) return set_error(C2B_ERR_INVALID, "c2b_download_obs: null argument");
  CtxExtra *x = ctx->extra.get();
  if (!x->have_result) return set_error(C2B_ERR_INVALID, "no resident result to download");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const uint64_t C = ctx->out_C, O = ctx->out_O;
  C2B_TRY(ctx->h_offsets.ensure((C + 1) * 8));
  C2B_TRY(ctx->h_idx.ensure(std::max<uint64_t>(O, 1) * 4));
  C2B_TRY(ctx->h_uv.ensure(std::max<uint64_t>(O, 1) * 16));
  cudaEvent_t e0 = ctx->ev[EV_COMPACT], e1 = ctx->ev[EV_D2H];
  C2B_CUDA(cudaEventRecord(e0, st));
  C2B_CUDA(cudaMemcpyAsync(ctx->h_offsets.p, ctx->out_offsets[ctx->out_sel].p, (C + 1) * 8, cudaMemcpyDeviceToHost, st));
  if (O) {
    C2B_CUDA(cudaMemcpyAsync(ctx->h_idx.p, ctx->out_idx[ctx->out_sel].p, O * 4, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaMemcpyAsync(ctx->h_uv.p, ctx->out_uv[ctx->out_sel].p, O * 16, cudaMemcpyDeviceToHost, st));
  }
  C2B_CUDA(cudaEventRecord(e1, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  out->n_cameras = C;
  out->n_obs = O;
  out->offsets = ctx->h_offsets.as<uint64_t>();
  out->point_idx = ctx->h_idx.as<uint32_t>();
  out->uv = ctx->h_uv.as<double>();
  out->d2h_bytes = (C + 1) * 8 + O * 20;
  float t = 0;
  cudaEventElapsedTime(&t, e0, e1);
  out->ms_d2h = t;
  return C2B_OK;
}

namespace {
__global__ void k_add_u64(uint64_t *v, uint64_t n, uint64_t add) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] += add;
}
}  // namespace

int c2b_download_obs_into(c2b_ctx *ctx, uint64_t obs_base, uint64_t *offsets_dst, uint32_t *idx_dst, double *uv_dst,
                          int with_end, float *ms_d2h) {
  if (!ctx || !offsets_dst) return set_error(C2B_ERR_INVALID, "c2b_download_obs_into: null argument");
  CtxExtra *x = ctx->extra.get();
  if (!x->have_result) return set_error(C2B_ERR_INVALID, "no resident result to download");
  const uint64_t C = ctx->out_C, O = ctx->out_O;
  if (O && (!idx_dst || !uv_dst)) return set_error(C2B_ERR_INVALID, "c2b_download_obs_into: null result array");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int sel = ctx->out_sel;
  if (obs_base) {
    k_add_u64<<<blocks_for(C + 1, 256), 256, 0, st>>>(ctx->out_offsets[sel].as<uint64_t>(), C + 1, obs_base);
    C2B_KERNEL_CHECK();
  }
  cudaEvent_t e0 = ctx->ev[EV_COMPACT], e1 = ctx->ev[EV_D2H];
  C2B_CUDA(cudaEventRecord(e0, st));
  C2B_CUDA(cudaMemcpyAsync(offsets_dst, ctx->out_offsets[sel].p, (C + (with_end ? 1 : 0)) * 8, cudaMemcpyDeviceToHost, st));
  if (O) {
    C2B_CUDA(cudaMemcpyAsync(idx_dst, ctx->out_idx[sel].p, O * 4, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaMemcpyAsync(uv_dst, ctx->out_uv[sel].p, O * 16, cudaMemcpyDeviceToHost, st));
  }
  C2B_CUDA(cudaEventRecord(e1, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  if (obs_base) {  // leave the resident CSR as it was (a second download must not rebase twice)
    k_add_u64<<<blocks_for(C + 1, 256), 256, 0, st>>>(ctx->out_offsets[sel].as<uint64_t>(), C + 1, (uint64_t)0 - obs_base);
    C2B_KERNEL_CHECK();
  }
  if (ms_d2h) {
    float t = 0;
    cudaEventElapsedTime(&t, e0, e1);
    *ms_d2h = t;
  }
  return C2B_OK;
}

namespace {

// grow a pinned result buffer while copies into it may be in flight: drain, allocate, carry over
int grow_pinned(c2b_ctx *ctx, PinBuf &b, size_t need, size_t used) {
  if (need <= b.cap) return C2B_OK;
  C2B_CUDA(cudaStreamSynchronize(ctx->copy_stream));
  PinBuf nb;
  nb.node = b.node;
  C2B_TRY(nb.ensure(need + need / 16));
  if (used) memcpy(nb.p, b.p, used);
  b = std::move(nb);
  return C2B_OK;
}
}  // namespace

int c2b_visibility_graph(c2b_ctx *ctx, const c2b_scene *scene, const double *cams, uint64_t C,
                         const double *pts, uint64_t P, double max_dist, const c2b_vis_options *opt,
                         c2b_obs *out) {
  if (!ctx || !out) return set_error(C2B_ERR_INVALID, "c2b_visibility_graph: null argument");
  if (C && !cams) return set_error(C2B_ERR_INVALID, "c2b_visibility_graph: null camera array");
  C2B_CUDA(cudaSetDevice(ctx->device));
  CtxExtra *x = ctx->extra.get();
  // pts == NULL: use the points already resident on the device (c2b_upload_points[_device])
  const bool resident_pts = P && !pts;
  if (resident_pts && !(x->have_points && ctx->P == P))
    return set_error(C2B_ERR_INVALID, "c2b_visibility_graph: pts is null and no %llu resident points were uploaded",
                     (unsigned long long)P);
  cudaStream_t st = ctx->stream, cs = ctx->copy_stream;
  // Camera batches: the CSR slab of batch b travels to the host while batch b+1 is computed.  A batch should
  // give every resident warp of the fused kernel more than one camera (a short batch leaves warps idle at its
  // tail and repeats the per-batch plan / scan / sync), and:
  //   * when the result transfer is the longest leg (20 B per observation over PCIe: cfg4) it should start
  //     early — a small first batch, then growing ones;
  //   * when the kernels are (fine meshes: cfg5) the batches should be few and equal — only the last slab's
  //     transfer is exposed.
  // Which case applies is taken from the previous call on this ctx; the first call assumes the transfer.
  std::vector<uint64_t> bounds;  // batch b = cameras [bounds[b], bounds[b+1])
  bounds.push_back(0);
  const uint64_t W = (uint64_t)ctx->sm_count * FU_RESIDENT_WARPS;  // resident warps of the fused kernel
  if (x->tun.batches > 0) {
    const uint64_t nb = std::max<uint64_t>(1, std::min<uint64_t>(C ? C : 1, (uint64_t)x->tun.batches));
    for (uint64_t b = 1; b <= nb; ++b) bounds.push_back((b * C) / nb);
  } else if (C < 3 * W) {
    bounds.push_back(C);
  } else if (x->hist.valid && x->hist.ms_compute_per_cam > x->hist.d2h_bytes_per_cam / 52e6) {
    const uint64_t nb = std::min<uint64_t>(std::max<uint64_t>(C / (3 * W), 2), 4);
    for (uint64_t b = 1; b <= nb; ++b) bounds.push_back((b * C) / nb);
  } else {
    uint64_t done = 0, size = std::max<uint64_t>(3 * W / 2, C / 32);
    const uint64_t cap = std::max<uint64_t>(3 * W, C / 6);
    while (C - done > size + size / 2) {
      done += size;
      bounds.push_back(done);
      size = std::min(2 * size, cap);
    }
    bounds.push_back(C);
  }
  const uint64_t n_batches = bounds.size() - 1;

  Event u0, u1, d0, d1;
  C2B_TRY(u0.create());
  C2B_TRY(u1.create());
  C2B_TRY(d0.create());
  C2B_TRY(d1.create());
  c2b_obs acc;
  memset(&acc, 0, sizeof acc);
  int rc = C2B_OK;
  uint64_t obs_base = 0;
  float ms_upload = 0, ms_copy = 0;
  // First host-buffer call on this ctx: the CSR goes to unpinned memory through the Drainer (see PageBuf).
  const bool staged = x->tun.cold_staged && x->tun.stage_threads > 0 && !x->hist.valid && ctx->h_uv.cap < (64u << 20);
  Drainer drain;
  std::chrono::steady_clock::time_point t_first_copy;
  bool copy_started = false;
  if (!staged) {
    x->pg_idx.release();
    x->pg_uv.release();
  }
  auto run = [&]() -> int {
    if (staged) {
      const int nthreads = std::max(2, x->tun.stage_threads);
      x->pin_out.node = ctx->numa_node;
      C2B_TRY(x->pin_out.ensure((size_t)nthreads * 2 * Drainer::CH));
      C2B_TRY(drain.start(ctx->device, nthreads, x->pin_out.as<char>()));
    }
    C2B_CUDA(cudaEventRecord(u0, st));
    if (!resident_pts) C2B_TRY(c2b_upload_points(ctx, pts, P));
    C2B_CUDA(cudaEventRecord(u1, st));
    // the point grid once, for the reach of ALL of this call's cameras (each batch's reach lies inside it)
    const bool grid_mode = !opt || opt->cull_mode == C2B_CULL_GRID;
    // all cameras cross PCIe once; the batches are device-side slices of that copy
    if (C) {
      C2B_TRY(ctx->cams_all.ensure(C * 120));
      C2B_TRY(copy_in(ctx, ctx->cams_all.p, cams, C * 120, cudaMemcpyHostToDevice));
    }
    if (grid_mode && n_batches > 1 && C && P) {
      C2B_TRY(select_cameras(ctx, 0, C));
      C2B_TRY(ensure_grid(ctx, x, max_dist));
      x->grid_locked = true;
    }
    C2B_TRY(ctx->h_offsets.ensure((C + 1) * 8));
    // camera ranges still to do, in order; a range that turns out too large for 32-bit offsets is halved
    std::vector<std::pair<uint64_t, uint64_t>> todo;
    for (uint64_t b = n_batches; b-- > 0;) todo.push_back({bounds[b], bounds[b + 1]});
    for (uint64_t b = 0; !todo.empty(); ++b) {
      const uint64_t c0 = todo.back().first, c1 = todo.back().second, nc = c1 - c0;
      todo.pop_back();
      const int sel = (int)(b & 1);
      ctx->out_sel = sel;
      if (b >= 2) {  // set `sel` is free again once batch b - 2 has left the device
        if (staged)
          drain.wait_dma((int)b - 2);
        else
          C2B_CUDA(cudaStreamWaitEvent(st, ctx->ev_copied[sel], 0));
      }
      C2B_TRY(select_cameras(ctx, c0, nc));
      c2b_obs s1;
      const int rcb = visibility_resident_impl(ctx, scene, max_dist, opt, &s1);
      if (rcb == ERR_TOO_LARGE && nc > 1) {
        todo.push_back({c0 + nc / 2, c1});
        todo.push_back({c0, c0 + nc / 2});
        --b;  // the buffer set was not used
        continue;
      }
      if (rcb != C2B_OK) return rcb == ERR_TOO_LARGE ? C2B_ERR_INVALID : rcb;
      const uint64_t O = ctx->out_O;
      if (obs_base)
        k_add_u64<<<blocks_for(nc + 1, 256), 256, 0, st>>>(ctx->out_offsets[sel].as<uint64_t>(), nc + 1, obs_base);
      ++launch_counter();
      C2B_CUDA(cudaEventRecord(ctx->ev_ready[sel], st));
      // result arrays: sized from the first batch's density, grown if the guess was short
      size_t need = obs_base + O;
      if (!todo.empty()) need = std::max<size_t>(need, (size_t)((double)(obs_base + O) * (double)C / (double)c1 * 1.05) + 1024);
      C2B_CUDA(cudaStreamWaitEvent(cs, ctx->ev_ready[sel], 0));
      if (b == 0) C2B_CUDA(cudaEventRecord(d0, cs));
      C2B_CUDA(cudaMemcpyAsync(ctx->h_offsets.as<uint64_t>() + c0, ctx->out_offsets[sel].p, (nc + 1) * 8,
                               cudaMemcpyDeviceToHost, cs));
      if (staged) {
        // untouched virtual memory costs nothing: reserve twice the estimate; a second reservation (after
        // draining, with the landed part carried over) only if even that was short
        for (PageBuf *pb : {&x->pg_idx, &x->pg_uv}) {
          const size_t unit = pb == &x->pg_idx ? 4 : 16;
          if (std::max<size_t>(need, 1) * unit > pb->cap) {
            drain.wait_all();
            PageBuf bigger;
            C2B_TRY(bigger.ensure_fresh(2 * std::max<size_t>(need, 1) * unit));
            if (obs_base) memcpy(bigger.p, pb->p, obs_base * unit);
            *pb = std::move(bigger);
          }
        }
        if (!copy_started) {
          copy_started = true;
          t_first_copy = std::chrono::steady_clock::now();
        }
        if (O) {
          drain.submit(ctx->out_idx[sel].p, x->pg_idx.as<uint32_t>() + obs_base, O * 4, ctx->ev_ready[sel], (int)b);
          drain.submit(ctx->out_uv[sel].p, x->pg_uv.as<double>() + 2 * obs_base, O * 16, ctx->ev_ready[sel], (int)b);
        }
      } else {
        C2B_TRY(grow_pinned(ctx, ctx->h_idx, std::max<size_t>(need, 1) * 4, obs_base * 4));
        C2B_TRY(grow_pinned(ctx, ctx->h_uv, std::max<size_t>(need, 1) * 16, obs_base * 16));
        if (O) {
          C2B_CUDA(cudaMemcpyAsync(ctx->h_idx.as<uint32_t>() + obs_base, ctx->out_idx[sel].p, O * 4,
                                   cudaMemcpyDeviceToHost, cs));
          C2B_CUDA(cudaMemcpyAsync(ctx->h_uv.as<double>() + 2 * obs_base, ctx->out_uv[sel].p, O * 16,
                                   cudaMemcpyDeviceToHost, cs));
        }
        C2B_CUDA(cudaEventRecord(ctx->ev_copied[sel], cs));
      }
      obs_base += O;
      acc.n_candidates += s1.n_candidates;
      acc.pairs_evaluated += s1.pairs_evaluated;
      acc.nodes_visited += s1.nodes_visited;
      acc.tris_tested += s1.tris_tested;
      acc.ms_prep += s1.ms_prep;
      acc.ms_cull += s1.ms_cull;
      acc.ms_sort += s1.ms_sort;
      acc.ms_traverse += s1.ms_traverse;
      acc.ms_compact += s1.ms_compact;
      acc.ms_total += s1.ms_total;
    }
    C2B_CUDA(cudaEventRecord(d1, cs));
    C2B_CUDA(cudaStreamSynchronize(cs));
    C2B_CUDA(cudaStreamSynchronize(st));
    C2B_CUDA(cudaEventElapsedTime(&ms_upload, u0, u1));
    C2B_CUDA(cudaEventElapsedTime(&ms_copy, d0, d1));
    if (staged) {
      const cudaError_t e = drain.finish();
      if (e != cudaSuccess) return set_error(C2B_ERR_CUDA, "staged device-to-host copy failed: %s", cudaGetErrorString(e));
      if (copy_started)
        ms_copy = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_first_copy).count();
    }
    return C2B_OK;
  };
  rc = run();
  x->grid_locked = false;
  ctx->out_sel = 0;
  x->have_result = false;  // the resident state now holds the last batch only
  x->host_call_last = true;
  if (rc != C2B_OK) {
    cudaStreamSynchronize(cs);
    return rc;
  }
  acc.n_cameras = C;
  acc.n_obs = obs_base;
  acc.offsets = ctx->h_offsets.as<uint64_t>();
  acc.point_idx = staged ? x->pg_idx.as<uint32_t>() : ctx->h_idx.as<uint32_t>();
  acc.uv = staged ? x->pg_uv.as<double>() : ctx->h_uv.as<double>();
  acc.ms_h2d = ms_upload;
  acc.h2d_bytes = (resident_pts ? 0 : P * 24) + C * 120;
  acc.d2h_bytes = (C + 1) * 8 + obs_base * 20;
  acc.ms_d2h = ms_copy;  // first to last result copy on the copy stream; overlaps the compute of later batches
  acc.ms_total += ms_upload;
  if (C) {
    x->hist.valid = true;
    x->hist.ms_compute_per_cam = (acc.ms_prep + acc.ms_cull + acc.ms_sort + acc.ms_traverse + acc.ms_compact) / (double)C;
    x->hist.d2h_bytes_per_cam = (double)acc.d2h_bytes / (double)C;
  }
  *out = acc;
  return C2B_OK;
}

void c2b_obs_free(c2b_ctx *ctx, c2b_obs *obs) {
  (void)ctx;  // the pinned buffers are pooled in the ctx and reused by the next call
  if (!obs) return;
  obs->offsets = nullptr;
  obs->point_idx = nullptr;
  obs->uv = nullptr;
  obs->n_obs = 0;
}

int c2b_reprojection_error_resident(c2b_ctx *ctx, double norm, double *out) {
  if (!ctx || !out) return set_error(C2B_ERR_INVALID, "c2b_reprojection_error_resident: null argument");
  CtxExtra *x = ctx->extra.get();
  if (!x->have_result) return set_error(C2B_ERR_INVALID, "no resident result");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const uint64_t C = ctx->out_C, O = ctx->out_O, P = ctx->P;
  *out = 0.0;
  if (O == 0) return C2B_OK;
  int nb = (int)std::min<uint64_t>(blocks_for(O, ST_THREADS), ST_BLOCKS);
  C2B_TRY(ctx->misc.ensure((size_t)nb * 8 + 64));
  const double *px = ctx->pts.as<double>();
  k_reproj_partial<<<nb, ST_THREADS, 0, st>>>(ctx->cams.as<double>(), px, px + P, px + 2 * P,
                                              ctx->out_offsets[ctx->out_sel].as<uint64_t>(), C,
                                              ctx->out_idx[ctx->out_sel].as<uint32_t>(), ctx->out_uv[ctx->out_sel].as<double2>(), O,
                                              norm, ctx->misc.as<double>());
  C2B_KERNEL_CHECK();
  std::vector<double> h(nb);
  C2B_CUDA(cudaMemcpyAsync(h.data(), ctx->misc.p, (size_t)nb * 8, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  double s = 0;
  for (double v : h) s += v;
  *out = std::pow(s, 1.0 / norm);
  return C2B_OK;
}

// ---- noise ----------------------------------------------------------------------------------------------
namespace {
// the arrays a noise pass works on, all on the device
struct NoiseView {
  double *cams = nullptr;     // [15 C]
  double *centers = nullptr;  // [3 C] SoA, up to date with cams
  double *pts = nullptr;      // [3 P] xyz records
  double2 *uv = nullptr;      // [O]
  uint64_t C = 0, P = 0, O = 0;
};

// device time of the last noise call: [0] upload, [1] statistics + kernels, [2] download
struct NoiseTimer {
  c2b_ctx *ctx;
  Event ev[4];
  explicit NoiseTimer(c2b_ctx *c) : ctx(c) {
    for (auto &e : ev) (void)e.create();
    cudaEventRecord(ev[0], ctx->stream);
  }
  void mark(int k) { cudaEventRecord(ev[k], ctx->stream); }
  void finish() {
    for (int k = 0; k < 3; ++k) {
      float t = 0;
      if (cudaEventElapsedTime(&t, ev[k], ev[k + 1]) != cudaSuccess) (void)cudaGetLastError();
      ctx->noise_ms[k] = t;
    }
  }
};

inline unsigned nz_grid(c2b_ctx *ctx, uint64_t n) {
  return (unsigned)std::min<uint64_t>(std::max<uint64_t>(blocks_for(n, NZ_THREADS), 1), (uint64_t)ctx->sm_count * 8);
}

// mean / std / nearest-origin of the chained sequence on the device.  scratch layout (doubles):
// [0..2] mean, [3..5] sumsq, [6..8] origin, then partials.
int device_stats(c2b_ctx *ctx, const NoiseView &v, double mean[3], double sd[3], bool want_origin, bool to_host = true) {
  cudaStream_t st = ctx->stream;
  const uint64_t C = v.C, P = v.P, n = C + P;
  const double num = (double)n;
  int blocks = (int)std::min<uint64_t>(std::max<uint64_t>(blocks_for(n, ST_THREADS), 1), ST_BLOCKS);
  C2B_TRY(ctx->nz_scratch.ensure((size_t)(16 + 8 * blocks) * 8));
  double *s = ctx->nz_scratch.as<double>();
  double *partial = s + 16;
  const double *cx = v.centers;
  const double *pts = v.pts;
  // the chain stays on the device: the second pass reads the mean the first one left in s[0..2]
  k_stats_partial<0><<<blocks, ST_THREADS, 0, st>>>(cx, cx + C, cx + 2 * C, C, pts, P, num, s, partial);
  C2B_KERNEL_CHECK();
  k_stats_final<<<1, 32, 0, st>>>(partial, blocks, s);
  C2B_KERNEL_CHECK();
  k_stats_partial<1><<<blocks, ST_THREADS, 0, st>>>(cx, cx + C, cx + 2 * C, C, pts, P, num, s, partial);
  C2B_KERNEL_CHECK();
  k_stats_final<<<1, 32, 0, st>>>(partial, blocks, s + 3);
  C2B_KERNEL_CHECK();
  k_bal_std<<<1, 32, 0, st>>>(s, num);
  C2B_KERNEL_CHECK();
  if (want_origin) {
    double *pd = partial;
    unsigned long long *pi = reinterpret_cast<unsigned long long *>(partial + blocks);
    k_nearest_partial<<<blocks, ST_THREADS, 0, st>>>(cx, cx + C, cx + 2 * C, C, pts, P, pd, pi);
    C2B_KERNEL_CHECK();
    k_nearest_final<<<1, 32, 0, st>>>(pd, pi, blocks, cx, cx + C, cx + 2 * C, C, pts, s + 6);
    C2B_KERNEL_CHECK();
  }
  if (to_host) {
    double h[6];
    C2B_CUDA(cudaMemcpyAsync(h, s, 48, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaStreamSynchronize(st));
    for (int k = 0; k < 3; ++k) {
      mean[k] = h[k];
      sd[k] = std::sqrt(h[3 + k] / num);
    }
  }
  return C2B_OK;
}

// host arrays -> the ctx's noise buffers (grow-only, kept between calls)
int noise_upload(c2b_ctx *ctx, NoiseView &v, const double *cams, uint64_t C, const double *pts, uint64_t P) {
  cudaStream_t st = ctx->stream;
  C2B_TRY(ctx->nz_cams.ensure(std::max<uint64_t>(C, 1) * 120));
  C2B_TRY(ctx->nz_centers.ensure(std::max<uint64_t>(C, 1) * 24));
  C2B_TRY(ctx->nz_pts.ensure(std::max<uint64_t>(P, 1) * 24));
  v.cams = ctx->nz_cams.as<double>();
  v.centers = ctx->nz_centers.as<double>();
  v.pts = ctx->nz_pts.as<double>();
  v.C = C;
  v.P = P;
  if (C) {
    C2B_TRY(copy_in(ctx, v.cams, cams, C * 120, cudaMemcpyHostToDevice));
    k_cam_prep<<<blocks_for(C, 128), 128, 0, st>>>(v.cams, C, v.centers, v.centers + C, v.centers + 2 * C);
    C2B_KERNEL_CHECK();
  }
  if (P) C2B_TRY(copy_in(ctx, v.pts, pts, P * 24, cudaMemcpyHostToDevice));
  return C2B_OK;
}

// the resident problem as a NoiseView (cameras + points of the last uploads, (u, v) of the last resident pass)
int resident_view(c2b_ctx *ctx, NoiseView &v, const char *who) {
  CtxExtra *x = ctx->extra.get();
  if (!x->have_points || !x->have_cameras) return set_error(C2B_ERR_INVALID, "%s: upload cameras and points first", who);
  v.cams = ctx->cams.as<double>();
  v.centers = ctx->cam_center.as<double>();
  v.pts = ctx->pts_aos.as<double>();
  v.C = ctx->C;
  v.P = ctx->P;
  v.uv = x->have_result ? ctx->out_uv[ctx->out_sel].as<double2>() : nullptr;
  v.O = x->have_result ? ctx->out_O : 0;
  return C2B_OK;
}

// after a resident noise pass: camera centres and the SoA points / bounds / grid follow the new values
int resident_refresh(c2b_ctx *ctx, bool cams_moved, bool pts_moved) {
  if (cams_moved && ctx->C) {
    double *cx = ctx->cam_center.as<double>();
    k_cam_prep<<<blocks_for(ctx->C, 128), 128, 0, ctx->stream>>>(ctx->cams.as<double>(), ctx->C, cx, cx + ctx->C, cx + 2 * ctx->C);
    C2B_KERNEL_CHECK();
  }
  if (pts_moved) {
    CtxExtra *x = ctx->extra.get();
    const bool had = x->have_result;
    C2B_TRY(c2b_points_commit(ctx, ctx->P));
    x->have_result = had;  // the CSR is still the graph of this problem
  }
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));
  return C2B_OK;
}

int drift_kernels(c2b_ctx *ctx, const NoiseView &v, double strength, double angle_strength, double std_,
                  const double *dir_in, bool normalized, uint64_t seed) {
  cudaStream_t st = ctx->stream;
  double mean[3], sd[3];
  C2B_TRY(device_stats(ctx, v, mean, sd, true));
  V3 dir;
  if (normalized) {
    // add_drift_normalized, src/noise.rs:53-55
    V3 s{sd[0], sd[1], sd[2]};
    double m = std::sqrt((s.x * s.x + s.y * s.y) + s.z * s.z);
    double inv = 1.0 / m;
    dir = V3{s.x * inv, s.y * inv, s.z * inv};
    strength = strength * m;
  } else {
    dir = V3{dir_in[0], dir_in[1], dir_in[2]};
  }
  const double *origin = ctx->nz_scratch.as<double>() + 6;
  if (v.C) {
    k_drift_cams<<<blocks_for(v.C, NZ_THREADS), NZ_THREADS, 0, st>>>(v.cams, v.C, origin, dir, strength, angle_strength, std_, seed);
    C2B_KERNEL_CHECK();
  }
  if (v.P) {
    k_drift_pts<<<nz_grid(ctx, v.P), NZ_THREADS, 0, st>>>(v.pts, v.P, origin, dir, strength, std_, seed);
    C2B_KERNEL_CHECK();
  }
  return C2B_OK;
}

int drift_impl(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, double strength,
               double angle_strength, double std_, const double *dir_in, bool normalized,
               uint64_t seed) {
  if (!ctx || (C && !cams) || (P && !pts)) return set_error(C2B_ERR_INVALID, "add_drift: null argument");
  if (C + P == 0) return set_error(C2B_ERR_EMPTY, "add_drift: problem has no cameras and no points");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  NoiseView v;
  NoiseTimer tm(ctx);
  C2B_TRY(noise_upload(ctx, v, cams, C, pts, P));
  tm.mark(1);
  C2B_TRY(drift_kernels(ctx, v, strength, angle_strength, std_, dir_in, normalized, seed));
  tm.mark(2);
  if (C) C2B_CUDA(cudaMemcpyAsync(cams, v.cams, C * 120, cudaMemcpyDeviceToHost, st));
  if (P) C2B_CUDA(cudaMemcpyAsync(pts, v.pts, P * 24, cudaMemcpyDeviceToHost, st));
  tm.mark(3);
  C2B_CUDA(cudaStreamSynchronize(st));
  tm.finish();
  return C2B_OK;
}

// cameras and points of add_noise (the observations are separate: the host entry streams them in chunks)
int noise_kernels(c2b_ctx *ctx, const NoiseView &v, double translation_std, double rotation_std, double point_std,
                  uint64_t seed) {
  cudaStream_t st = ctx->stream;
  // |std()| scales the camera translations (src/noise.rs:127,141); it stays on the device (scratch[9])
  C2B_TRY(device_stats(ctx, v, nullptr, nullptr, false, false));
  if (v.C) {
    k_noise_cams<<<blocks_for(v.C, NZ_THREADS), NZ_THREADS, 0, st>>>(v.cams, v.C, ctx->nz_scratch.as<double>() + 9,
                                                                    translation_std, rotation_std, seed);
    C2B_KERNEL_CHECK();
  }
  // a zero standard deviation adds unit_random() * 0 (src/noise.rs:149,159-168): the array is unchanged, so its
  // kernel — and in the host entry its round trip over PCIe — is skipped
  if (v.P && point_std != 0.0) {
    k_noise_pts<<<nz_grid(ctx, v.P), NZ_THREADS, 0, st>>>(v.pts, v.P, point_std, seed);
    C2B_KERNEL_CHECK();
  }
  return C2B_OK;
}

int sin_kernels(c2b_ctx *ctx, const NoiseView &v, const double dir[3], const double noise_dir[3], double strength,
                double frequency) {
  cudaStream_t st = ctx->stream;
  const uint64_t C = v.C, P = v.P, n = C + P;
  int blocks = (int)std::min<uint64_t>(std::max<uint64_t>(blocks_for(n, ST_THREADS), 1), ST_BLOCKS);
  C2B_TRY(ctx->nz_scratch.ensure((size_t)(8 + 6 * blocks) * 8));
  double *s = ctx->nz_scratch.as<double>();
  const double *cx = v.centers;
  k_extent_partial<<<blocks, ST_THREADS, 0, st>>>(cx, cx + C, cx + 2 * C, C, v.pts, P, s + 8);
  C2B_KERNEL_CHECK();
  k_extent_final<<<1, 32, 0, st>>>(s + 8, blocks, s);
  C2B_KERNEL_CHECK();
  double ext[6];
  C2B_CUDA(cudaMemcpyAsync(ext, s, 48, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  V3 dim{ext[3] - ext[0], ext[4] - ext[1], ext[5] - ext[2]};
  // "Add epsilon to nonexistent dimensions" (src/noise.rs:395-396)
  if (dim.x == 0.0) dim.x = 1e-8;
  if (dim.y == 0.0) dim.y = 1e-8;
  if (dim.z == 0.0) dim.z = 1e-8;
  const double nm = std::sqrt((noise_dir[0] * noise_dir[0] + noise_dir[1] * noise_dir[1]) + noise_dir[2] * noise_dir[2]);
  const double inv = 1.0 / nm;
  const V3 nd{noise_dir[0] * inv, noise_dir[1] * inv, noise_dir[2] * inv}, d{dir[0], dir[1], dir[2]};
  if (C) {
    k_sin_cams<<<blocks_for(C, 128), 128, 0, st>>>(v.cams, C, dim, d, nd, strength, frequency);
    C2B_KERNEL_CHECK();
  }
  if (P) {
    k_sin_pts<<<blocks_for(P, 256), 256, 0, st>>>(v.pts, P, dim, d, nd, strength, frequency);
    C2B_KERNEL_CHECK();
  }
  return C2B_OK;
}
}  // namespace

int c2b_add_drift(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, double strength,
                  double angle_strength, double std_, const double dir[3], uint64_t seed) {
  if (!dir) return set_error(C2B_ERR_INVALID, "c2b_add_drift: dir is null");
  return drift_impl(ctx, cams, C, pts, P, strength, angle_strength, std_, dir, false, seed);
}

int c2b_add_drift_normalized(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P,
                             double strength, double angle_strength, double std_, uint64_t seed) {
  return drift_impl(ctx, cams, C, pts, P, strength, angle_strength, std_, nullptr, true, seed);
}

int c2b_add_noise(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, double *uv,
                  uint64_t O, double translation_std, double rotation_std, double point_std,
                  double observations_std, uint64_t seed) {
  if (!ctx || (C && !cams) || (P && !pts) || (O && !uv))
    return set_error(C2B_ERR_INVALID, "c2b_add_noise: null argument");
  if (C + P == 0) return set_error(C2B_ERR_EMPTY, "add_noise: problem has no cameras and no points");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream, cs = ctx->copy_stream;
  NoiseView v;
  NoiseTimer tm(ctx);
  if (observations_std == 0.0) O = 0;
  // The observations (16 B each way, by far the largest array) stream through the GPU in chunks on the copy
  // stream while cameras and points are handled on the main one: PCIe is full duplex, so chunk k's download
  // overlaps chunk k+1's upload and the call costs about one direction of the transfer, not two.
  Event obs_done;
  if (O) {
    const uint64_t chunk = std::max<uint64_t>(1u << 20, (O + 15) / 16);
    C2B_TRY(ctx->nz_uv.ensure(std::min(O, 2 * chunk) * 16));
    double2 *buf = ctx->nz_uv.as<double2>();
    Event slot_free[2], up[2];
    for (int k = 0; k < 2; ++k) {
      C2B_TRY(slot_free[k].create(cudaEventDisableTiming));
      C2B_TRY(up[k].create(cudaEventDisableTiming));
    }
    C2B_TRY(obs_done.create(cudaEventDisableTiming));
    // uploads + kernels on the aux stream, downloads on the copy stream; two slots
    cudaStream_t ax = ctx->aux_stream;
    uint64_t k = 0;
    for (uint64_t first = 0; first < O; first += chunk, ++k) {
      const uint64_t n = std::min(chunk, O - first);
      const int slot = (int)(k & 1);
      double2 *d = buf + (uint64_t)slot * chunk;
      if (k >= 2) C2B_CUDA(cudaStreamWaitEvent(ax, slot_free[slot], 0));
      C2B_CUDA(cudaMemcpyAsync(d, uv + 2 * first, n * 16, cudaMemcpyHostToDevice, ax));
      k_noise_obs<<<nz_grid(ctx, n), NZ_THREADS, 0, ax>>>(d, n, first, observations_std, seed);
      C2B_KERNEL_CHECK();
      C2B_CUDA(cudaEventRecord(up[slot], ax));
      C2B_CUDA(cudaStreamWaitEvent(cs, up[slot], 0));
      C2B_CUDA(cudaMemcpyAsync(uv + 2 * first, d, n * 16, cudaMemcpyDeviceToHost, cs));
      C2B_CUDA(cudaEventRecord(slot_free[slot], cs));
    }
    C2B_CUDA(cudaEventRecord(obs_done, cs));
  }
  C2B_TRY(noise_upload(ctx, v, cams, C, pts, P));
  tm.mark(1);
  C2B_TRY(noise_kernels(ctx, v, translation_std, rotation_std, point_std, seed));
  tm.mark(2);
  if (C) C2B_CUDA(cudaMemcpyAsync(cams, v.cams, C * 120, cudaMemcpyDeviceToHost, st));
  if (P && point_std != 0.0) C2B_CUDA(cudaMemcpyAsync(pts, v.pts, P * 24, cudaMemcpyDeviceToHost, st));
  if (obs_done) C2B_CUDA(cudaStreamWaitEvent(st, obs_done, 0));
  tm.mark(3);
  C2B_CUDA(cudaStreamSynchronize(st));
  tm.finish();
  return C2B_OK;
}

int c2b_add_sin_noise(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, const double dir[3],
                      const double noise_dir[3], double strength, double frequency) {
  if (!ctx || (C && !cams) || (P && !pts) || !dir || !noise_dir)
    return set_error(C2B_ERR_INVALID, "c2b_add_sin_noise: null argument");
  if (C + P == 0) return set_error(C2B_ERR_EMPTY, "add_sin_noise: problem has no cameras and no points");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  NoiseView v;
  NoiseTimer tm(ctx);
  C2B_TRY(noise_upload(ctx, v, cams, C, pts, P));
  tm.mark(1);
  C2B_TRY(sin_kernels(ctx, v, dir, noise_dir, strength, frequency));
  tm.mark(2);
  if (C) C2B_CUDA(cudaMemcpyAsync(cams, v.cams, C * 120, cudaMemcpyDeviceToHost, st));
  if (P) C2B_CUDA(cudaMemcpyAsync(pts, v.pts, P * 24, cudaMemcpyDeviceToHost, st));
  tm.mark(3);
  C2B_CUDA(cudaStreamSynchronize(st));
  tm.finish();
  return C2B_OK;
}

// ---- the same passes on the RESIDENT problem: no PCIe traffic at all -------------------------------------
int c2b_add_drift_resident(c2b_ctx *ctx, double strength, double angle_strength, double std_, const double *dir,
                           uint64_t seed) {
  if (!ctx) return set_error(C2B_ERR_INVALID, "c2b_add_drift_resident: null ctx");
  C2B_CUDA(cudaSetDevice(ctx->device));
  NoiseView v;
  C2B_TRY(resident_view(ctx, v, "c2b_add_drift_resident"));
  if (v.C + v.P == 0) return set_error(C2B_ERR_EMPTY, "add_drift: problem has no cameras and no points");
  NoiseTimer tm(ctx);
  tm.mark(1);
  C2B_TRY(drift_kernels(ctx, v, strength, angle_strength, std_, dir, dir == nullptr, seed));
  tm.mark(2);
  tm.mark(3);
  C2B_TRY(resident_refresh(ctx, true, true));
  tm.finish();
  return C2B_OK;
}

int c2b_add_noise_resident(c2b_ctx *ctx, double translation_std, double rotation_std, double point_std,
                           double observations_std, uint64_t seed) {
  if (!ctx) return set_error(C2B_ERR_INVALID, "c2b_add_noise_resident: null ctx");
  C2B_CUDA(cudaSetDevice(ctx->device));
  NoiseView v;
  C2B_TRY(resident_view(ctx, v, "c2b_add_noise_resident"));
  if (v.C + v.P == 0) return set_error(C2B_ERR_EMPTY, "add_noise: problem has no cameras and no points");
  NoiseTimer tm(ctx);
  tm.mark(1);
  C2B_TRY(noise_kernels(ctx, v, translation_std, rotation_std, point_std, seed));
  if (v.O && observations_std != 0.0) {
    k_noise_obs<<<nz_grid(ctx, v.O), NZ_THREADS, 0, ctx->stream>>>(v.uv, v.O, 0, observations_std, seed);
    C2B_KERNEL_CHECK();
  }
  tm.mark(2);
  tm.mark(3);
  C2B_TRY(resident_refresh(ctx, true, point_std != 0.0));
  tm.finish();
  return C2B_OK;
}

int c2b_add_sin_noise_resident(c2b_ctx *ctx, const double dir[3], const double noise_dir[3], double strength,
                               double frequency) {
  if (!ctx || !dir || !noise_dir) return set_error(C2B_ERR_INVALID, "c2b_add_sin_noise_resident: null argument");
  C2B_CUDA(cudaSetDevice(ctx->device));
  NoiseView v;
  C2B_TRY(resident_view(ctx, v, "c2b_add_sin_noise_resident"));
  if (v.C + v.P == 0) return set_error(C2B_ERR_EMPTY, "add_sin_noise: problem has no cameras and no points");
  NoiseTimer tm(ctx);
  tm.mark(1);
  C2B_TRY(sin_kernels(ctx, v, dir, noise_dir, strength, frequency));
  tm.mark(2);
  tm.mark(3);
  C2B_TRY(resident_refresh(ctx, true, true));
  tm.finish();
  return C2B_OK;
}

int c2b_download_problem(c2b_ctx *ctx, double *cams_out, double *pts_out) {
  if (!ctx) return set_error(C2B_ERR_INVALID, "c2b_download_problem: null ctx");
  NoiseView v;
  C2B_TRY(resident_view(ctx, v, "c2b_download_problem"));
  if ((v.C && !cams_out) || (v.P && !pts_out)) return set_error(C2B_ERR_INVALID, "c2b_download_problem: null output array");
  C2B_CUDA(cudaSetDevice(ctx->device));
  if (v.C) C2B_CUDA(cudaMemcpyAsync(cams_out, v.cams, v.C * 120, cudaMemcpyDeviceToHost, ctx->stream));
  if (v.P) C2B_CUDA(cudaMemcpyAsync(pts_out, v.pts, v.P * 24, cudaMemcpyDeviceToHost, ctx->stream));
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));
  return C2B_OK;
}

int c2b_noise_timing(c2b_ctx *ctx, float ms[3]) {
  if (!ctx || !ms) return set_error(C2B_ERR_INVALID, "c2b_noise_timing: null argument");
  for (int k = 0; k < 3; ++k) ms[k] = ctx->noise_ms[k];
  return C2B_OK;
}

// ---- input generation: world points (src/generate.rs:356-420) -----------------------------------------
int c2b_generate_world_points_uniform(c2b_ctx *ctx, const float *xyz, uint64_t nv, const uint32_t *tri,
                                      uint64_t nt, const double *cams, uint64_t C, uint64_t num_points,
                                      double max_dist, uint64_t seed, double *pts_out, uint64_t *n_out) {
  if (!ctx || !n_out || (nv && !xyz) || (nt && !tri) || (C && !cams) || (num_points && !pts_out))
    return set_error(C2B_ERR_INVALID, "c2b_generate_world_points_uniform: null argument");
  *n_out = 0;
  if (C == 0)
    return set_error(C2B_ERR_INVALID, "Cannot generate world points with 0 cameras. Try increasing the number of "
                                      "cameras generated (via --cameras).");
  if (num_points == 0) return C2B_OK;
  if (num_points >= 0x7fffffffull) return set_error(C2B_ERR_INVALID, "too many points requested");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // areas and their running sum (sequential f64, the WeightedIndex table); vertices as float4 triples
  std::vector<double> cdf(nt);
  std::vector<float4> tv(3 * nt);
  double run = 0.0;
  for (uint64_t i = 0; i < nt; ++i) {
    V3 v[3];
    for (int j = 0; j < 3; ++j) {
      const uint64_t k = tri[3 * i + j];
      if (k >= nv) return set_error(C2B_ERR_INVALID, "triangle %llu references vertex >= %llu", (unsigned long long)i,
                                    (unsigned long long)nv);
      tv[3 * i + j] = make_float4(xyz[3 * k], xyz[3 * k + 1], xyz[3 * k + 2], 0.0f);
      v[j] = V3{(double)xyz[3 * k], (double)xyz[3 * k + 1], (double)xyz[3 * k + 2]};
    }
    const V3 e1{v[1].x - v[0].x, v[1].y - v[0].y, v[1].z - v[0].z}, e2{v[2].x - v[0].x, v[2].y - v[0].y, v[2].z - v[0].z};
    run += mag(cross(e1, e2)) / 2.0;
    cdf[i] = run;
  }
  if (nt == 0 || !(run > 0.0) || !std::isfinite(run))
    return set_error(C2B_ERR_INVALID, "mesh has no triangle of positive area to sample points on");
  // camera centres -> uniform grid with cells of side >= max_dist
  std::vector<double> cen(3 * C);
  double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (uint64_t i = 0; i < C; ++i) {
    const V3 c = camera_center(cams + 15 * i);
    const double a[3] = {c.x, c.y, c.z};
    for (int k = 0; k < 3; ++k) {
      cen[3 * i + k] = a[k];
      if (a[k] < lo[k]) lo[k] = a[k];
      if (a[k] > hi[k]) hi[k] = a[k];
    }
  }
  CamGrid g;
  double h = (max_dist > 0.0 && std::isfinite(max_dist)) ? max_dist : 1.0;
  for (int k = 0; k < 3; ++k) {
    if (!std::isfinite(lo[k]) || !std::isfinite(hi[k])) lo[k] = hi[k] = 0.0;  // NaN / inf centres: one cell
    h = std::max(h, (hi[k] - lo[k]) / 128.0);
  }
  if (!std::isfinite(max_dist) && max_dist > 0.0) h = INFINITY;  // everything is near: a single cell
  uint64_t cells = 1;
  for (int k = 0; k < 3; ++k) {
    g.lo[k] = lo[k];
    g.n[k] = std::isfinite(h) ? (int)std::floor((hi[k] - lo[k]) / h) + 1 : 1;
    cells *= (uint64_t)g.n[k];
  }
  g.inv_h = std::isfinite(h) ? 1.0 / h : 0.0;
  std::vector<uint32_t> cell_start(cells + 1, 0), cell_of(C);
  for (uint64_t i = 0; i < C; ++i) {
    const int cx = cam_grid_coord(g, 0, cen[3 * i]), cy = cam_grid_coord(g, 1, cen[3 * i + 1]),
              cz = cam_grid_coord(g, 2, cen[3 * i + 2]);
    cell_of[i] = ((uint32_t)cz * g.n[1] + cy) * g.n[0] + cx;
    cell_start[cell_of[i] + 1]++;
  }
  for (uint64_t c = 0; c < cells; ++c) cell_start[c + 1] += cell_start[c];
  std::vector<double> cen_sorted(3 * C);
  {
    std::vector<uint32_t> cur(cell_start.begin(), cell_start.end() - 1);
    for (uint64_t i = 0; i < C; ++i) {
      const uint32_t p = cur[cell_of[i]]++;
      for (int k = 0; k < 3; ++k) cen_sorted[3 * p + k] = cen[3 * i + k];
    }
  }
  DevBuf d_tv, d_cdf, d_cs, d_cen, d_cand, d_keep, d_rank, d_out, d_small;
  C2B_TRY(d_tv.ensure(tv.size() * 16));
  C2B_TRY(d_cdf.ensure(nt * 8));
  C2B_TRY(d_cs.ensure((cells + 1) * 4));
  C2B_TRY(d_cen.ensure(C * 24));
  C2B_TRY(d_out.ensure(num_points * 24));
  C2B_TRY(d_small.ensure(64));
  C2B_CUDA(cudaMemcpyAsync(d_tv.p, tv.data(), tv.size() * 16, cudaMemcpyHostToDevice, st));
  C2B_CUDA(cudaMemcpyAsync(d_cdf.p, cdf.data(), nt * 8, cudaMemcpyHostToDevice, st));
  C2B_CUDA(cudaMemcpyAsync(d_cs.p, cell_start.data(), (cells + 1) * 4, cudaMemcpyHostToDevice, st));
  C2B_CUDA(cudaMemcpyAsync(d_cen.p, cen_sorted.data(), C * 24, cudaMemcpyHostToDevice, st));
  SampleArgs a;
  a.tri_v = d_tv.as<float4>();
  a.cdf = d_cdf.as<double>();
  a.nt = nt;
  a.total = run;
  a.g = g;
  a.cell_start = d_cs.as<uint32_t>();
  a.cen = d_cen.as<double>();
  a.max_d2 = max_dist * max_dist;
  a.seed = seed;
  const uint64_t threshold = 10 * num_points;
  uint64_t got = 0, consumed = 0;
  while (got < num_points) {
    const uint64_t want = num_points - got;
    const uint64_t n = std::min<uint64_t>(want + want / 4 + 1024, 1ull << 26);
    C2B_TRY(d_cand.ensure(n * 24));
    C2B_TRY(d_keep.ensure((n + 1) * 4));
    C2B_TRY(d_rank.ensure((n + 1) * 4));
    a.first = consumed;
    a.n = n;
    a.cand = d_cand.as<double>();
    a.keep = d_keep.as<uint32_t>();
    C2B_CUDA(cudaMemsetAsync(d_small.p, 0, 64, st));
    k_sample_points<<<blocks_for(n, 256), 256, 0, st>>>(a);
    C2B_KERNEL_CHECK();
    uint32_t *d_total = d_small.as<uint32_t>() + 4;
    C2B_TRY(exclusive_scan_u32(st, a.keep, d_rank.as<uint32_t>(), n, d_total, ctx->scan_tmp));
    k_sample_compact<<<blocks_for(n, 256), 256, 0, st>>>(a.cand, a.keep, d_rank.as<uint32_t>(), n, got, num_points,
                                                         d_out.as<double>(), d_small.as<unsigned long long>());
    C2B_KERNEL_CHECK();
    unsigned long long h[4];
    C2B_CUDA(cudaMemcpyAsync(h, d_small.p, 32, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaStreamSynchronize(st));
    uint32_t accepted;
    memcpy(&accepted, reinterpret_cast<const char *>(h) + 16, 4);
    if (got + accepted >= num_points) {
      // h[0] = round-local index of the candidate that completed the request
      const uint64_t used = consumed + h[0] + 1;
      if (used - num_points >= threshold)
        return set_error(C2B_ERR_INVALID, "Failed to generate enough points. %llu successes, %llu failures, %llu "
                                          "requested points.", (unsigned long long)num_points,
                         (unsigned long long)(used - num_points), (unsigned long long)num_points);
      got = num_points;
      break;
    }
    got += accepted;
    consumed += n;
    if (consumed - got >= threshold)
      return set_error(C2B_ERR_INVALID, "Failed to generate enough points. %llu successes, %llu failures, %llu "
                                        "requested points.", (unsigned long long)got,
                       (unsigned long long)(consumed - got), (unsigned long long)num_points);
  }
  C2B_CUDA(cudaMemcpyAsync(pts_out, d_out.p, num_points * 24, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  *n_out = num_points;
  return C2B_OK;
}

int c2b_probe_fp64(c2b_ctx *ctx, double *dfma_per_s) {
  if (!ctx || !dfma_per_s) return set_error(C2B_ERR_INVALID, "c2b_probe_fp64: null argument");
  C2B_CUDA(cudaSetDevice(ctx->device));
  C2B_TRY(ctx->misc.ensure(8));
  cudaStream_t st = ctx->stream;
  const int blocks = ctx->sm_count * 8, threads = 256, iters = 4096;
  Event e0, e1;
  C2B_TRY(e0.create());
  C2B_TRY(e1.create());
  float best = 0.0f;
  for (int rep = 0; rep < 4; ++rep) {  // first repetition warms up
    C2B_CUDA(cudaEventRecord(e0, st));
    k_probe_dfma<<<blocks, threads, 0, st>>>(ctx->misc.as<double>(), iters, 1.0000001);
    C2B_KERNEL_CHECK();
    C2B_CUDA(cudaEventRecord(e1, st));
    C2B_CUDA(cudaEventSynchronize(e1));
    float ms = 0.0f;
    C2B_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    if (rep && (best == 0.0f || ms < best)) best = ms;
  }
  *dfma_per_s = (double)blocks * threads * iters * PROBE_CHAINS / (best * 1e-3);
  return C2B_OK;
}

int c2b_mean_std(c2b_ctx *ctx, const double *cams, uint64_t C, const double *pts, uint64_t P,
                 double mean[3], double sd[3]) {
  if (!ctx || (C && !cams) || (P && !pts) || !mean || !sd)
    return set_error(C2B_ERR_INVALID, "c2b_mean_std: null argument");
  if (C + P == 0) return set_error(C2B_ERR_EMPTY, "mean/std of an empty problem");
  C2B_CUDA(cudaSetDevice(ctx->device));
  NoiseView v;
  C2B_TRY(noise_upload(ctx, v, cams, C, pts, P));
  return device_stats(ctx, v, mean, sd, false);
}

// ---- BAProblem::cull: LCC + remove_singletons to a fixed point (c2b_graph_cull.cuh) -------------------------
static int cull_limits(uint64_t C, uint64_t P, uint64_t O, const char *who) {
  if (C + P >= 0xffffffffull)
    return set_error(C2B_ERR_INVALID, "%s: %llu cameras + %llu points exceed the 32-bit entity ids (C + P < 2^32 - 1)",
                     who, (unsigned long long)C, (unsigned long long)P);
  if (O >= 0xffffffffull)
    return set_error(C2B_ERR_INVALID, "%s: %llu observations exceed the 32-bit compaction (O < 2^32 - 1)", who,
                     (unsigned long long)O);
  return C2B_OK;
}

int c2b_cull_problem(c2b_ctx *ctx, double *cams, uint64_t C, double *pts, uint64_t P, uint64_t *offsets,
                     uint32_t *point_idx, double *uv, c2b_cull_stats *out) {
  if (!ctx || !offsets || (C && !cams) || (P && !pts)) return set_error(C2B_ERR_INVALID, "c2b_cull_problem: null argument");
  const uint64_t O = offsets[C];
  if (O && (!point_idx || !uv)) return set_error(C2B_ERR_INVALID, "c2b_cull_problem: null observation array");
  C2B_TRY(cull_limits(C, P, O, "c2b_cull_problem"));
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  PruneSet sets[2];
  for (int i = 0; i < 2; ++i) sets[i] = PruneSet{&ctx->pr_cams[i], &ctx->pr_pts[i], &ctx->pr_off[i], &ctx->pr_idx[i], &ctx->pr_uv[i]};
  C2B_TRY(ctx->pr_cams[0].ensure(std::max<uint64_t>(C, 1) * 120));
  C2B_TRY(ctx->pr_pts[0].ensure(std::max<uint64_t>(P, 1) * 24));
  C2B_TRY(ctx->pr_off[0].ensure((C + 1) * 8));
  C2B_TRY(ctx->pr_idx[0].ensure(std::max<uint64_t>(O, 1) * 4));
  C2B_TRY(ctx->pr_uv[0].ensure(std::max<uint64_t>(O, 1) * 16));
  C2B_TRY(ctx->pr_small.ensure(64));
  C2B_TRY(ctx->h_small.ensure(256));
  Event ev[4];  // timing
  for (auto &e : ev) C2B_TRY(e.create());
  int rc = [&]() -> int {
    C2B_CUDA(cudaEventRecord(ev[0], st));
    if (C) C2B_TRY(copy_in(ctx, ctx->pr_cams[0].p, cams, C * 120, cudaMemcpyHostToDevice));
    if (P) C2B_TRY(copy_in(ctx, ctx->pr_pts[0].p, pts, P * 24, cudaMemcpyHostToDevice));
    C2B_TRY(copy_in(ctx, ctx->pr_off[0].p, offsets, (C + 1) * 8, cudaMemcpyHostToDevice));
    if (O) {
      C2B_TRY(copy_in(ctx, ctx->pr_idx[0].p, point_idx, O * 4, cudaMemcpyHostToDevice));
      C2B_TRY(copy_in(ctx, ctx->pr_uv[0].p, uv, O * 16, cudaMemcpyHostToDevice));
    }
    // from_visibility's asserts, on the device: offsets start at 0 and do not decrease, indices < P
    uint32_t *flag = ctx->pr_small.as<uint32_t>() + 8;
    C2B_CUDA(cudaMemsetAsync(flag, 0, 4, st));
    const uint64_t nv = std::max<uint64_t>(std::max(C, O), 1);
    k_prune_validate<<<(unsigned)std::min<uint64_t>(prune_blocks(nv), (uint64_t)ctx->sm_count * 8), PR_THREADS, 0, st>>>(
        ctx->pr_off[0].as<uint64_t>(), C, ctx->pr_idx[0].as<uint32_t>(), O, P, flag);
    C2B_KERNEL_CHECK();
    C2B_CUDA(cudaMemcpyAsync(ctx->h_small.p, flag, 4, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaEventRecord(ev[1], st));
    C2B_CUDA(cudaStreamSynchronize(st));
    const uint32_t bad = *ctx->h_small.as<uint32_t>();
    if (bad & 1u) return set_error(C2B_ERR_INVALID, "c2b_cull_problem: offsets[0] != 0 or the CSR offsets decrease");
    if (bad & 2u) return set_error(C2B_ERR_INVALID, "c2b_cull_problem: an observation references a point >= %llu",
                                   (unsigned long long)P);
    int cur = 0;
    uint64_t c = C, p = P, o = O;
    uint32_t it = 0;
    C2B_TRY(prune_fixed_point(ctx, sets, &cur, &c, &p, &o, &it));
    C2B_CUDA(cudaEventRecord(ev[2], st));
    const PruneSet &r = sets[cur];
    if (c) C2B_CUDA(cudaMemcpyAsync(cams, r.cams->p, c * 120, cudaMemcpyDeviceToHost, st));
    if (p) C2B_CUDA(cudaMemcpyAsync(pts, r.pts->p, p * 24, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaMemcpyAsync(offsets, r.off->p, (c + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (o) {
      C2B_CUDA(cudaMemcpyAsync(point_idx, r.idx->p, o * 4, cudaMemcpyDeviceToHost, st));
      C2B_CUDA(cudaMemcpyAsync(uv, r.uv->p, o * 16, cudaMemcpyDeviceToHost, st));
    }
    C2B_CUDA(cudaEventRecord(ev[3], st));
    C2B_CUDA(cudaStreamSynchronize(st));
    if (out) {
      memset(out, 0, sizeof *out);
      out->n_cameras = c;
      out->n_points = p;
      out->n_obs = o;
      out->iterations = it;
      cudaEventElapsedTime(&out->ms_h2d, ev[0], ev[1]);
      cudaEventElapsedTime(&out->ms_compute, ev[1], ev[2]);
      cudaEventElapsedTime(&out->ms_d2h, ev[2], ev[3]);
    }
    return C2B_OK;
  }();
  if (rc != C2B_OK) cudaStreamSynchronize(st);
  return rc;
}

int c2b_cull_problem_resident(c2b_ctx *ctx, c2b_cull_stats *out) {
  if (!ctx) return set_error(C2B_ERR_INVALID, "c2b_cull_problem_resident: null ctx");
  CtxExtra *x = ctx->extra.get();
  if (x->host_call_last)
    return set_error(C2B_ERR_INVALID, "c2b_cull_problem_resident: the resident CSR is the last camera batch of the "
                                      "host-buffer c2b_visibility_graph, not the graph of an uploaded problem; run "
                                      "c2b_visibility_graph_resident first");
  if (!x->have_result || !x->have_points || !x->have_cameras)
    return set_error(C2B_ERR_INVALID, "c2b_cull_problem_resident: no resident result (upload cameras and points, "
                                      "then c2b_visibility_graph_resident)");
  uint64_t C = ctx->out_C, P = ctx->P, O = ctx->out_O;
  C2B_TRY(cull_limits(C, P, O, "c2b_cull_problem_resident"));
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int sel = ctx->out_sel;
  // set 0: the resident problem; set 1: the other half of the double-buffered CSR and spare camera / point arrays
  PruneSet sets[2] = {{&ctx->cams, &ctx->pts_aos, &ctx->out_offsets[sel], &ctx->out_idx[sel], &ctx->out_uv[sel]},
                      {&ctx->pr_cams[1], &ctx->pr_pts[1], &ctx->out_offsets[sel ^ 1], &ctx->out_idx[sel ^ 1],
                       &ctx->out_uv[sel ^ 1]}};
  Event ev[4];  // timing
  for (auto &e : ev) C2B_TRY(e.create());
  int cur = 0;
  uint32_t it = 0;
  int rc = [&]() -> int {
    C2B_CUDA(cudaEventRecord(ev[0], st));
    C2B_TRY(prune_fixed_point(ctx, sets, &cur, &C, &P, &O, &it));
    C2B_CUDA(cudaEventRecord(ev[1], st));
    return C2B_OK;
  }();
  if (rc == C2B_OK && cur == 1) {
    std::swap(ctx->cams, ctx->pr_cams[1]);
    std::swap(ctx->pts_aos, ctx->pr_pts[1]);
    ctx->out_sel = sel ^ 1;
  }
  if (rc != C2B_OK) {
    // the resident arrays may be half rewritten: nothing of the resident problem is usable any more
    cudaStreamSynchronize(st);
    x->have_result = x->have_cameras = x->have_points = false;
    return rc;
  }
  // the culled problem becomes the resident one: camera centres, SoA points, bounds; the point grid is stale
  ctx->C = C;
  ctx->out_C = C;
  ctx->out_O = O;
  if (C) {
    double *cx = ctx->cam_center.as<double>();
    k_cam_prep<<<blocks_for(C, 128), 128, 0, st>>>(ctx->cams.as<double>(), C, cx, cx + C, cx + 2 * C);
    C2B_KERNEL_CHECK();
  }
  C2B_TRY(c2b_points_commit(ctx, P));
  x->have_result = true;  // the CSR is the graph of the culled problem
  C2B_CUDA(cudaStreamSynchronize(st));
  if (out) {
    memset(out, 0, sizeof *out);
    out->n_cameras = C;
    out->n_points = P;
    out->n_obs = O;
    out->iterations = it;
    cudaEventElapsedTime(&out->ms_compute, ev[0], ev[1]);
  }
  return C2B_OK;
}

// ---- noise::add_incorrect_correspondences (c2b_mismatch.cuh) -------------------------------------------------------
// the message of a failed selection: camera, observation within it, CSR index, and the reference's panic text
static int mismatch_error(const char *who, const uint64_t *offsets, uint64_t C, unsigned long long err) {
  const uint64_t o = err >> 1;
  const uint64_t c = (uint64_t)(std::upper_bound(offsets, offsets + C + 1, o) - offsets) - 1;
  return set_error(C2B_ERR_INVALID, "%s: camera %llu, observation %llu (CSR index %llu): called `Result::unwrap()` on an "
                                    "`Err` value: %s",
                   who, (unsigned long long)c, (unsigned long long)(o - offsets[c]), (unsigned long long)o,
                   (err & 1) == MM_NEGATIVE_WEIGHT ? "NegativeWeight" : "AllWeightsZero");
}

int c2b_add_incorrect_correspondences(c2b_ctx *ctx, const uint64_t *offsets, uint64_t C, uint32_t *point_idx,
                                      const double *uv, double mismatch_chance, uint64_t seed,
                                      c2b_mismatch_stats *out) {
  static const char *who = "c2b_add_incorrect_correspondences";
  if (!ctx || !offsets) return set_error(C2B_ERR_INVALID, "%s: null argument", who);
  const uint64_t O = offsets[C];
  if (O && (!point_idx || !uv)) return set_error(C2B_ERR_INVALID, "%s: null observation array", who);
  C2B_TRY(cull_limits(C, 0, O, who));
  C2B_CUDA(cudaSetDevice(ctx->device));
  CtxExtra *x = ctx->extra.get();
  cudaStream_t st = ctx->stream;
  // the host-array cull's set 0: never the resident problem
  C2B_TRY(ctx->pr_off[0].ensure((C + 1) * 8));
  C2B_TRY(ctx->pr_idx[0].ensure(std::max<uint64_t>(O, 1) * 4));
  C2B_TRY(ctx->pr_uv[0].ensure(std::max<uint64_t>(O, 1) * 16));
  C2B_TRY(ctx->pr_small.ensure(64));
  C2B_TRY(ctx->h_small.ensure(256));
  Event ev[4];  // timing
  for (auto &e : ev) C2B_TRY(e.create());
  int rc = [&]() -> int {
    C2B_CUDA(cudaEventRecord(ev[0], st));
    C2B_TRY(copy_in(ctx, ctx->pr_off[0].p, offsets, (C + 1) * 8, cudaMemcpyHostToDevice));
    if (O) {
      C2B_TRY(copy_in(ctx, ctx->pr_idx[0].p, point_idx, O * 4, cudaMemcpyHostToDevice));
      C2B_TRY(copy_in(ctx, ctx->pr_uv[0].p, uv, O * 16, cudaMemcpyHostToDevice));
    }
    // offsets start at 0 and do not decrease; there is no point count, so no u32 index is out of range
    uint32_t *flag = ctx->pr_small.as<uint32_t>() + 8;
    C2B_CUDA(cudaMemsetAsync(flag, 0, 4, st));
    const uint64_t nv = std::max<uint64_t>(std::max(C, O), 1);
    k_prune_validate<<<(unsigned)std::min<uint64_t>(prune_blocks(nv), (uint64_t)ctx->sm_count * 8), PR_THREADS, 0, st>>>(
        ctx->pr_off[0].as<uint64_t>(), C, ctx->pr_idx[0].as<uint32_t>(), O, 1ull << 32, flag);
    C2B_KERNEL_CHECK();
    C2B_CUDA(cudaMemcpyAsync(ctx->h_small.p, flag, 4, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaEventRecord(ev[1], st));
    C2B_CUDA(cudaStreamSynchronize(st));
    if (*ctx->h_small.as<uint32_t>() & 1u)
      return set_error(C2B_ERR_INVALID, "%s: offsets[0] != 0 or the CSR offsets decrease", who);
    uint64_t ns = 0, nw = 0;
    unsigned long long err = MM_NO_ERROR;
    C2B_TRY(mismatch_pass(ctx, MismatchBufs{&x->mm_cnt, &x->mm_sel, &x->mm_small}, ctx->pr_off[0].as<uint64_t>(), C,
                          ctx->pr_idx[0].as<uint32_t>(), ctx->pr_uv[0].as<double2>(), mismatch_chance, seed, &ns, &nw,
                          &err));
    if (err != MM_NO_ERROR) return mismatch_error(who, offsets, C, err);
    C2B_CUDA(cudaEventRecord(ev[2], st));
    if (O) C2B_CUDA(cudaMemcpyAsync(point_idx, ctx->pr_idx[0].p, O * 4, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaEventRecord(ev[3], st));
    C2B_CUDA(cudaStreamSynchronize(st));
    if (out) {
      memset(out, 0, sizeof *out);
      out->n_selected = ns;
      out->n_swapped = nw;
      cudaEventElapsedTime(&out->ms_h2d, ev[0], ev[1]);
      cudaEventElapsedTime(&out->ms_compute, ev[1], ev[2]);
      cudaEventElapsedTime(&out->ms_d2h, ev[2], ev[3]);
    }
    return C2B_OK;
  }();
  if (rc != C2B_OK) cudaStreamSynchronize(st);
  return rc;
}

int c2b_add_incorrect_correspondences_resident(c2b_ctx *ctx, double mismatch_chance, uint64_t seed,
                                               c2b_mismatch_stats *out) {
  static const char *who = "c2b_add_incorrect_correspondences_resident";
  if (!ctx) return set_error(C2B_ERR_INVALID, "%s: null ctx", who);
  CtxExtra *x = ctx->extra.get();
  if (x->host_call_last)
    return set_error(C2B_ERR_INVALID, "%s: the resident CSR is the last camera batch of the host-buffer "
                                      "c2b_visibility_graph, not the graph of an uploaded problem; run "
                                      "c2b_visibility_graph_resident first", who);
  if (!x->have_result || !x->have_points || !x->have_cameras)
    return set_error(C2B_ERR_INVALID, "%s: no resident result (upload cameras and points, then "
                                      "c2b_visibility_graph_resident)", who);
  const uint64_t C = ctx->out_C, O = ctx->out_O;
  C2B_TRY(cull_limits(C, 0, O, who));
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int sel = ctx->out_sel;
  Event ev[2];  // timing
  for (auto &e : ev) C2B_TRY(e.create());
  uint64_t ns = 0, nw = 0;
  unsigned long long err = MM_NO_ERROR;
  int rc = [&]() -> int {
    C2B_CUDA(cudaEventRecord(ev[0], st));
    C2B_TRY(mismatch_pass(ctx, MismatchBufs{&x->mm_cnt, &x->mm_sel, &x->mm_small}, ctx->out_offsets[sel].as<uint64_t>(),
                          C, ctx->out_idx[sel].as<uint32_t>(), ctx->out_uv[sel].as<double2>(), mismatch_chance, seed,
                          &ns, &nw, &err));
    C2B_CUDA(cudaEventRecord(ev[1], st));
    return C2B_OK;
  }();
  if (rc != C2B_OK) {
    // a failure of the library, not of the input: the point indices may be half permuted
    cudaStreamSynchronize(st);
    x->have_result = false;
    return rc;
  }
  if (err != MM_NO_ERROR) {
    // the resident problem is unchanged; the offsets name the camera in the message
    std::vector<uint64_t> offsets(C + 1);
    C2B_CUDA(cudaMemcpyAsync(offsets.data(), ctx->out_offsets[sel].p, (C + 1) * 8, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaStreamSynchronize(st));
    return mismatch_error(who, offsets.data(), C, err);
  }
  C2B_CUDA(cudaStreamSynchronize(st));
  if (out) {
    memset(out, 0, sizeof *out);
    out->n_selected = ns;
    out->n_swapped = nw;
    cudaEventElapsedTime(&out->ms_compute, ev[0], ev[1]);
  }
  return C2B_OK;
}


// ---- BAL files (c2b_bal.cuh) ----------------------------------------------------------------------------------
namespace {
constexpr int BAL_RING = 3;                 // pinned chunk slots: D2H of chunk k while chunk k-1 is written
constexpr uint32_t BAL_WINDOW = 1u << 20;   // lines per length pass: 2^20 lines of <= 2952 bytes keep the u32 scan exact

// the camera 9-vectors of C records (host memory) -> x->bal_vecs
int bal_upload_vecs(c2b_ctx *ctx, CtxExtra *x, const double *cams, uint64_t C) {
  C2B_TRY(x->bal_vecs.ensure(std::max<uint64_t>(C, 1) * 72));
  if (!C) return C2B_OK;
  std::vector<double> vecs(9 * C);
  for (uint64_t c = 0; c < C; ++c) c2b_camera_to_vec(cams + 15 * c, &vecs[9 * c]);
  C2B_CUDA(cudaMemcpyAsync(x->bal_vecs.p, vecs.data(), C * 72, cudaMemcpyHostToDevice, ctx->stream));
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));  // vecs is freed on return
  return C2B_OK;
}

// Encodes the problem `v` (device arrays) chunk by chunk and writes it to `path`.  Chunk k: the encoding kernels on
// the ctx stream into device buffer k % 2, its copy on the copy stream into ring slot k % 3, then write(2) on a
// writer thread; the host waits only for the chunk's line count (text) and for a free ring slot.
int bal_stream(c2b_ctx *ctx, const char *path, int format, const BalView &v, c2b_bal_stats *out) {
  CtxExtra *x = ctx->extra.get();
  const uint64_t B = x->tun.bal_chunk_bytes;
  const bool text = format == C2B_BAL_TEXT;
  cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
  C2B_TRY(x->bal_out[0].ensure(B));
  C2B_TRY(x->bal_out[1].ensure(B));
  x->bal_ring.node = ctx->numa_node;
  C2B_TRY(x->bal_ring.ensure(BAL_RING * B));
  if (text) {
    C2B_TRY(x->bal_scan.ensure((size_t)(BAL_WINDOW + 1) * 4));
    C2B_TRY(ctx->h_small.ensure(256));
  }
  Event ev[BAL_RING][4];  // per ring slot: encode start / end (ctx stream), copy start / end (copy stream)
  for (auto &slot : ev)
    for (auto &e : slot) C2B_TRY(e.create());
  const int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0666);
  if (fd < 0) return set_error(C2B_ERR_IO, "cannot create %s: %s", path, strerror(errno));
  struct stat sb;
  const bool regular = fstat(fd, &sb) == 0 && S_ISREG(sb.st_mode);  // /dev/null and pipes are never removed

  struct Job {
    int slot;
    uint64_t bytes;
  };
  std::mutex mu;
  std::condition_variable cv;
  std::deque<Job> jobs;
  bool quit = false;
  uint64_t chunks_done = 0;
  int io_errno = 0;
  cudaError_t cuda_err = cudaSuccess;
  float ms_encode = 0, ms_d2h = 0;
  double ms_write = 0;
  char *ring = x->bal_ring.as<char>();
  const int device = ctx->device;
  std::thread writer([&]() {
    cudaError_t e = cudaSetDevice(device);
    for (;;) {
      Job j;
      {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return !jobs.empty() || quit; });
        if (jobs.empty()) break;
        j = jobs.front();
        jobs.pop_front();
      }
      if (e == cudaSuccess) e = cudaEventSynchronize(ev[j.slot][3]);
      float a = 0, b = 0;
      int err = 0;
      double ms = 0;
      if (e == cudaSuccess) {
        cudaEventElapsedTime(&a, ev[j.slot][0], ev[j.slot][1]);
        cudaEventElapsedTime(&b, ev[j.slot][2], ev[j.slot][3]);
        const auto t0 = std::chrono::steady_clock::now();
        const char *p = ring + (size_t)j.slot * B;
        for (uint64_t left = j.bytes; left && !io_errno;) {
          const ssize_t r = ::write(fd, p, left);
          if (r < 0 && errno == EINTR) continue;
          if (r <= 0) {
            err = r < 0 ? errno : EIO;
            break;
          }
          p += r;
          left -= (uint64_t)r;
        }
        ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      }
      {
        std::lock_guard<std::mutex> lk(mu);
        ms_encode += a;
        ms_d2h += b;
        ms_write += ms;
        if (err && !io_errno) io_errno = err;
        if (e != cudaSuccess) cuda_err = e;
        ++chunks_done;
      }
      cv.notify_all();
    }
  });

  uint64_t chunks = 0, bytes = 0;
  int rc = [&]() -> int {
    const uint64_t units = text ? 1 + v.O + v.C + v.P : 3 + v.C + 3 * v.O + 9 * v.C + 3 * v.P;  // lines or words
    uint32_t window = (uint32_t)std::min<uint64_t>(BAL_WINDOW, std::max<uint64_t>(1024, B / 64));
    uint32_t *scan = x->bal_scan.as<uint32_t>();
    const uint32_t *res = ctx->h_small.as<uint32_t>();
    for (uint64_t pos = 0; pos < units; ++chunks) {
      const int slot = (int)(chunks % BAL_RING);
      char *dbuf = x->bal_out[chunks % 2].as<char>();
      {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return chunks_done + BAL_RING > chunks; });  // the slot's previous chunk is on disk
        if (io_errno) return set_error(C2B_ERR_IO, "write to %s failed: %s", path, strerror(io_errno));
        if (cuda_err != cudaSuccess) return set_error(C2B_ERR_CUDA, "BAL chunk copy: %s", cudaGetErrorString(cuda_err));
      }
      // the device buffer's previous chunk (k - 2) has been copied out
      if (chunks >= 2) C2B_CUDA(cudaStreamWaitEvent(st, ev[(chunks - 2) % BAL_RING][3], 0));
      C2B_CUDA(cudaEventRecord(ev[slot][0], st));
      uint64_t n_bytes;
      if (text) {
        const uint32_t n = (uint32_t)std::min<uint64_t>(window, units - pos);
        k_bal_text_len<<<blocks_for(n, BAL_THREADS), BAL_THREADS, 0, st>>>(v, pos, n, scan);
        C2B_KERNEL_CHECK();
        C2B_TRY(exclusive_scan_u32(st, scan, scan, n, scan + BAL_WINDOW, ctx->scan_tmp));
        k_bal_text_cut<<<1, 1, 0, st>>>(scan, scan + BAL_WINDOW, n, (uint32_t)B, ctx->h_small.as<uint32_t>());
        C2B_KERNEL_CHECK();
        C2B_CUDA(cudaStreamSynchronize(st));
        const uint32_t k = res[0];
        n_bytes = res[1];
        k_bal_text_write<<<blocks_for(k, BAL_THREADS), BAL_THREADS, 0, st>>>(v, pos, k, scan, dbuf);
        C2B_KERNEL_CHECK();
        pos += k;
        // next window: the lines that fitted, and some more; twice as many when all of them fitted
        window = (uint32_t)std::min<uint64_t>(BAL_WINDOW, k == n ? 2ull * n : k + k / 8 + 64);
      } else {
        const uint64_t n = std::min<uint64_t>(B / 8, units - pos);
        k_bal_binary<<<(unsigned)((n + BAL_THREADS - 1) / BAL_THREADS), BAL_THREADS, 0, st>>>(
            v, pos, n, reinterpret_cast<uint64_t *>(dbuf));
        C2B_KERNEL_CHECK();
        n_bytes = 8 * n;
        pos += n;
      }
      C2B_CUDA(cudaEventRecord(ev[slot][1], st));
      C2B_CUDA(cudaStreamWaitEvent(cp, ev[slot][1], 0));
      C2B_CUDA(cudaEventRecord(ev[slot][2], cp));
      C2B_CUDA(cudaMemcpyAsync(ring + (size_t)slot * B, dbuf, n_bytes, cudaMemcpyDeviceToHost, cp));
      C2B_CUDA(cudaEventRecord(ev[slot][3], cp));
      {
        std::lock_guard<std::mutex> lk(mu);
        jobs.push_back(Job{slot, n_bytes});
      }
      cv.notify_all();
      bytes += n_bytes;
    }
    return C2B_OK;
  }();
  {
    std::lock_guard<std::mutex> lk(mu);
    quit = true;
  }
  cv.notify_all();
  writer.join();
  if (rc == C2B_OK && io_errno) rc = set_error(C2B_ERR_IO, "write to %s failed: %s", path, strerror(io_errno));
  if (rc == C2B_OK && cuda_err != cudaSuccess)
    rc = set_error(C2B_ERR_CUDA, "BAL chunk copy: %s", cudaGetErrorString(cuda_err));
  if (close(fd) != 0 && rc == C2B_OK) rc = set_error(C2B_ERR_IO, "closing %s failed: %s", path, strerror(errno));
  if (rc != C2B_OK) {
    cudaStreamSynchronize(st);
    cudaStreamSynchronize(cp);
    if (regular) unlink(path);  // no truncated file behind a failed call
    return rc;
  }
  if (out) {
    memset(out, 0, sizeof *out);
    out->bytes = bytes;
    out->chunks = chunks;
    out->ms_encode = ms_encode;
    out->ms_d2h = ms_d2h;
    out->ms_write = (float)ms_write;
  }
  return C2B_OK;
}
}  // namespace

int c2b_write_bal(c2b_ctx *ctx, const char *path, int format, const double *cams, uint64_t C, const double *pts,
                  uint64_t P, const uint64_t *offsets, const uint32_t *point_idx, const double *uv,
                  c2b_bal_stats *out) {
  if (!ctx || !path || !offsets || (C && !cams) || (P && !pts)) return set_error(C2B_ERR_INVALID, "c2b_write_bal: null argument");
  if (format != C2B_BAL_TEXT && format != C2B_BAL_BINARY) return set_error(C2B_ERR_INVALID, "c2b_write_bal: unknown format %d", format);
  const uint64_t O = offsets[C];
  if (O && (!point_idx || !uv)) return set_error(C2B_ERR_INVALID, "c2b_write_bal: null observation array");
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  CtxExtra *x = ctx->extra.get();
  // the cull's host-entry buffers (set 0): never the resident problem
  C2B_TRY(ctx->pr_pts[0].ensure(std::max<uint64_t>(P, 1) * 24));
  C2B_TRY(ctx->pr_off[0].ensure((C + 1) * 8));
  C2B_TRY(ctx->pr_idx[0].ensure(std::max<uint64_t>(O, 1) * 4));
  C2B_TRY(ctx->pr_uv[0].ensure(std::max<uint64_t>(O, 1) * 16));
  C2B_TRY(ctx->pr_small.ensure(64));
  C2B_TRY(ctx->h_small.ensure(256));
  int rc = [&]() -> int {
    if (P) C2B_TRY(copy_in(ctx, ctx->pr_pts[0].p, pts, P * 24, cudaMemcpyHostToDevice));
    C2B_TRY(copy_in(ctx, ctx->pr_off[0].p, offsets, (C + 1) * 8, cudaMemcpyHostToDevice));
    if (O) {
      C2B_TRY(copy_in(ctx, ctx->pr_idx[0].p, point_idx, O * 4, cudaMemcpyHostToDevice));
      C2B_TRY(copy_in(ctx, ctx->pr_uv[0].p, uv, O * 16, cudaMemcpyHostToDevice));
    }
    // the checks of c2b_cull_problem (from_visibility's asserts), before the file exists
    uint32_t *flag = ctx->pr_small.as<uint32_t>() + 8;
    C2B_CUDA(cudaMemsetAsync(flag, 0, 4, st));
    const uint64_t nv = std::max<uint64_t>(std::max(C, O), 1);
    k_prune_validate<<<(unsigned)std::min<uint64_t>(prune_blocks(nv), (uint64_t)ctx->sm_count * 8), PR_THREADS, 0, st>>>(
        ctx->pr_off[0].as<uint64_t>(), C, ctx->pr_idx[0].as<uint32_t>(), O, P, flag);
    C2B_KERNEL_CHECK();
    C2B_CUDA(cudaMemcpyAsync(ctx->h_small.p, flag, 4, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaStreamSynchronize(st));
    const uint32_t bad = *ctx->h_small.as<uint32_t>();
    if (bad & 1u) return set_error(C2B_ERR_INVALID, "c2b_write_bal: offsets[0] != 0 or the CSR offsets decrease");
    if (bad & 2u) return set_error(C2B_ERR_INVALID, "c2b_write_bal: an observation references a point >= %llu",
                                   (unsigned long long)P);
    C2B_TRY(bal_upload_vecs(ctx, x, cams, C));
    const BalView v{x->bal_vecs.as<double>(), ctx->pr_pts[0].as<double>(), ctx->pr_off[0].as<uint64_t>(),
                    ctx->pr_idx[0].as<uint32_t>(), ctx->pr_uv[0].as<double>(), C, P, O};
    return bal_stream(ctx, path, format, v, out);
  }();
  if (rc != C2B_OK) cudaStreamSynchronize(st);
  return rc;
}

int c2b_write_bal_resident(c2b_ctx *ctx, const char *path, int format, c2b_bal_stats *out) {
  if (!ctx || !path) return set_error(C2B_ERR_INVALID, "c2b_write_bal_resident: null argument");
  if (format != C2B_BAL_TEXT && format != C2B_BAL_BINARY)
    return set_error(C2B_ERR_INVALID, "c2b_write_bal_resident: unknown format %d", format);
  CtxExtra *x = ctx->extra.get();
  if (x->host_call_last)
    return set_error(C2B_ERR_INVALID, "c2b_write_bal_resident: the resident CSR is the last camera batch of the "
                                      "host-buffer c2b_visibility_graph, not the graph of an uploaded problem; run "
                                      "c2b_visibility_graph_resident first");
  if (!x->have_result || !x->have_points || !x->have_cameras)
    return set_error(C2B_ERR_INVALID, "c2b_write_bal_resident: no resident result (upload cameras and points, "
                                      "then c2b_visibility_graph_resident)");
  C2B_CUDA(cudaSetDevice(ctx->device));
  const uint64_t C = ctx->out_C, P = ctx->P, O = ctx->out_O;
  const int sel = ctx->out_sel;
  std::vector<double> cams(15 * C);
  if (C) C2B_CUDA(cudaMemcpyAsync(cams.data(), ctx->cams.p, C * 120, cudaMemcpyDeviceToHost, ctx->stream));
  C2B_CUDA(cudaStreamSynchronize(ctx->stream));
  C2B_TRY(bal_upload_vecs(ctx, x, cams.data(), C));
  const BalView v{x->bal_vecs.as<double>(), ctx->pts_aos.as<double>(), ctx->out_offsets[sel].as<uint64_t>(),
                  ctx->out_idx[sel].as<uint32_t>(), ctx->out_uv[sel].as<double>(), C, P, O};
  return bal_stream(ctx, path, format, v, out);
}

// ---- reading BAL files (c2b_bal_read.cuh) ----------------------------------------------------------------------------
namespace {
constexpr unsigned long long BAL_NO_ERR = ~0ull;

// pread until `want` bytes or the end of the file; the bytes read, or -1 with errno
int64_t bal_pread(int fd, char *dst, uint64_t want, uint64_t off, double &ms) {
  const auto t0 = std::chrono::steady_clock::now();
  uint64_t got = 0;
  while (got < want) {
    const ssize_t r = ::pread(fd, dst + got, want - got, (off_t)(off + got));
    if (r < 0 && errno == EINTR) continue;
    if (r < 0) return -1;
    if (r == 0) break;
    got += (uint64_t)r;
  }
  ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return (int64_t)got;
}

struct BalReadState {
  c2b_ctx *ctx;
  CtxExtra *x;
  const char *path;
  int fd;
  uint64_t size, B;
  uint64_t C = 0, P = 0, O = 0;
  Event ev[BAL_RING][4] = {};  // per ring slot: H2D start / end (copy stream), parse start / end (ctx stream)
  double ms_read = 0;
  float ms_h2d = 0, ms_parse = 0;
  uint64_t chunks = 0, bytes = 0, slow = 0;
  uint32_t regrouped = 0;
  unsigned long long *d_err = nullptr;  // [0] malformed token, [1] index out of range; then u64 base, u32 total, ...
  double *vecs = nullptr, *pts = nullptr;
  // the device times of the chunk in ring slot `slot` (its parse has finished)
  void add_times(int slot) {
    float a = 0, b = 0;
    cudaEventElapsedTime(&a, ev[slot][0], ev[slot][1]);
    cudaEventElapsedTime(&b, ev[slot][2], ev[slot][3]);
    ms_h2d += a;
    ms_parse += b;
  }
};

// C, P and O known: checks the limits and sizes the resident arrays (the old resident problem is gone from here on)
int bal_read_alloc(BalReadState &s) {
  c2b_ctx *ctx = s.ctx;
  CtxExtra *x = s.x;
  if (s.C >= 0xffffffffull || s.P >= 0xffffffffull || s.O >= 0xffffffffull)
    return set_error(C2B_ERR_INVALID, "c2b_read_bal_resident: %s: C = %llu, P = %llu, O = %llu; each must be below "
                     "2^32 - 1", s.path, (unsigned long long)s.C, (unsigned long long)s.P, (unsigned long long)s.O);
  const int sel = ctx->out_sel;
  C2B_TRY(ctx->out_offsets[sel].ensure((s.C + 1) * 8));
  C2B_TRY(ctx->out_idx[sel].ensure(std::max<uint64_t>(s.O, 1) * 4));
  C2B_TRY(ctx->out_uv[sel].ensure(std::max<uint64_t>(s.O, 1) * 16));
  C2B_TRY(x->bal_vecs.ensure(std::max<uint64_t>(s.C, 1) * 72));
  C2B_TRY(c2b_points_device_buffer(ctx, s.P, &s.pts));
  s.vecs = x->bal_vecs.as<double>();
  C2B_TRY(x->bal_out[0].ensure(s.B));
  C2B_TRY(x->bal_out[1].ensure(s.B));
  C2B_TRY(x->bal_small.ensure(64));
  s.d_err = x->bal_small.as<unsigned long long>();
  C2B_CUDA(cudaMemsetAsync(s.d_err, 0xff, 16, ctx->stream));
  C2B_CUDA(cudaMemsetAsync(s.d_err + 2, 0, 48, ctx->stream));
  return C2B_OK;
}

// the observations in file order (idx / uv of set `sel`, cam_of) -> the CSR grouped by camera, in file order within
// a camera: offsets from a per-camera count and scan; a stable sort by camera and a gather when the file was not
// already camera-major
int bal_group(BalReadState &s) {
  c2b_ctx *ctx = s.ctx;
  CtxExtra *x = s.x;
  cudaStream_t st = ctx->stream;
  const uint64_t C = s.C, O = s.O;
  const int sel = ctx->out_sel;
  C2B_TRY(x->bal_cnt.ensure((C + 1) * 4));
  uint32_t *cnt = x->bal_cnt.as<uint32_t>();
  uint32_t *unordered = reinterpret_cast<uint32_t *>(s.d_err + 4);
  C2B_CUDA(cudaMemsetAsync(cnt, 0, (C + 1) * 4, st));
  if (O) {
    k_bal_cam_count<<<blocks_for(O, BALR_THREADS), BALR_THREADS, 0, st>>>(x->bal_cam.as<uint32_t>(), O, cnt, unordered);
    C2B_KERNEL_CHECK();
  }
  C2B_CUDA(cudaMemcpyAsync(ctx->h_small.p, unordered, 4, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  s.regrouped = *ctx->h_small.as<uint32_t>() ? 1u : 0u;
  const int fs = s.regrouped ? sel ^ 1 : sel;
  C2B_TRY(ctx->out_offsets[fs].ensure((C + 1) * 8));
  C2B_TRY(exclusive_scan_u32(st, cnt, cnt, C, nullptr, ctx->scan_tmp));
  k_bal_offsets<<<blocks_for(C + 1, BALR_THREADS), BALR_THREADS, 0, st>>>(cnt, C, O, ctx->out_offsets[fs].as<uint64_t>());
  C2B_KERNEL_CHECK();
  if (s.regrouped) {
    C2B_TRY(ctx->out_idx[fs].ensure(O * 4));
    C2B_TRY(ctx->out_uv[fs].ensure(O * 16));
    for (int i = 0; i < 2; ++i) {
      C2B_TRY(ctx->sort_keys[i].ensure(O * 8));
      C2B_TRY(ctx->sort_vals[i].ensure(O * 4));
    }
    uint64_t *keys[2] = {ctx->sort_keys[0].as<uint64_t>(), ctx->sort_keys[1].as<uint64_t>()};
    uint32_t *vals[2] = {ctx->sort_vals[0].as<uint32_t>(), ctx->sort_vals[1].as<uint32_t>()};
    k_bal_regroup_keys<<<blocks_for(O, BALR_THREADS), BALR_THREADS, 0, st>>>(x->bal_cam.as<uint32_t>(), O, keys[0], vals[0]);
    C2B_KERNEL_CHECK();
    int res = 0;
    C2B_TRY(radix_sort_pairs(st, keys, vals, O, bit_length(C - 1), ctx->sort_hist, ctx->scan_tmp, &res));
    k_bal_regroup_gather<<<blocks_for(O, BALR_THREADS), BALR_THREADS, 0, st>>>(
        vals[res], O, ctx->out_idx[sel].as<uint32_t>(), ctx->out_uv[sel].as<double2>(), ctx->out_idx[fs].as<uint32_t>(),
        ctx->out_uv[fs].as<double2>());
    C2B_KERNEL_CHECK();
    ctx->out_sel = fs;
  }
  return C2B_OK;
}

int bal_read_text(BalReadState &s) {
  c2b_ctx *ctx = s.ctx;
  CtxExtra *x = s.x;
  cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
  const uint64_t B = s.B;
  char *ring = x->bal_ring.as<char>();
  auto &ev = s.ev;
  // the header, on the host, from the first chunk
  const int64_t got0 = bal_pread(s.fd, ring, std::min(B, s.size), 0, s.ms_read);
  if (got0 < 0) return set_error(C2B_ERR_IO, "cannot read %s: %s", s.path, strerror(errno));
  uint64_t hdr[3];
  {
    uint64_t i = 0;
    for (int k = 0; k < 3; ++k) {
      while (i < (uint64_t)got0 && bal_ws(ring[i])) ++i;
      if (i == (uint64_t)got0) {
        if ((uint64_t)got0 == s.size)
          return set_error(C2B_ERR_PARSE, "%s: byte %llu: the file ends inside the header", s.path, (unsigned long long)s.size);
        return set_error(C2B_ERR_PARSE, "%s: byte %llu: the header does not fit in one chunk (bal_chunk_bytes)", s.path,
                         (unsigned long long)i);
      }
      const uint64_t b = i;
      while (i < (uint64_t)got0 && !bal_ws(ring[i])) ++i;
      if (i == (uint64_t)got0 && (uint64_t)got0 < s.size)
        return set_error(C2B_ERR_PARSE, "%s: byte %llu: the header does not fit in one chunk (bal_chunk_bytes)", s.path,
                         (unsigned long long)b);
      if (!bal_parse_index(ring + b, (uint32_t)(i - b), hdr[k]))
        return set_error(C2B_ERR_PARSE, "%s: byte %llu: malformed header count", s.path, (unsigned long long)b);
    }
  }
  s.C = hdr[0], s.P = hdr[1], s.O = hdr[2];
  // 3 + 4 O + 9 C + 3 P tokens of at least one byte, separated by at least one byte
  const unsigned __int128 need = (unsigned __int128)3 + (unsigned __int128)4 * s.O + (unsigned __int128)9 * s.C +
                                 (unsigned __int128)3 * s.P;
  if (2 * need - 1 > s.size)
    return set_error(C2B_ERR_PARSE, "%s: byte 0: the header's counts need more bytes than the file has (%llu)", s.path,
                     (unsigned long long)s.size);
  C2B_TRY(bal_read_alloc(s));
  const uint64_t C = s.C, P = s.P, O = s.O, n_tok = (uint64_t)need;
  C2B_TRY(x->bal_cam.ensure(std::max<uint64_t>(O, 1) * 4));
  const uint64_t max_words = (B + 31) / 32;
  C2B_TRY(x->bal_scan.ensure(max_words * 8 + 64));
  // a slow token has more than 19 digits: at most B / 20 + 1 of them per chunk
  C2B_TRY(x->bal_slow[0].ensure((B / 20 + 2) * sizeof(BalSlow)));
  C2B_TRY(x->bal_slow[1].ensure((B / 20 + 2) * sizeof(BalSlow)));
  uint32_t *words = x->bal_scan.as<uint32_t>(), *first = words + max_words, *total = first + max_words;
  uint64_t *base = reinterpret_cast<uint64_t *>(s.d_err + 2);
  uint32_t *n_slow = reinterpret_cast<uint32_t *>(s.d_err + 3);  // [0], [1]: the two chunk buffers
  const int sel = ctx->out_sel;
  BalTextArgs a{};
  a.C = C, a.P = P, a.O = O;
  a.cam_of = x->bal_cam.as<uint32_t>();
  a.idx = ctx->out_idx[sel].as<uint32_t>();
  a.uv = ctx->out_uv[sel].as<double>();
  a.vecs = s.vecs;
  a.pts = s.pts;
  a.err = s.d_err;
  a.words = words;
  a.first = first;
  a.base = base;
  // per ring slot, in pinned memory once the chunk's parse is done: its slow-token count and the running ordinal
  uint64_t *h_tail = ctx->h_small.as<uint64_t>() + 4;
  std::vector<uint64_t> slow_pairs;  // (ordinal, bits)
  std::vector<BalSlow> recs;
  uint64_t ordinals_done = 0;
  // chunk j's parse is finished: its times, its slow tokens converted from the ring slot's bytes
  auto drain = [&](uint64_t j, uint32_t n_bytes) -> int {
    const int slot = (int)(j % BAL_RING);
    C2B_CUDA(cudaEventSynchronize(ev[slot][3]));
    s.add_times(slot);
    const uint32_t k = (uint32_t)h_tail[2 * slot];
    ordinals_done = h_tail[2 * slot + 1];
    if (k) {
      recs.resize(k);
      C2B_CUDA(cudaMemcpyAsync(recs.data(), x->bal_slow[j % 2].p, (size_t)k * sizeof(BalSlow), cudaMemcpyDeviceToHost,
                               ctx->aux_stream));
      C2B_CUDA(cudaStreamSynchronize(ctx->aux_stream));
      const char *bytes = ring + (size_t)slot * B;
      for (const BalSlow &r : recs) {
        const uint32_t len = r.len & 0x7fffffffu;
        if (r.pos + len > n_bytes) return set_error(C2B_ERR_CUDA, "BAL reader: slow token record out of its chunk");
        const char *t = bytes + r.pos, *e = t + len;
        const bool neg = *t == '-';
        if (*t == '-' || *t == '+') ++t;
        double v = 0;
        const auto res = std::from_chars(t, e, v, std::chars_format::general);
        if (res.ptr != e || (res.ec != std::errc() && res.ec != std::errc::result_out_of_range))
          return set_error(C2B_ERR_PARSE, "%s: malformed number (host conversion)", s.path);
        if (res.ec == std::errc::result_out_of_range) v = (r.len & 0x80000000u) ? INFINITY : 0.0;
        if (neg) v = -v;
        uint64_t bits;
        memcpy(&bits, &v, 8);
        slow_pairs.push_back(r.ordinal);
        slow_pairs.push_back(bits);
      }
      s.slow += k;
    }
    return C2B_OK;
  };
  uint64_t read_pos = (uint64_t)got0, chunk_off = 0, have = (uint64_t)got0;
  uint64_t prev_n = 0, tail = 0;
  int64_t pending = -1;
  uint32_t pending_n = 0;
  for (uint64_t k = 0;; ++k) {
    const int slot = (int)(k % BAL_RING);
    char *sp = ring + (size_t)slot * B;
    if (k > 0) {
      // the slot's previous chunk (k - 3) left with the copy that preceded chunk k - 2's parse, which was drained
      memcpy(sp, ring + (size_t)((k - 1) % BAL_RING) * B + prev_n, tail);
      const int64_t r = bal_pread(s.fd, sp + tail, B - tail, read_pos, s.ms_read);
      if (r < 0) return set_error(C2B_ERR_IO, "cannot read %s: %s", s.path, strerror(errno));
      read_pos += (uint64_t)r;
      have = tail + (uint64_t)r;
    }
    const bool eof = read_pos >= s.size;
    uint64_t n = have;
    if (!eof) {
      while (n > 0 && !bal_ws(sp[n - 1])) --n;
      if (n == 0)
        return set_error(C2B_ERR_PARSE, "%s: byte %llu: a token longer than bal_chunk_bytes (%llu)", s.path,
                         (unsigned long long)chunk_off, (unsigned long long)B);
    }
    if (n) {
      const uint32_t nw = (uint32_t)((n + 31) / 32);
      char *dbuf = x->bal_out[k % 2].as<char>();
      C2B_CUDA(cudaEventRecord(ev[slot][0], cp));
      C2B_CUDA(cudaMemcpyAsync(dbuf, sp, n, cudaMemcpyHostToDevice, cp));
      C2B_CUDA(cudaEventRecord(ev[slot][1], cp));
      C2B_CUDA(cudaStreamWaitEvent(st, ev[slot][1], 0));
      C2B_CUDA(cudaEventRecord(ev[slot][2], st));
      C2B_CUDA(cudaMemsetAsync(n_slow + (k % 2), 0, 4, st));
      k_bal_tok_flags<<<blocks_for(n, BALR_THREADS), BALR_THREADS, 0, st>>>(dbuf, (uint32_t)n, words, first);
      C2B_KERNEL_CHECK();
      C2B_TRY(exclusive_scan_u32(st, first, first, nw, total, ctx->scan_tmp));
      a.buf = dbuf;
      a.n = (uint32_t)n;
      a.file_off = chunk_off;
      a.slow = x->bal_slow[k % 2].as<BalSlow>();
      a.n_slow = n_slow + (k % 2);
      k_bal_parse_text<<<blocks_for(nw, BALR_THREADS), BALR_THREADS, 0, st>>>(a, nw);
      C2B_KERNEL_CHECK();
      k_bal_tok_advance<<<1, 1, 0, st>>>(base, total);
      C2B_KERNEL_CHECK();
      C2B_CUDA(cudaMemcpyAsync(h_tail + 2 * slot, n_slow + (k % 2), 4, cudaMemcpyDeviceToHost, st));
      C2B_CUDA(cudaMemcpyAsync(h_tail + 2 * slot + 1, base, 8, cudaMemcpyDeviceToHost, st));
      C2B_CUDA(cudaEventRecord(ev[slot][3], st));
      ++s.chunks;
    }
    // lag one: the previous chunk's slow tokens, while this one is on its way
    if (pending >= 0) C2B_TRY(drain((uint64_t)pending, pending_n));
    pending = n ? (int64_t)k : -1;
    pending_n = (uint32_t)n;
    if (eof || ordinals_done >= n_tok) break;  // tokens after the points are never read
    chunk_off += n;
    prev_n = n;
    tail = have - n;
  }
  if (pending >= 0) C2B_TRY(drain((uint64_t)pending, pending_n));
  s.bytes = read_pos;
  C2B_CUDA(cudaMemcpyAsync(ctx->h_small.p, s.d_err, 24, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  const unsigned long long *h = ctx->h_small.as<unsigned long long>();
  if (h[0] != BAL_NO_ERR) return set_error(C2B_ERR_PARSE, "%s: byte %llu: malformed token", s.path, h[0]);
  if (h[2] < n_tok)
    return set_error(C2B_ERR_PARSE, "%s: byte %llu: the file ends after %llu of the %llu tokens its header needs", s.path,
                     (unsigned long long)s.size, (unsigned long long)h[2], (unsigned long long)n_tok);
  if (h[1] != BAL_NO_ERR)
    return set_error(C2B_ERR_INVALID, "%s: byte %llu: observation index out of range (camera >= %llu or point >= %llu)",
                     s.path, h[1], (unsigned long long)C, (unsigned long long)P);
  if (!slow_pairs.empty()) {
    const uint64_t ns = slow_pairs.size() / 2;
    C2B_TRY(x->bal_slow[0].ensure(ns * 16));
    C2B_CUDA(cudaMemcpyAsync(x->bal_slow[0].p, slow_pairs.data(), ns * 16, cudaMemcpyHostToDevice, st));
    k_bal_scatter_slow<<<blocks_for(ns, BALR_THREADS), BALR_THREADS, 0, st>>>(x->bal_slow[0].as<uint64_t>(), ns, C, O,
                                                                              a.uv, s.vecs, s.pts);
    C2B_KERNEL_CHECK();
  }
  return bal_group(s);
}

int bal_read_binary(BalReadState &s) {
  c2b_ctx *ctx = s.ctx;
  CtxExtra *x = s.x;
  cudaStream_t st = ctx->stream, cp = ctx->copy_stream;
  const uint64_t B = s.B, W = B / 8;
  char *ring = x->bal_ring.as<char>();
  auto &ev = s.ev;
  unsigned char h24[24];
  const int64_t g = bal_pread(s.fd, reinterpret_cast<char *>(h24), 24, 0, s.ms_read);
  if (g < 0) return set_error(C2B_ERR_IO, "cannot read %s: %s", s.path, strerror(errno));
  if (g < 24) return set_error(C2B_ERR_PARSE, "%s: byte %llu: truncated binary BAL file", s.path, (unsigned long long)g);
  auto be = [](const unsigned char *b) {
    uint64_t v = 0;
    for (int k = 0; k < 8; ++k) v = (v << 8) | b[k];
    return v;
  };
  s.C = be(h24), s.P = be(h24 + 8), s.O = be(h24 + 16);
  if (s.C > s.size / 80 || s.P > s.size / 24 || s.O > s.size / 24)
    return set_error(C2B_ERR_PARSE, "%s: byte 0: binary BAL header counts exceed the file size", s.path);
  const uint64_t C = s.C, P = s.P, O = s.O;
  const uint64_t words = 3 + C + 3 * O + 9 * C + 3 * P;
  if (s.size < 8 * words)
    return set_error(C2B_ERR_PARSE, "%s: byte %llu: truncated binary BAL file (%llu bytes needed)", s.path,
                     (unsigned long long)s.size, (unsigned long long)(8 * words));
  C2B_TRY(bal_read_alloc(s));
  const int sel = ctx->out_sel;
  std::vector<uint64_t> off(C + 1, 0);
  uint64_t c = 0, seen = 0, next = 3;  // next: word of camera c's count
  BalBinArgs a{};
  a.C = C, a.P = P, a.O = O;
  uint64_t *d_off = ctx->out_offsets[sel].as<uint64_t>();
  a.off = d_off;
  a.idx = ctx->out_idx[sel].as<uint32_t>();
  a.uv = ctx->out_uv[sel].as<double>();
  a.vecs = s.vecs;
  a.pts = s.pts;
  a.err = s.d_err;
  for (uint64_t k = 0, w0 = 0; w0 < words; ++k, w0 += W) {
    const int slot = (int)(k % BAL_RING);
    char *sp = ring + (size_t)slot * B;
    const uint64_t n = std::min(W, words - w0);
    if (k >= BAL_RING) {  // the slot's previous chunk has been copied and parsed
      C2B_CUDA(cudaEventSynchronize(ev[slot][3]));
      s.add_times(slot);
    }
    const int64_t r = bal_pread(s.fd, sp, 8 * n, 8 * w0, s.ms_read);
    if (r < 0) return set_error(C2B_ERR_IO, "cannot read %s: %s", s.path, strerror(errno));
    if ((uint64_t)r < 8 * n)
      return set_error(C2B_ERR_PARSE, "%s: byte %llu: truncated binary BAL file", s.path,
                       (unsigned long long)(8 * w0 + (uint64_t)r));
    // the chain of count words inside this chunk
    const uint64_t c0 = c;
    while (c < C && next < w0 + n) {
      const uint64_t cnt = be(reinterpret_cast<const unsigned char *>(sp) + 8 * (next - w0));
      if (cnt > O - seen)
        return set_error(C2B_ERR_PARSE, "%s: byte %llu: camera %llu's observation count %llu exceeds the %llu left",
                         s.path, (unsigned long long)(8 * next), (unsigned long long)c, (unsigned long long)cnt,
                         (unsigned long long)(O - seen));
      off[c] = seen;
      seen += cnt;
      ++c;
      next = 3 + c + 3 * seen;
    }
    char *dbuf = x->bal_out[k % 2].as<char>();
    if (k >= 2) C2B_CUDA(cudaStreamWaitEvent(cp, ev[(k - 2) % BAL_RING][3], 0));  // chunk k - 2 left dbuf
    C2B_CUDA(cudaEventRecord(ev[slot][0], cp));
    if (c > c0)
      C2B_CUDA(cudaMemcpyAsync(d_off + c0, off.data() + c0, (c - c0) * 8, cudaMemcpyHostToDevice, cp));
    C2B_CUDA(cudaMemcpyAsync(dbuf, sp, 8 * n, cudaMemcpyHostToDevice, cp));
    C2B_CUDA(cudaEventRecord(ev[slot][1], cp));
    C2B_CUDA(cudaStreamWaitEvent(st, ev[slot][1], 0));
    C2B_CUDA(cudaEventRecord(ev[slot][2], st));
    a.buf = reinterpret_cast<const uint64_t *>(dbuf);
    a.w0 = w0;
    a.n = n;
    a.c_known = c;
    k_bal_parse_binary<<<blocks_for(n, BALR_THREADS), BALR_THREADS, 0, st>>>(a);
    C2B_KERNEL_CHECK();
    C2B_CUDA(cudaEventRecord(ev[slot][3], st));
    ++s.chunks;
    s.bytes += 8 * n;
  }
  C2B_CUDA(cudaStreamSynchronize(st));
  for (uint64_t k = s.chunks >= BAL_RING ? s.chunks - BAL_RING : 0; k < s.chunks; ++k) s.add_times((int)(k % BAL_RING));
  if (seen != O)
    return set_error(C2B_ERR_PARSE, "%s: byte %llu: the cameras' observation counts sum to %llu, the header says %llu",
                     s.path, (unsigned long long)(8 * (3 + C + 3 * seen)), (unsigned long long)seen,
                     (unsigned long long)O);
  off[C] = O;
  C2B_CUDA(cudaMemcpyAsync(d_off + C, off.data() + C, 8, cudaMemcpyHostToDevice, st));
  C2B_CUDA(cudaMemcpyAsync(ctx->h_small.p, s.d_err, 16, cudaMemcpyDeviceToHost, st));
  C2B_CUDA(cudaStreamSynchronize(st));
  const unsigned long long bad = ctx->h_small.as<unsigned long long>()[1];
  if (bad != BAL_NO_ERR)
    return set_error(C2B_ERR_INVALID, "%s: byte %llu: observation index out of range (point >= %llu)", s.path, bad,
                     (unsigned long long)P);
  return C2B_OK;
}
}  // namespace

int c2b_read_bal_resident(c2b_ctx *ctx, const char *path, int format, c2b_bal_read_stats *out) {
  if (!ctx || !path) return set_error(C2B_ERR_INVALID, "c2b_read_bal_resident: null argument");
  if (format != C2B_BAL_TEXT && format != C2B_BAL_BINARY)
    return set_error(C2B_ERR_INVALID, "c2b_read_bal_resident: unknown format %d", format);
  CtxExtra *x = ctx->extra.get();
  C2B_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // whatever happens below, the previous resident problem is replaced
  x->have_result = x->have_cameras = x->have_points = false;
  x->host_call_last = false;
  x->grid.valid = false;
  BalReadState s{ctx, x, path, -1, 0, x->tun.bal_chunk_bytes};
  s.fd = open(path, O_RDONLY | O_CLOEXEC);
  if (s.fd < 0) return set_error(C2B_ERR_IO, "cannot open %s: %s", path, strerror(errno));
  int rc = [&]() -> int {
    struct stat sb;
    if (fstat(s.fd, &sb) != 0 || !S_ISREG(sb.st_mode)) return set_error(C2B_ERR_IO, "%s is not a regular file", path);
    s.size = (uint64_t)sb.st_size;
    for (auto &slot : s.ev)
      for (auto &e : slot) C2B_TRY(e.create());
    x->bal_ring.node = ctx->numa_node;
    C2B_TRY(x->bal_ring.ensure(BAL_RING * s.B));
    C2B_TRY(ctx->h_small.ensure(256));
    C2B_TRY(format == C2B_BAL_TEXT ? bal_read_text(s) : bal_read_binary(s));
    // install as c2b_cull_problem_resident does: camera records on the host (from_vec), points, CSR
    const uint64_t C = s.C, P = s.P, O = s.O;
    std::vector<double> vecs(9 * C), cams(15 * C);
    if (C) C2B_CUDA(cudaMemcpyAsync(vecs.data(), s.vecs, C * 72, cudaMemcpyDeviceToHost, st));
    C2B_CUDA(cudaStreamSynchronize(st));
    for (uint64_t c = 0; c < C; ++c) c2b_camera_from_vec(&vecs[9 * c], &cams[15 * c]);
    C2B_TRY(c2b_upload_cameras(ctx, cams.data(), C));
    C2B_TRY(c2b_points_commit(ctx, P));
    ctx->out_C = C;
    ctx->out_O = O;
    C2B_CUDA(cudaStreamSynchronize(st));
    x->have_result = true;
    return C2B_OK;
  }();
  close(s.fd);
  if (rc != C2B_OK) {
    cudaStreamSynchronize(st);
    cudaStreamSynchronize(ctx->copy_stream);
    x->have_result = x->have_cameras = x->have_points = false;
    return rc;
  }
  if (out) {
    memset(out, 0, sizeof *out);
    out->n_cameras = s.C;
    out->n_points = s.P;
    out->n_obs = s.O;
    out->bytes = s.bytes;
    out->chunks = s.chunks;
    out->slow_tokens = s.slow;
    out->regrouped = s.regrouped;
    out->ms_read = (float)s.ms_read;
    out->ms_h2d = s.ms_h2d;
    out->ms_parse = s.ms_parse;
  }
  return C2B_OK;
}


}  // extern "C"
