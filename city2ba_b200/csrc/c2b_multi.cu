// c2b_multi.cu — the visibility path on several GPUs of one box, inside the library (SURVEY 8e):
// one process, one c2b_ctx + stream set + worker thread per device, one NCCL communicator
// (ncclCommInitAll), contiguous camera ranges, mesh / BVH / points replicated.
//
//   phase 1  (workers)   every GPU uploads 1/G of the point array over its own PCIe link into its slot of
//                        its own point array
//   exchange (caller)    ncclAllGather of the shards, in place, one group call  -> every GPU holds all points
//   phase 2  (workers)   SoA copy + bounds, camera range upload, the resident pass of c2b_api.cu
//   exchange (caller)    ONE ncclAllGather of the per-GPU observation counts (north star: "per-GPU observation
//                        counts and offsets are exchanged with a single NCCL allgather") -> slab offsets
//   phase 3  (workers)   offsets rebased on the device, slab copied into the ONE pinned host CSR at its offset
//
// The collectives are issued by the calling thread between the phases, after every worker has reported
// success, so a failure on one GPU (out of memory, a bad argument) can never leave the others waiting inside
// a collective.  replaces: rayon's par_iter over cameras + order-preserving collect, src/generate.rs:434-441,
// 479-481.  NCCL is loaded with dlopen (libnccl.so.2): the single-GPU library has no NCCL dependency.
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "c2b_common.cuh"
#include "c2b_internal.h"

using namespace c2b;

namespace {

struct NcclApi {
  void *handle = nullptr;
  ncclResult_t (*GetVersion)(int *) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char *(*GetErrorString)(ncclResult_t) = nullptr;
  std::string path;
};

NcclApi &nccl() {
  static NcclApi a;
  return a;
}

int load_nccl() {
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  NcclApi &a = nccl();
  if (a.handle) return C2B_OK;
  std::vector<std::string> names;
  if (const char *e = getenv("C2B_NCCL_LIB")) names.push_back(e);
  names.push_back("libnccl.so.2");  // the copy the process already mapped (e.g. torch's), else the system's
  names.push_back("libnccl.so");
  std::string why;
  for (const std::string &n : names) {
    void *h = dlopen(n.c_str(), RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      why += n + ": " + (dlerror() ? dlerror() : "?") + "; ";
      continue;
    }
    auto sym = [&](const char *s) { return dlsym(h, s); };
    a.GetVersion = reinterpret_cast<decltype(a.GetVersion)>(sym("ncclGetVersion"));
    a.CommInitAll = reinterpret_cast<decltype(a.CommInitAll)>(sym("ncclCommInitAll"));
    a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(sym("ncclCommDestroy"));
    a.AllGather = reinterpret_cast<decltype(a.AllGather)>(sym("ncclAllGather"));
    a.GroupStart = reinterpret_cast<decltype(a.GroupStart)>(sym("ncclGroupStart"));
    a.GroupEnd = reinterpret_cast<decltype(a.GroupEnd)>(sym("ncclGroupEnd"));
    a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(sym("ncclGetErrorString"));
    if (a.CommInitAll && a.CommDestroy && a.AllGather && a.GroupStart && a.GroupEnd && a.GetErrorString) {
      a.handle = h;
      a.path = n;
      return C2B_OK;
    }
    why += n + ": symbols missing; ";
    dlclose(h);
  }
  return set_error(C2B_ERR_NCCL, "cannot load NCCL (%s)", why.c_str());
}

#define C2B_NCCL(call)                                                                              \
  do {                                                                                              \
    ncclResult_t _r = (call);                                                                       \
    if (_r != ncclSuccess)                                                                          \
      return set_error(C2B_ERR_NCCL, "%s:%d %s -> %s", __FILE__, __LINE__, #call, nccl().GetErrorString(_r)); \
  } while (0)

__global__ void k_set_u64(uint64_t *p, uint64_t v) { *p = v; }

// persistent worker: runs job(g) when told to, reports its status and last-error text
struct Worker {
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::function<int()> job;
  bool has_job = false, done = false, quit = false;
  int rc = C2B_OK;
  std::string err;
  void loop() {
    for (;;) {
      std::function<int()> j;
      {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return has_job || quit; });
        if (quit) return;
        j = job;
        has_job = false;
      }
      const int r = j();
      {
        std::lock_guard<std::mutex> lk(mu);
        rc = r;
        err = r == C2B_OK ? std::string() : last_error_ref();
        done = true;
      }
      cv.notify_all();
    }
  }
  void start(std::function<int()> j) {
    {
      std::lock_guard<std::mutex> lk(mu);
      job = std::move(j);
      has_job = true;
      done = false;
    }
    cv.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return done; });
    return rc;
  }
};

}  // namespace

struct c2b_multi {
  int n = 0;
  int dev[C2B_MAX_GPUS] = {};
  c2b_ctx *ctx[C2B_MAX_GPUS] = {};
  ncclComm_t comm[C2B_MAX_GPUS] = {};
  bool have_comm = false;
  std::unique_ptr<Worker> worker[C2B_MAX_GPUS];
  DevBuf d_counts[C2B_MAX_GPUS];
  PinBuf h_counts[C2B_MAX_GPUS];
  Event ev[C2B_MAX_GPUS][4];
  PinBuf h_offsets, h_idx, h_uv;  // the ONE host CSR
  std::mutex mu;
  // share of the cameras each GPU gets: equal at first, then following each GPU's measured speed (pass + slab
  // transfer per camera) in the previous call.  The result transfer is usually the longest leg of a call and the
  // GPUs of a box do not all reach host memory equally fast (8-GPU box, all copying at once: 6.5-7.5 ms for GPUs
  // 4-7, 11 ms for GPUs 0-3, profiles/r02k_bench_cfg4_8gpu.json), so equal ranges wait for the slowest link.
  double share[C2B_MAX_GPUS] = {};
  bool adaptive = true;
  int adjustments = 0;
};

struct c2b_multi_scene {
  int n = 0;
  c2b_scene *scene[C2B_MAX_GPUS] = {};
};

namespace {

// run job(g) on every worker; first failure wins (its message becomes the caller's last error)
int run_all(c2b_multi *m, const std::function<int(int)> &job) {
  for (int g = 0; g < m->n; ++g) m->worker[g]->start([=]() { return job(g); });
  int rc = C2B_OK;
  for (int g = 0; g < m->n; ++g) {
    const int r = m->worker[g]->wait();
    if (r != C2B_OK && rc == C2B_OK) {
      rc = r;
      last_error_ref() = "GPU " + std::to_string(m->dev[g]) + ": " + m->worker[g]->err;
    }
  }
  return rc;
}

}  // namespace

extern "C" {

int c2b_init_multi(int n_gpus, const int *devices, c2b_multi **out) {
  if (!out) return set_error(C2B_ERR_INVALID, "c2b_init_multi: out is null");
  *out = nullptr;
  if (n_gpus < 1 || n_gpus > C2B_MAX_GPUS)
    return set_error(C2B_ERR_INVALID, "c2b_init_multi: n_gpus %d out of range [1,%d]", n_gpus, C2B_MAX_GPUS);
  int have = 0;
  if (cudaGetDeviceCount(&have) != cudaSuccess || have == 0) {
    (void)cudaGetLastError();
    return set_error(C2B_ERR_NO_DEVICE, "no CUDA device visible; this library has no CPU fallback");
  }
  c2b_multi *m = new (std::nothrow) c2b_multi();
  if (!m) return set_error(C2B_ERR_OOM, "out of host memory");
  m->n = n_gpus;
  m->h_offsets.portable = m->h_idx.portable = m->h_uv.portable = true;
  for (int g = 0; g < n_gpus; ++g) m->share[g] = 1.0 / n_gpus;
  if (const char *e = getenv("C2B_MULTI_ADAPTIVE")) m->adaptive = atoi(e) != 0;
  for (int g = 0; g < n_gpus; ++g) {
    m->dev[g] = devices ? devices[g] : g;
    for (int q = 0; q < g; ++q)
      if (m->dev[q] == m->dev[g]) {
        delete m;
        return set_error(C2B_ERR_INVALID, "c2b_init_multi: device %d listed twice", devices[g]);
      }
  }
  auto fail = [&](int rc) {
    const std::string keep = last_error_ref();
    c2b_shutdown_multi(m);
    last_error_ref() = keep;
    return rc;
  };
  for (int g = 0; g < n_gpus; ++g) {
    const int rc = c2b_init(m->dev[g], &m->ctx[g]);
    if (rc != C2B_OK) return fail(rc);
    if (cudaSetDevice(m->dev[g]) != cudaSuccess) return fail(set_error(C2B_ERR_CUDA, "cudaSetDevice(%d) failed", m->dev[g]));
    for (auto &e : m->ev[g]) {
      const int rc = e.create();
      if (rc != C2B_OK) return fail(rc);
    }
    if (m->d_counts[g].ensure(C2B_MAX_GPUS * 8) != C2B_OK || m->h_counts[g].ensure(C2B_MAX_GPUS * 8) != C2B_OK)
      return fail(C2B_ERR_OOM);
  }
  if (n_gpus > 1) {
    const int rc = load_nccl();
    if (rc != C2B_OK) return fail(rc);
    // NCCL announces its version on stdout when the first communicator is created; a command line whose stdout
    // lines are the reference's (and bench.py's one JSON line) keeps it on stderr
    fflush(stdout);
    const int saved_stdout = dup(1);
    if (saved_stdout >= 0) dup2(2, 1);
    const ncclResult_t r = nccl().CommInitAll(m->comm, n_gpus, m->dev);
    if (saved_stdout >= 0) {
      fflush(stdout);
      dup2(saved_stdout, 1);
      close(saved_stdout);
    }
    if (r != ncclSuccess)
      return fail(set_error(C2B_ERR_NCCL, "ncclCommInitAll(%d devices) -> %s", n_gpus, nccl().GetErrorString(r)));
    m->have_comm = true;
  }
  for (int g = 0; g < n_gpus; ++g) {
    m->worker[g] = std::make_unique<Worker>();
    Worker *w = m->worker[g].get();
    w->th = std::thread([w]() { w->loop(); });
  }
  *out = m;
  return C2B_OK;
}

void c2b_shutdown_multi(c2b_multi *m) {
  if (!m) return;
  for (int g = 0; g < m->n; ++g)
    if (m->worker[g]) {
      {
        std::lock_guard<std::mutex> lk(m->worker[g]->mu);
        m->worker[g]->quit = true;
      }
      m->worker[g]->cv.notify_all();
      if (m->worker[g]->th.joinable()) m->worker[g]->th.join();
      m->worker[g].reset();
    }
  for (int g = 0; g < m->n; ++g) {
    if (!m->ctx[g]) continue;
    cudaSetDevice(m->dev[g]);
    cudaDeviceSynchronize();
    if (m->have_comm && m->comm[g]) nccl().CommDestroy(m->comm[g]);
    for (auto &e : m->ev[g]) e.release();
    m->d_counts[g].release();
    m->h_counts[g].release();
  }
  for (int g = 0; g < m->n; ++g)
    if (m->ctx[g]) c2b_shutdown(m->ctx[g]);
  delete m;
}

int c2b_multi_num_gpus(const c2b_multi *m) { return m ? m->n : 0; }
c2b_ctx *c2b_multi_ctx(c2b_multi *m, int g) { return (m && g >= 0 && g < m->n) ? m->ctx[g] : nullptr; }

int c2b_scene_create_multi(c2b_multi *m, const float *xyz, uint64_t nv, const uint32_t *tri, uint64_t nt,
                           c2b_multi_scene **out) {
  if (!m || !out) return set_error(C2B_ERR_INVALID, "c2b_scene_create_multi: null argument");
  *out = nullptr;
  c2b_multi_scene *s = new (std::nothrow) c2b_multi_scene();
  if (!s) return set_error(C2B_ERR_OOM, "out of host memory");
  s->n = m->n;
  const int rc = run_all(m, [=](int g) { return c2b_scene_create(m->ctx[g], xyz, nv, tri, nt, &s->scene[g]); });
  if (rc != C2B_OK) {
    const std::string keep = last_error_ref();
    c2b_scene_destroy_multi(s);
    last_error_ref() = keep;
    return rc;
  }
  *out = s;
  return C2B_OK;
}

c2b_scene *c2b_multi_scene_get(const c2b_multi_scene *s, int g) {
  return (s && g >= 0 && g < s->n) ? s->scene[g] : nullptr;
}

void c2b_scene_destroy_multi(c2b_multi_scene *s) {
  if (!s) return;
  for (int g = 0; g < s->n; ++g) c2b_scene_destroy(s->scene[g]);
  delete s;
}

int c2b_visibility_graph_multi(c2b_multi *m, const c2b_multi_scene *scene, const double *cams, uint64_t C,
                               const double *pts, uint64_t P, double max_dist, const c2b_vis_options *opt_in,
                               c2b_obs *out, c2b_multi_stats *stats) {
  if (!m || !out) return set_error(C2B_ERR_INVALID, "c2b_visibility_graph_multi: null argument");
  if ((C && !cams) || (P && !pts)) return set_error(C2B_ERR_INVALID, "c2b_visibility_graph_multi: null input array");
  if (scene && scene->n != m->n) return set_error(C2B_ERR_INVALID, "scene was built for %d GPUs, not %d", scene->n, m->n);
  c2b_vis_options opt;
  if (opt_in)
    opt = *opt_in;
  else
    c2b_vis_options_default(&opt);
  if (opt.occlusion == C2B_OCC_MESH && !scene) return set_error(C2B_ERR_INVALID, "C2B_OCC_MESH needs a scene");
  const int G = m->n;
  const auto t0 = std::chrono::steady_clock::now();
  const uint64_t per = (P + (uint64_t)G - 1) / (uint64_t)G;  // points per shard (the last one may be short)
  // contiguous camera ranges, sized by the GPUs' shares
  std::vector<uint64_t> cam_lo((size_t)G + 1, 0);
  {
    double cum = 0.0;
    for (int g = 0; g < G; ++g) {
      cum += m->share[g];
      cam_lo[(size_t)g + 1] = g == G - 1 ? C : std::min<uint64_t>(C, std::max<uint64_t>(cam_lo[(size_t)g], (uint64_t)(cum * (double)C + 0.5)));
    }
  }
  std::vector<double *> d_pts((size_t)G, nullptr);
  std::vector<c2b_obs> part((size_t)G);

  // ---- phase 1: 1/G of the points per GPU, each over its own PCIe link ----
  C2B_TRY(run_all(m, [&](int g) -> int {
    c2b_ctx *ctx = m->ctx[g];
    C2B_CUDA(cudaSetDevice(m->dev[g]));
    C2B_CUDA(cudaEventRecord(m->ev[g][0], ctx->stream));
    C2B_TRY(c2b_points_device_buffer(ctx, per * (uint64_t)G, &d_pts[(size_t)g]));
    const uint64_t lo = std::min(P, (uint64_t)g * per), hi = std::min(P, ((uint64_t)g + 1) * per);
    if (G == 1) return hi > lo ? c2b_internal_copy_in(ctx, d_pts[0], pts, P * 24) : C2B_OK;
    if (hi > lo) C2B_TRY(c2b_internal_copy_in(ctx, d_pts[(size_t)g] + 3 * lo, pts + 3 * lo, (hi - lo) * 24));
    return C2B_OK;
  }));
  // ---- exchange 1: all-gather the shards over NVLink, in place ----
  if (G > 1 && per) {
    C2B_NCCL(nccl().GroupStart());
    for (int g = 0; g < G; ++g) {
      const ncclResult_t r = nccl().AllGather(d_pts[(size_t)g] + 3 * (uint64_t)g * per, d_pts[(size_t)g], (size_t)(3 * per),
                                              ncclDouble, m->comm[g], m->ctx[g]->stream);
      if (r != ncclSuccess) {
        nccl().GroupEnd();
        return set_error(C2B_ERR_NCCL, "ncclAllGather(points) -> %s", nccl().GetErrorString(r));
      }
    }
    C2B_NCCL(nccl().GroupEnd());
  }
  // ---- phase 2: the resident pass on each GPU's camera range ----
  static const bool trace = getenv("C2B_TRACE") != nullptr;
  auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
  if (trace) fprintf(stderr, "[c2b_multi] phase 2 starts at %.3f ms\n", since());
  C2B_TRY(run_all(m, [&](int g) -> int {
    c2b_ctx *ctx = m->ctx[g];
    C2B_CUDA(cudaSetDevice(m->dev[g]));
    const double ta = since();
    C2B_TRY(c2b_points_commit(ctx, P));
    C2B_CUDA(cudaEventRecord(m->ev[g][1], ctx->stream));
    const uint64_t c0 = cam_lo[(size_t)g], c1 = cam_lo[(size_t)g + 1];
    const double tb = since();
    C2B_TRY(c2b_upload_cameras(ctx, cams ? cams + 15 * c0 : nullptr, c1 - c0));
    const double tc = since();
    C2B_TRY(c2b_visibility_graph_resident(ctx, scene ? scene->scene[g] : nullptr, max_dist, &opt, &part[(size_t)g]));
    if (trace)
      fprintf(stderr, "[c2b_multi] gpu %d phase 2: start %.3f commit %.3f cameras %.3f resident pass %.3f ms (host clock)\n", g, ta,
              tb - ta, tc - tb, since() - tc);
    C2B_CUDA(cudaEventRecord(m->ev[g][2], ctx->stream));
    k_set_u64<<<1, 1, 0, ctx->stream>>>(m->d_counts[g].as<uint64_t>() + g, part[(size_t)g].n_obs);
    C2B_KERNEL_CHECK();
    return C2B_OK;
  }));
  // ---- exchange 2: ONE all-gather of the per-GPU observation counts ----
  if (G > 1) {
    C2B_NCCL(nccl().GroupStart());
    for (int g = 0; g < G; ++g) {
      const ncclResult_t r = nccl().AllGather(m->d_counts[g].as<uint64_t>() + g, m->d_counts[g].p, 1, ncclUint64,
                                              m->comm[g], m->ctx[g]->stream);
      if (r != ncclSuccess) {
        nccl().GroupEnd();
        return set_error(C2B_ERR_NCCL, "ncclAllGather(counts) -> %s", nccl().GetErrorString(r));
      }
    }
    C2B_NCCL(nccl().GroupEnd());
  }
  // ---- phase 3: every GPU learns its slab's offset from the gathered counts and copies the slab home ----
  std::vector<uint64_t> base((size_t)G, 0), total((size_t)G, 0);
  std::vector<float> ms_d2h((size_t)G, 0.0f);
  C2B_TRY(run_all(m, [&](int g) -> int {
    c2b_ctx *ctx = m->ctx[g];
    C2B_CUDA(cudaSetDevice(m->dev[g]));
    uint64_t *hc = m->h_counts[g].as<uint64_t>();
    C2B_CUDA(cudaMemcpyAsync(hc, m->d_counts[g].p, (size_t)G * 8, cudaMemcpyDeviceToHost, ctx->stream));
    C2B_CUDA(cudaEventRecord(m->ev[g][3], ctx->stream));
    C2B_CUDA(cudaStreamSynchronize(ctx->stream));
    uint64_t b = 0, t = 0;
    for (int r = 0; r < G; ++r) {
      if (r < g) b += hc[r];
      t += hc[r];
    }
    if (hc[g] != part[(size_t)g].n_obs) return set_error(C2B_ERR_NCCL, "count all-gather returned %llu for this GPU, expected %llu",
                                                         (unsigned long long)hc[g], (unsigned long long)part[(size_t)g].n_obs);
    base[(size_t)g] = b;
    total[(size_t)g] = t;
    {
      // the one host CSR: the first GPU to get here sizes it, the others find it large enough
      std::lock_guard<std::mutex> lk(m->mu);
      C2B_TRY(m->h_offsets.ensure((C + 1) * 8));
      C2B_TRY(m->h_idx.ensure(std::max<uint64_t>(t, 1) * 4));
      C2B_TRY(m->h_uv.ensure(std::max<uint64_t>(t, 1) * 16));
    }
    const uint64_t c0 = cam_lo[(size_t)g];
    return c2b_download_obs_into(ctx, b, m->h_offsets.as<uint64_t>() + c0, m->h_idx.as<uint32_t>() + b,
                                 m->h_uv.as<double>() + 2 * b, g == G - 1, &ms_d2h[(size_t)g]);
  }));

  c2b_obs acc;
  memset(&acc, 0, sizeof acc);
  acc.n_cameras = C;
  acc.n_obs = total[0];
  acc.offsets = m->h_offsets.as<uint64_t>();
  acc.point_idx = m->h_idx.as<uint32_t>();
  acc.uv = m->h_uv.as<double>();
  acc.h2d_bytes = P * 24 + C * 120;
  acc.d2h_bytes = (C + 1) * 8 + acc.n_obs * 20;
  c2b_multi_stats st;
  memset(&st, 0, sizeof st);
  st.n_gpus = G;
  for (int g = 0; g < G; ++g) {
    const c2b_obs &p = part[(size_t)g];
    acc.n_candidates += p.n_candidates;
    acc.pairs_evaluated += p.pairs_evaluated;
    acc.nodes_visited += p.nodes_visited;
    acc.tris_tested += p.tris_tested;
    acc.ms_prep = std::max(acc.ms_prep, p.ms_prep);
    acc.ms_cull = std::max(acc.ms_cull, p.ms_cull);
    acc.ms_sort = std::max(acc.ms_sort, p.ms_sort);
    acc.ms_traverse = std::max(acc.ms_traverse, p.ms_traverse);
    acc.ms_compact = std::max(acc.ms_compact, p.ms_compact);
    cudaSetDevice(m->dev[g]);
    float a = 0, b = 0, c = 0;
    if (cudaEventElapsedTime(&a, m->ev[g][0], m->ev[g][1]) != cudaSuccess) (void)cudaGetLastError();
    if (cudaEventElapsedTime(&b, m->ev[g][1], m->ev[g][2]) != cudaSuccess) (void)cudaGetLastError();
    if (cudaEventElapsedTime(&c, m->ev[g][2], m->ev[g][3]) != cudaSuccess) (void)cudaGetLastError();
    st.cam_begin[g] = cam_lo[(size_t)g];
    st.cam_end[g] = cam_lo[(size_t)g + 1];
    st.n_obs[g] = p.n_obs;
    st.obs_base[g] = base[(size_t)g];
    st.ms_points[g] = a;
    st.ms_compute[g] = b;
    st.ms_exchange[g] = c;
    st.ms_d2h[g] = ms_d2h[(size_t)g];
    acc.ms_h2d = std::max(acc.ms_h2d, a);
    acc.ms_d2h = std::max(acc.ms_d2h, ms_d2h[(size_t)g]);
    acc.ms_total = std::max(acc.ms_total, a + b + c + ms_d2h[(size_t)g]);
  }
  // next call's shares: what a GPU spends per camera AFTER the point exchange — its pass plus its slab's way to
  // host memory — is estimated from this call: the pass as cameras x the SMALLEST per-camera pass time any GPU
  // showed (the GPUs are alike; a call in which a GPU had to grow its buffers or repeat an optimistic pass would
  // otherwise pollute the estimate), the transfer as measured (CUDA events around the copies).  When the slowest
  // GPU took clearly longer than the fastest (> 15 %; > 50 % after two adjustments), the shares become
  // proportional to the GPUs' speeds, each within [1/2, 2] of an equal share; otherwise they stay, so that the
  // ranges — and with them every per-GPU buffer size — settle after a call or two
  if (m->adaptive && G > 1 && acc.n_obs * 20 >= (64ull << 20)) {
    double c_bar = 1e300;
    for (int g = 0; g < G; ++g) {
      const uint64_t nc = cam_lo[(size_t)g + 1] - cam_lo[(size_t)g];
      if (nc && st.ms_compute[g] > 0.0f) c_bar = std::min(c_bar, (double)st.ms_compute[g] / (double)nc);
    }
    double speed[C2B_MAX_GPUS], total_speed = 0.0, tmin = 1e300, tmax = 0.0;
    bool ok = c_bar < 1e300;
    for (int g = 0; g < G && ok; ++g) {
      const uint64_t nc = cam_lo[(size_t)g + 1] - cam_lo[(size_t)g];
      const double t = (double)nc * c_bar + (double)st.ms_d2h[g];
      speed[g] = t > 0.0 && nc ? (double)nc / t : 0.0;
      ok = speed[g] > 0.0;
      total_speed += speed[g];
      tmin = std::min(tmin, t);
      tmax = std::max(tmax, t);
    }
    if (ok && tmax > (m->adjustments < 2 ? 1.15 : 1.50) * tmin) {
      double sum = 0.0;
      for (int g = 0; g < G; ++g) {
        m->share[g] = std::min(std::max(speed[g] / total_speed, 0.5 / G), 2.0 / G);
        sum += m->share[g];
      }
      for (int g = 0; g < G; ++g) m->share[g] /= sum;
      ++m->adjustments;
    }
  }
  st.ms_wall = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (stats) *stats = st;
  *out = acc;
  return C2B_OK;
}

}  // extern "C"
