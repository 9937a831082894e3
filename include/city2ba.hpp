// city2ba.hpp — C++17 host mirror of the reference's library surface for the visibility / noise
// hot path, over the C ABI of libcity2ba_cuda.so (include/city2ba_cuda.h).
//
// The reference is a Rust crate (tkonolige/city2ba); this image has no rustc, so the host side a
// Rust maintainer would keep is restated here in C++ with the SAME names, argument order and error
// behaviour, so that tests written against it read like the reference's own (tests/cpp/).
//   city2ba::SnavelyCamera            src/baproblem.rs:107-225   (project_world, project, center,
//                                     from_position_direction, transform, from_vec / to_vec)
//   city2ba::BAProblem                src/baproblem.rs:256-801   (from_visibility, cull, BAL text/binary I/O)
//   city2ba::tobj::load_obj           tobj 0.1.12 (Cargo.lock:1149-1150) as called at src/bin/city2ba.rs:481
//   city2ba::generate::*              src/generate.rs:109-544    (generate_cameras_{path,path_step,poisson},
//                                     generate_world_points_uniform, visibility_graph, move_to_origin,
//                                     modify_intrinsics)
//   city2ba::synthetic::*             src/synthetic.rs:163-381   (synthetic_grid, synthetic_line)
//   city2ba::noise::*                 src/noise.rs:47-416        (add_drift*, add_noise, add_sin_noise on the GPU;
//                                     add_incorrect_correspondences, drop_features, split_landmarks,
//                                     join_landmarks: sequential graph edits, host)
// Precondition failures that `panic!`/`assert!` in the reference throw std::logic_error here;
// city2ba::Error carries the reference's Error kinds (src/baproblem.rs:32-62).  Randomness: the
// reference draws from thread_rng(); every noise function here takes a seed (Philox4x32-10 stream).
// There is no CPU fallback: everything that computes goes through the GPU library.
#pragma once
#include <algorithm>
#include <array>
#include <charconv>
#include <cctype>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <fstream>
#include <numeric>
#include <optional>
#include <sstream>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "city2ba_cuda.h"

namespace city2ba {

using Vector3 = std::array<double, 3>;
using Point3 = std::array<double, 3>;
using Observation = std::pair<size_t, std::pair<double, double>>;  // (point index, (u, v))
using VisGraph = std::vector<std::vector<Observation>>;

// city2ba::Error, src/baproblem.rs:32-62
struct Error : std::runtime_error {
  enum Kind { ParseError, EmptyProblem, IOError, Gpu } kind;
  Error(Kind k, const std::string &what) : std::runtime_error(what), kind(k) {}
};

namespace detail {
inline void check(int rc) {
  if (rc == C2B_OK) return;
  throw Error(rc == C2B_ERR_EMPTY   ? Error::EmptyProblem
              : rc == C2B_ERR_IO    ? Error::IOError
              : rc == C2B_ERR_PARSE ? Error::ParseError
                                    : Error::Gpu,
              c2b_last_error());
}
inline void require(bool ok, const char *what) {
  if (!ok) throw std::logic_error(what);  // the reference's assert! / panic!
}
}  // namespace detail

// ---- rotations in cgmath's conventions (column-major 3x3 as 9 doubles) ------------------------------
using Basis3 = std::array<double, 9>;
inline Basis3 basis_one() { return {1, 0, 0, 0, 1, 0, 0, 0, 1}; }
inline Basis3 from_angle_y(double rad) {
  const double s = std::sin(rad), c = std::cos(rad);
  return {c, 0, -s, 0, 1, 0, s, 0, c};
}
inline Basis3 from_angle_x(double rad) {
  const double s = std::sin(rad), c = std::cos(rad);
  return {1, 0, 0, 0, c, s, 0, -s, c};
}
inline Basis3 from_axis_angle(const Vector3 &a, double rad) {
  const double s = std::sin(rad), c = std::cos(rad), k = 1.0 - c;
  return {k * a[0] * a[0] + c,        k * a[0] * a[1] + s * a[2], k * a[0] * a[2] - s * a[1],
          k * a[0] * a[1] - s * a[2], k * a[1] * a[1] + c,        k * a[1] * a[2] + s * a[0],
          k * a[0] * a[2] + s * a[1], k * a[1] * a[2] - s * a[0], k * a[2] * a[2] + c};
}
namespace detail {
// cgmath Quaternion::from(Matrix3) (Shepperd branches); m column-major, returns (s, x, y, z)
inline std::array<double, 4> quat_from_mat(const Basis3 &m) {
  auto M = [&](int c, int r) { return m[c * 3 + r]; };
  const double trace = (M(0, 0) + M(1, 1)) + M(2, 2);
  if (trace >= 0.0) {
    double s = std::sqrt(1.0 + trace);
    const double w = 0.5 * s;
    s = 0.5 / s;
    return {w, (M(1, 2) - M(2, 1)) * s, (M(2, 0) - M(0, 2)) * s, (M(0, 1) - M(1, 0)) * s};
  }
  if (M(0, 0) > M(1, 1) && M(0, 0) > M(2, 2)) {
    double s = std::sqrt(((M(0, 0) - M(1, 1)) - M(2, 2)) + 1.0);
    const double x = 0.5 * s;
    s = 0.5 / s;
    return {(M(1, 2) - M(2, 1)) * s, x, (M(1, 0) + M(0, 1)) * s, (M(0, 2) + M(2, 0)) * s};
  }
  if (M(1, 1) > M(2, 2)) {
    double s = std::sqrt(((M(1, 1) - M(0, 0)) - M(2, 2)) + 1.0);
    const double y = 0.5 * s;
    s = 0.5 / s;
    return {(M(2, 0) - M(0, 2)) * s, (M(1, 0) + M(0, 1)) * s, y, (M(2, 1) + M(1, 2)) * s};
  }
  double s = std::sqrt(((M(2, 2) - M(0, 0)) - M(1, 1)) + 1.0);
  const double z = 0.5 * s;
  s = 0.5 / s;
  return {(M(0, 1) - M(1, 0)) * s, (M(0, 2) + M(2, 0)) * s, (M(2, 1) + M(1, 2)) * s, z};
}
inline Basis3 mat_from_quat(const std::array<double, 4> &q) {
  const double s = q[0], x = q[1], y = q[2], z = q[3];
  const double x2 = x + x, y2 = y + y, z2 = z + z;
  const double xx2 = x2 * x, xy2 = x2 * y, xz2 = x2 * z, yy2 = y2 * y, yz2 = y2 * z, zz2 = z2 * z;
  const double sy2 = y2 * s, sz2 = z2 * s, sx2 = x2 * s;
  return {1.0 - yy2 - zz2, xy2 + sz2, xz2 - sy2, xy2 - sz2, 1.0 - xx2 - zz2, yz2 + sx2,
          xz2 + sy2, yz2 - sx2, 1.0 - xx2 - yy2};
}
}  // namespace detail

// src/baproblem.rs:78-90
inline Basis3 from_rodrigues(const Vector3 &x) {
  const double theta2 = (x[0] * x[0] + x[1] * x[1]) + x[2] * x[2];
  if (theta2 > 2.220446049250313e-16) {
    const double angle = std::sqrt(theta2), inv = 1.0 / angle;
    return from_axis_angle({x[0] * inv, x[1] * inv, x[2] * inv}, angle);
  }
  return detail::mat_from_quat(detail::quat_from_mat({1.0, x[2], -x[1], -x[2], 1.0, x[0], x[1], -x[0], 1.0}));
}
// src/baproblem.rs:93-102
inline Vector3 to_rodrigues(const Basis3 &R) {
  const auto q = detail::quat_from_mat(R);
  const double angle = 2.0 * std::acos(std::max(-1.0, std::min(1.0, q[0])));
  const double d = 1.0 - q[0] * q[0];
  if (d < 2.220446049250313e-16) return {0.0, 0.0, 0.0};
  const double sd = std::sqrt(d);
  const Vector3 a{q[1] / sd, q[2] / sd, q[3] / sd};
  const double inv = 1.0 / std::sqrt((a[0] * a[0] + a[1] * a[1]) + a[2] * a[2]);
  return {a[0] * inv * angle, a[1] * inv * angle, a[2] * inv * angle};
}

namespace detail {
// approx::ulps_eq! with its defaults (epsilon = f64::EPSILON, max_ulps = 4), as cgmath 0.17 uses it
inline bool ulps_eq(double a, double b) {
  if (std::fabs(a - b) <= 2.220446049250313e-16) return true;
  if (std::signbit(a) != std::signbit(b)) return false;
  int64_t ia, ib;
  std::memcpy(&ia, &a, 8);
  std::memcpy(&ib, &b, 8);
  return (ia > ib ? ia - ib : ib - ia) <= 4;
}
inline Vector3 cross(const Vector3 &a, const Vector3 &b) {
  return {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
}
inline double dot(const Vector3 &a, const Vector3 &b) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }
inline double magnitude(const Vector3 &a) { return std::sqrt(dot(a, a)); }
inline Vector3 normalize(const Vector3 &a) {
  const double inv = 1.0 / magnitude(a);
  return {a[0] * inv, a[1] * inv, a[2] * inv};
}
inline Vector3 sub(const Point3 &a, const Point3 &b) { return {a[0] - b[0], a[1] - b[1], a[2] - b[2]}; }

// The reference draws from rand 0.6.5's thread_rng() (OS-seeded, no seed option anywhere); the
// sequential host-side procedures here take a seed and draw from SplitMix64 instead, so parity with
// the reference is distributional by construction.
struct Rng {
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed) {}
  uint64_t next() {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  double uniform() { return (double)(next() >> 11) * 0x1.0p-53; }          // gen_range(0.0, 1.0)
  double range(double lo, double hi) { return lo + (hi - lo) * uniform(); }  // gen_range(lo, hi)
  size_t below(size_t n) {                                                   // gen_range(0, n)
    const size_t k = (size_t)(uniform() * (double)n);
    return k < n ? k : n - 1;
  }
  bool coin() { return (next() >> 63) != 0; }  // rand::random::<bool>()
  // WeightedIndex::new(w).unwrap().sample(): panics on an empty list, a negative weight or a zero total
  size_t weighted(const std::vector<double> &w) {
    double total = 0.0;
    for (double x : w) {
      if (!(x >= 0.0)) throw std::logic_error("called `Result::unwrap()` on an `Err` value: NegativeWeight");
      total += x;
    }
    if (w.empty()) throw std::logic_error("called `Result::unwrap()` on an `Err` value: NoItem");
    if (!(total > 0.0)) throw std::logic_error("called `Result::unwrap()` on an `Err` value: AllWeightsZero");
    const double t = uniform() * total;
    double acc = 0.0;
    for (size_t i = 0; i < w.size(); ++i) {
      acc += w[i];
      if (t < acc) return i;
    }
    size_t last = w.size() - 1;
    while (last > 0 && w[last] == 0.0) --last;
    return last;
  }
  template <class T>
  void shuffle(std::vector<T> &v) {  // SliceRandom::shuffle (Fisher-Yates from the back)
    for (size_t i = v.size(); i > 1; --i) std::swap(v[i - 1], v[below(i)]);
  }
  // IteratorRandom::choose_multiple over 0..len: reservoir sampling, at most `amount` values, order arbitrary
  std::vector<size_t> choose_multiple(size_t len, size_t amount) {
    std::vector<size_t> r;
    r.reserve(std::min(len, amount));
    for (size_t i = 0; i < len; ++i) {
      if (r.size() < amount)
        r.push_back(i);
      else {
        const size_t k = below(i + 1);
        if (k < amount) r[k] = i;
      }
    }
    return r;
  }
};
}  // namespace detail

// cgmath 0.17 Basis3::between_vectors (through Quaternion::between_vectors), used by the path cameras
// (src/generate.rs:144,200)
inline Basis3 between_vectors(const Vector3 &a, const Vector3 &b) {
  const double k_cos_theta = detail::dot(a, b);
  if (detail::ulps_eq(k_cos_theta, 1.0)) return basis_one();  // same direction
  const double k = std::sqrt(detail::dot(a, a) * detail::dot(b, b));
  if (detail::ulps_eq(k_cos_theta / k, -1.0)) {  // opposite direction: half a turn about an orthogonal axis
    Vector3 orthogonal = detail::cross({1.0, 0.0, 0.0}, a);
    if (detail::ulps_eq(detail::dot(orthogonal, orthogonal), 0.0)) orthogonal = detail::cross({0.0, 1.0, 0.0}, a);
    const Vector3 o = detail::normalize(orthogonal);
    return detail::mat_from_quat({0.0, o[0], o[1], o[2]});
  }
  const Vector3 v = detail::cross(a, b);
  const double s = k + k_cos_theta;
  const double inv = 1.0 / std::sqrt(s * s + detail::dot(v, v));
  return detail::mat_from_quat({s * inv, v[0] * inv, v[1] * inv, v[2] * inv});
}

// ---- SnavelyCamera, src/baproblem.rs:130-225 -------------------------------------------------------
struct SnavelyCamera {
  // the C ABI's record: dir as column-major 3x3 [0..9), loc [9..12), intrin f,k1,k2 [12..15)
  double rec[C2B_CAM_STRIDE];

  // src/baproblem.rs:153-159
  static SnavelyCamera from_position_direction(const Point3 &position, const Basis3 &dir) {
    SnavelyCamera c;
    c2b_camera_from_position_direction(position.data(), dir.data(), c.rec);
    return c;
  }
  // src/baproblem.rs:180-190: [rodrigues 3, translation 3, f, k1, k2]
  static SnavelyCamera from_vec(const std::array<double, 9> &x) {
    SnavelyCamera c;
    const Basis3 R = from_rodrigues({x[0], x[1], x[2]});
    std::copy(R.begin(), R.end(), c.rec);
    for (int k = 0; k < 6; ++k) c.rec[9 + k] = x[3 + k];
    return c;
  }
  // src/baproblem.rs:192-202
  std::array<double, 9> to_vec() const {
    Basis3 R;
    std::copy(rec, rec + 9, R.begin());
    const Vector3 r = to_rodrigues(R);
    return {r[0], r[1], r[2], rec[9], rec[10], rec[11], rec[12], rec[13], rec[14]};
  }
  // src/baproblem.rs:141-143
  Point3 project_world(const Point3 &p) const {
    Point3 o;
    c2b_camera_project_world(rec, p.data(), o.data());
    return o;
  }
  // src/baproblem.rs:145-151
  std::array<double, 2> project(const Point3 &pc) const {
    std::array<double, 2> uv;
    c2b_camera_project(rec, pc.data(), uv.data());
    return uv;
  }
  // Camera::to_world, src/baproblem.rs:117-119: dir^-1 * (p - loc), through the centre helper's
  // general inverse: R^-1 (p - t) = R^-1 p + centre
  Point3 to_world(const Point3 &pc) const {
    // solve R x = pc - t with the cofactor inverse used everywhere else (c2b_camera_center does
    // -(R^-1 t)); x = R^-1 pc + centre
    SnavelyCamera probe = *this;
    probe.rec[9] = -pc[0];
    probe.rec[10] = -pc[1];
    probe.rec[11] = -pc[2];
    const Point3 rinv_pc = probe.center();  // -(R^-1 (-pc)) = R^-1 pc
    const Point3 c = center();
    return {rinv_pc[0] + c[0], rinv_pc[1] + c[1], rinv_pc[2] + c[2]};
  }
  // src/baproblem.rs:161-163
  Point3 center() const {
    Point3 o;
    c2b_camera_center(rec, o.data());
    return o;
  }
  // src/baproblem.rs:165-171
  SnavelyCamera transform(const Basis3 &delta_dir, const Vector3 &delta_loc) const {
    SnavelyCamera c;
    c2b_camera_transform(rec, delta_dir.data(), delta_loc.data(), c.rec);
    return c;
  }
  Basis3 rotation() const {
    Basis3 R;
    std::copy(rec, rec + 9, R.begin());
    return R;
  }
};

// ---- GPU context and scene (where embree_rs::Device / CommittedScene stood) ------------------------
// n_gpus > 1: GPUs device .. device + n_gpus - 1 of this box behind one c2b_multi (one process, camera ranges,
// one NCCL communicator); visibility_graph then runs on all of them and returns the same graph, everything
// else (noise, ray queries, point sampling) runs on the first.
class Context {
 public:
  explicit Context(int device = 0, int n_gpus = 1) {
    if (n_gpus > 1) {
      std::vector<int> dev((size_t)n_gpus);
      for (int g = 0; g < n_gpus; ++g) dev[(size_t)g] = device + g;
      detail::check(c2b_init_multi(n_gpus, dev.data(), &m_));
      h_ = c2b_multi_ctx(m_, 0);
    } else {
      detail::check(c2b_init(device, &h_));
    }
  }
  ~Context() {
    if (m_)
      c2b_shutdown_multi(m_);
    else
      c2b_shutdown(h_);
  }
  Context(const Context &) = delete;
  Context &operator=(const Context &) = delete;
  c2b_ctx *handle() const { return h_; }
  c2b_multi *multi() const { return m_; }
  int num_gpus() const { return m_ ? c2b_multi_num_gpus(m_) : 1; }

 private:
  c2b_ctx *h_ = nullptr;
  c2b_multi *m_ = nullptr;
};

class Scene {
 public:
  // Scene::new + model_to_geometry per model + attach + commit (src/bin/city2ba.rs:515-521);
  // xyz: 3 floats per vertex, tri: 3 indices per triple, all models concatenated
  Scene(const Context &ctx, const std::vector<float> &xyz, const std::vector<uint32_t> &tri) : ctx_(&ctx) {
    if (ctx.multi()) {  // the BVH on every GPU; ray queries go to the first copy
      detail::check(c2b_scene_create_multi(ctx.multi(), xyz.data(), xyz.size() / 3, tri.data(), tri.size() / 3, &ms_));
      h_ = c2b_multi_scene_get(ms_, 0);
    } else {
      detail::check(c2b_scene_create(ctx.handle(), xyz.data(), xyz.size() / 3, tri.data(), tri.size() / 3, &h_));
    }
  }
  ~Scene() {
    if (ms_)
      c2b_scene_destroy_multi(ms_);
    else
      c2b_scene_destroy(h_);
  }
  c2b_multi_scene *multi_handle() const { return ms_; }
  Scene(const Scene &) = delete;
  Scene &operator=(const Scene &) = delete;
  const Context &context() const { return *ctx_; }
  c2b_scene *handle() const { return h_; }
  uint64_t num_triangles() const { return c2b_scene_num_triangles(h_); }
  // scene.bounds(), src/generate.rs:237
  std::pair<std::array<float, 3>, std::array<float, 3>> bounds() const {
    std::array<float, 3> lo, hi;
    detail::check(c2b_scene_bounds(h_, lo.data(), hi.data()));
    return {lo, hi};
  }
  // scene.intersect on one ray, src/generate.rs:253-262: (hit, tfar)
  std::pair<bool, float> intersect(const std::array<float, 3> &org, const std::array<float, 3> &dir) const {
    int hit = 0;
    float t = 0;
    detail::check(c2b_intersect1(ctx_->handle(), h_, org.data(), dir.data(), &hit, &t));
    return {hit != 0, t};
  }
  // the same closest-hit query for a whole batch of rays in one launch (flags = 1 and tfar = distance on a hit)
  void intersect(std::vector<c2b_ray48> &rays) const {
    detail::check(c2b_intersect(ctx_->handle(), h_, rays.data(), rays.size()));
  }

 private:
  const Context *ctx_;
  c2b_scene *h_ = nullptr;
  c2b_multi_scene *ms_ = nullptr;
};

namespace detail {
inline std::vector<double> flatten(const std::vector<SnavelyCamera> &cams) {
  std::vector<double> f(cams.size() * C2B_CAM_STRIDE);
  for (size_t i = 0; i < cams.size(); ++i) std::memcpy(&f[i * C2B_CAM_STRIDE], cams[i].rec, sizeof cams[i].rec);
  return f;
}
inline VisGraph unpack(const c2b_obs &o) {
  VisGraph g(o.n_cameras);
  for (uint64_t c = 0; c < o.n_cameras; ++c) {
    g[c].reserve(o.offsets[c + 1] - o.offsets[c]);
    for (uint64_t i = o.offsets[c]; i < o.offsets[c + 1]; ++i)
      g[c].push_back({(size_t)o.point_idx[i], {o.uv[2 * i], o.uv[2 * i + 1]}});
  }
  return g;
}
inline VisGraph run_visibility(const Context &ctx, const Scene *scene, const std::vector<SnavelyCamera> &cameras,
                               const std::vector<Point3> &points, double max_dist, int occlusion,
                               double block_length, double block_inset, int predicate = C2B_PRED_WATERTIGHT) {
  const std::vector<double> cams = flatten(cameras);
  c2b_vis_options opt;
  c2b_vis_options_default(&opt);
  opt.occlusion = occlusion;
  opt.predicate = predicate;
  opt.block_length = block_length;
  opt.block_inset = block_inset;
  c2b_obs out;
  std::memset(&out, 0, sizeof out);
  if (ctx.multi())
    check(c2b_visibility_graph_multi(ctx.multi(), scene ? scene->multi_handle() : nullptr, cams.data(), cameras.size(),
                                     points.empty() ? nullptr : points[0].data(), points.size(), max_dist, &opt, &out,
                                     nullptr));
  else
    check(c2b_visibility_graph(ctx.handle(), scene ? scene->handle() : nullptr, cams.data(), cameras.size(),
                               points.empty() ? nullptr : points[0].data(), points.size(), max_dist, &opt, &out));
  VisGraph g = unpack(out);
  c2b_obs_free(ctx.handle(), &out);
  return g;
}
}  // namespace detail

// ---- OBJ ingest with the rules of tobj 0.1.12 (Cargo.lock:1149-1150; src/bin/city2ba.rs:481) --------------
// One Model per `o` / `g` statement that is followed by elements; per-model vertex arrays holding only
// the vertices its elements use, in order of first use (de-duplicated by the v/vt/vn index triple);
// triangles as they are, quads as (a,b,c),(a,c,d), larger polygons as a fan from their first vertex;
// `l` records with two vertices append TWO indices and `p` records one (so a model of lines is a list of
// index pairs: what generate_cameras_path reads, and what model_to_geometry regroups into harmless
// degenerate triples when --path is not given, src/generate.rs:74-105).  Materials are not read.
namespace tobj {
struct Mesh {
  std::vector<float> positions;   // 3 per vertex
  std::vector<uint32_t> indices;  // into positions / 3
};
struct Model {
  Mesh mesh;
  std::string name;
};

inline std::vector<Model> load_obj(const std::string &path) {
  std::ifstream f(path);
  if (!f) throw Error(Error::IOError, "Could not open file \"" + path + "\"");
  std::vector<float> pos;
  size_t n_vt = 0, n_vn = 0;
  struct Key {
    int64_t v, vt, vn;
    bool operator==(const Key &o) const { return v == o.v && vt == o.vt && vn == o.vn; }
  };
  struct KeyHash {
    size_t operator()(const Key &k) const {
      return std::hash<int64_t>()(k.v * 1000003 ^ (k.vt + 1) * 10007 ^ (k.vn + 1));
    }
  };
  std::vector<std::vector<Key>> faces;  // elements of the model being read
  std::string name = "unnamed_object";
  std::vector<Model> models;
  auto flush = [&]() {
    if (faces.empty()) return;
    Model m;
    m.name = name;
    std::unordered_map<Key, uint32_t, KeyHash> seen;
    auto add = [&](const Key &k) {
      auto it = seen.find(k);
      if (it == seen.end()) {
        it = seen.emplace(k, (uint32_t)(m.mesh.positions.size() / 3)).first;
        for (int c = 0; c < 3; ++c) m.mesh.positions.push_back(pos[3 * (size_t)k.v + c]);
      }
      m.mesh.indices.push_back(it->second);
    };
    for (const auto &e : faces) {
      if (e.size() <= 3) {  // point, line, triangle
        for (const auto &k : e) add(k);
      } else if (e.size() == 4) {
        for (int i : {0, 1, 2, 0, 2, 3}) add(e[i]);
      } else {
        for (size_t i = 1; i + 1 < e.size(); ++i) {
          add(e[0]);
          add(e[i]);
          add(e[i + 1]);
        }
      }
    }
    models.push_back(std::move(m));
    faces.clear();
  };
  std::string line;
  size_t lineno = 0;
  auto bad = [&](const char *what) {
    return Error(Error::IOError, "Load error: " + std::string(what) + " (" + path + ":" + std::to_string(lineno) + ")");
  };
  while (std::getline(f, line)) {
    ++lineno;
    std::istringstream ls(line);
    std::string tag;
    if (!(ls >> tag) || tag[0] == '#') continue;
    if (tag == "v") {
      float x, y, z;
      if (!(ls >> x >> y >> z)) throw bad("position parse error");
      pos.insert(pos.end(), {x, y, z});
    } else if (tag == "vt") {
      ++n_vt;
    } else if (tag == "vn") {
      ++n_vn;
    } else if (tag == "f" || tag == "l" || tag == "p") {
      std::vector<Key> e;
      std::string tok;
      while (ls >> tok) {
        int64_t idx[3] = {0, 0, 0};
        size_t k = 0, start = 0;
        while (k < 3 && start <= tok.size()) {
          const size_t slash = tok.find('/', start);
          const std::string part = tok.substr(start, slash == std::string::npos ? std::string::npos : slash - start);
          if (!part.empty()) {
            char *end = nullptr;
            idx[k] = std::strtoll(part.c_str(), &end, 10);
            if (*end) throw bad("face parse error");
          }
          ++k;
          if (slash == std::string::npos) break;
          start = slash + 1;
        }
        // 1-based; negative = relative to what has been read so far; 0 = absent
        auto fix = [&](int64_t i, size_t n) -> int64_t { return i > 0 ? i - 1 : i < 0 ? (int64_t)n + i : -1; };
        const Key key{fix(idx[0], pos.size() / 3), fix(idx[1], n_vt), fix(idx[2], n_vn)};
        if (key.v < 0 || (size_t)key.v >= pos.size() / 3) throw bad("face vertex index out of range");
        e.push_back(key);
      }
      if (e.empty()) throw bad("face parse error");
      faces.push_back(std::move(e));
    } else if (tag == "o" || tag == "g") {
      flush();
      std::string rest;
      std::getline(ls, rest);
      const size_t a = rest.find_first_not_of(" \t\r"), b = rest.find_last_not_of(" \t\r");
      name = a == std::string::npos ? "unnamed_object" : rest.substr(a, b - a + 1);
    }
    // mtllib / usemtl / s and anything else: ignored
  }
  flush();
  return models;
}
}  // namespace tobj

namespace detail {
// all models as ONE vertex / index-triple array for c2b_scene_create and the point sampler: each model's
// index list is regrouped into triples on its own (num_tri = indices.len() / 3, src/generate.rs:78) and
// offset by the vertices that precede it
inline void concat_models(const std::vector<tobj::Model> &models, std::vector<float> &xyz, std::vector<uint32_t> &tri) {
  xyz.clear();
  tri.clear();
  for (const auto &m : models) {
    const uint32_t base = (uint32_t)(xyz.size() / 3);
    xyz.insert(xyz.end(), m.mesh.positions.begin(), m.mesh.positions.end());
    const size_t n = m.mesh.indices.size() / 3 * 3;
    for (size_t i = 0; i < n; ++i) tri.push_back(base + m.mesh.indices[i]);
  }
}
// Poisson-disk samples in the unit square.  The reference asks the `poisson` crate (0.10.1, Ebeida's
// maximal sampler) for `samples` points at relative radius 1.0, i.e. the largest radius at which that
// many discs could still be packed; the crate is not vendored, so this is Bridson's dart throwing
// (30 attempts per active sample) at the hexagonal-packing radius for `samples` discs.  Like the
// crate it yields noticeably fewer than `samples` points ("x2 seems to get us closer to the desired
// amount", src/generate.rs:230).  Distributional parity only.
inline std::vector<std::array<double, 2>> poisson_disk(size_t samples, Rng &rng) {
  std::vector<std::array<double, 2>> out;
  if (samples == 0) return out;
  const double r = 2.0 * std::sqrt(0.9068996821171089 / ((double)samples * 3.141592653589793));
  const double cell = r / std::sqrt(2.0);
  const int n = std::max(1, (int)std::ceil(1.0 / cell));
  std::vector<int> grid((size_t)n * n, -1);
  auto cell_of = [&](double x) { return std::min(n - 1, (int)(x / cell)); };
  auto fits = [&](double x, double y) {
    const int cx = cell_of(x), cy = cell_of(y);
    for (int j = std::max(0, cy - 2); j <= std::min(n - 1, cy + 2); ++j)
      for (int i = std::max(0, cx - 2); i <= std::min(n - 1, cx + 2); ++i) {
        const int k = grid[(size_t)j * n + i];
        if (k >= 0) {
          const double dx = out[k][0] - x, dy = out[k][1] - y;
          if (dx * dx + dy * dy < r * r) return false;
        }
      }
    return true;
  };
  std::vector<int> active;
  auto push = [&](double x, double y) {
    grid[(size_t)cell_of(y) * n + cell_of(x)] = (int)out.size();
    active.push_back((int)out.size());
    out.push_back({x, y});
  };
  push(rng.uniform(), rng.uniform());
  while (!active.empty()) {
    const size_t a = rng.below(active.size());
    const auto base = out[active[a]];
    bool placed = false;
    for (int attempt = 0; attempt < 30 && !placed; ++attempt) {
      const double ang = rng.range(0.0, 6.283185307179586), rad = r * std::sqrt(rng.range(1.0, 4.0));
      const double x = base[0] + rad * std::cos(ang), y = base[1] + rad * std::sin(ang);
      if (x < 0.0 || x >= 1.0 || y < 0.0 || y >= 1.0 || !fits(x, y)) continue;
      push(x, y);
      placed = true;
    }
    if (!placed) {
      active[a] = active.back();
      active.pop_back();
    }
  }
  return out;
}
inline std::vector<std::pair<Point3, Point3>> path_segments(const tobj::Model &path) {
  std::vector<Point3> v;
  for (size_t i = 0; i + 2 < path.mesh.positions.size(); i += 3)
    v.push_back({(double)path.mesh.positions[i], (double)path.mesh.positions[i + 1], (double)path.mesh.positions[i + 2]});
  std::vector<std::pair<Point3, Point3>> seg;
  for (size_t i = 0; i + 1 < path.mesh.indices.size(); i += 2)
    seg.push_back({v.at(path.mesh.indices[i]), v.at(path.mesh.indices[i + 1])});
  return seg;
}
}  // namespace detail

namespace generate {
// src/generate.rs:424-481.  Per camera: every point within max_dist, in front, inside the frustum and
// not occluded by the scene, in ascending point order, with its projection.
// predicate: C2B_PRED_WATERTIGHT (default) or C2B_PRED_MT, the Moeller-Trumbore test of Embree's default
// intersector — what the reference's scene runs (not in the reference's signature).
inline VisGraph visibility_graph(const Scene &scene, const std::vector<SnavelyCamera> &cameras,
                                 const std::vector<Point3> &points, double max_dist, bool /*verbose*/,
                                 int predicate = C2B_PRED_WATERTIGHT) {
  return detail::run_visibility(scene.context(), &scene, cameras, points, max_dist, C2B_OCC_MESH, 20.0, 1.0, predicate);
}

// src/generate.rs:356-420 (seeded; the reference draws from thread_rng())
inline std::vector<Point3> generate_world_points_uniform(const Context &ctx, const std::vector<float> &xyz,
                                                         const std::vector<uint32_t> &tri,
                                                         const std::vector<SnavelyCamera> &cameras,
                                                         size_t num_points, double max_dist, uint64_t seed) {
  detail::require(!cameras.empty(), "Cannot generate world points with 0 cameras. Try increasing the number of "
                                    "cameras generated (via --cameras).");
  const std::vector<double> cams = detail::flatten(cameras);
  std::vector<Point3> pts(num_points);
  uint64_t n = 0;
  const int rc = c2b_generate_world_points_uniform(ctx.handle(), xyz.data(), xyz.size() / 3, tri.data(), tri.size() / 3,
                                                   cams.data(), cameras.size(), num_points, max_dist, seed,
                                                   num_points ? pts[0].data() : nullptr, &n);
  if (rc != C2B_OK) throw std::logic_error(c2b_last_error());  // the reference panics
  pts.resize(n);
  return pts;
}

// the call sequence of src/bin/city2ba.rs:515-521 (Device::new, Scene::new, model_to_geometry per model,
// attach_geometry, commit) in one step
inline Scene commit_scene(const Context &ctx, const std::vector<tobj::Model> &models) {
  std::vector<float> xyz;
  std::vector<uint32_t> tri;
  detail::concat_models(models, xyz, tri);
  return Scene(ctx, xyz, tri);
}

// src/generate.rs:356-420 with the reference's `&[tobj::Model]` argument
inline std::vector<Point3> generate_world_points_uniform(const Context &ctx, const std::vector<tobj::Model> &models,
                                                         const std::vector<SnavelyCamera> &cameras,
                                                         size_t num_points, double max_dist, uint64_t seed) {
  std::vector<float> xyz;
  std::vector<uint32_t> tri;
  detail::concat_models(models, xyz, tri);
  return generate_world_points_uniform(ctx, xyz, tri, cameras, num_points, max_dist, seed);
}

// src/generate.rs:109-148: cameras at random positions along a path (segments weighted by length),
// looking along the direction of travel
inline std::vector<SnavelyCamera> generate_cameras_path(const Scene & /*scene*/, const tobj::Model &path,
                                                        size_t num_cameras, uint64_t seed) {
  const auto paths = detail::path_segments(path);
  std::vector<double> lengths;
  for (const auto &[x, y] : paths) lengths.push_back(detail::magnitude(detail::sub(y, x)));
  detail::Rng rng(seed);
  std::vector<SnavelyCamera> cams;
  for (size_t n = 0; n < num_cameras; ++n) {
    const size_t i = rng.weighted(lengths);
    const auto &[x, y] = paths[i];
    const double d = rng.uniform();
    const Vector3 dir = detail::sub(y, x);
    const Point3 pos{x[0] + d * dir[0], x[1] + d * dir[1], x[2] + d * dir[2]};
    cams.push_back(SnavelyCamera::from_position_direction(pos, between_vectors(detail::normalize(dir), {0.0, 0.0, -1.0})));
  }
  return cams;
}

// src/generate.rs:152-213: fixed steps from the start of the path
inline std::vector<SnavelyCamera> generate_cameras_path_step(const Scene & /*scene*/, const tobj::Model &path,
                                                             size_t num_cameras, double step_size,
                                                             std::ostream *log = nullptr) {
  const auto paths = detail::path_segments(path);
  double total_length = 0.0;
  for (const auto &[x, y] : paths) total_length += detail::magnitude(detail::sub(y, x));
  if (!((double)num_cameras * step_size <= total_length)) {
    std::ostringstream m;
    m << "Length of path " << total_length << " is less than the number of cameras (" << num_cameras
      << ") times the step size (" << step_size << ") " << (double)num_cameras * step_size;
    throw std::logic_error(m.str());
  }
  if (log)
    *log << "Generating cameras along path. Path length: " << total_length << ", using "
         << (double)num_cameras * step_size << " of it.\n";
  size_t segment_index = 0;
  double dist = 0.0;
  std::vector<SnavelyCamera> cams;
  for (size_t n = 0; n < num_cameras; ++n) {
    detail::require(segment_index < paths.size(), "index out of bounds: the path ended before the last camera");
    Vector3 dir = detail::sub(paths[segment_index].second, paths[segment_index].first);
    const Point3 &start = paths[segment_index].first;
    const double t = dist / detail::magnitude(dir);
    cams.push_back(SnavelyCamera::from_position_direction({start[0] + t * dir[0], start[1] + t * dir[1], start[2] + t * dir[2]},
                                                          between_vectors(detail::normalize(dir), {0.0, 0.0, -1.0})));
    dist += step_size;
    while (dist >= detail::magnitude(dir)) {
      segment_index += 1;
      dist -= detail::magnitude(dir);
      // the reference indexes paths[segment_index] here, so a last step that lands exactly on the end of
      // the path panics there as well
      detail::require(segment_index < paths.size(), "index out of bounds: the path ended before the last camera");
      dir = detail::sub(paths[segment_index].second, paths[segment_index].first);
    }
  }
  return cams;
}

// src/generate.rs:217-280: Poisson-disk positions over the scene's (x, z) bounds, each dropped onto the
// tallest surface below it (closest hit of a ray straight down — ALL rays in one GPU batch instead of
// one rtcIntersect1 per sample) and raised by `height`; kept if pt[2] < lower_y + ground (the
// reference compares z, not y, :264 — kept as written); random yaw about y.
inline std::vector<SnavelyCamera> generate_cameras_poisson(const Scene &scene, size_t num_points, double height,
                                                           double ground, uint64_t seed) {
  detail::Rng rng(seed);
  const auto samples = detail::poisson_disk(num_points * 2, rng);
  const auto [lo, hi] = scene.bounds();
  const Point3 start{(double)hi[0], (double)hi[1] + 0.1, (double)hi[2]};
  const Vector3 delta{(double)(hi[0] - lo[0]), 0.0, (double)(hi[2] - lo[2])};
  std::vector<Point3> origins;
  std::vector<c2b_ray48> rays;
  for (const auto &smp : samples) {
    const Point3 o{start[0] - delta[0] * smp[0], start[1] - delta[1] * 0.0, start[2] - delta[2] * smp[1]};
    origins.push_back(o);
    c2b_ray48 r;
    std::memset(&r, 0, sizeof r);
    r.org_x = (float)o[0];
    r.org_y = (float)o[1];
    r.org_z = (float)o[2];
    r.dir_y = -1.0f;
    r.tfar = INFINITY;
    r.mask = 0xffffffffu;
    rays.push_back(r);
  }
  if (!rays.empty()) scene.intersect(rays);
  std::vector<SnavelyCamera> cams;
  for (size_t i = 0; i < rays.size(); ++i) {
    if (!rays[i].flags) continue;
    const Point3 pt{origins[i][0], origins[i][1] - (double)rays[i].tfar + height, origins[i][2]};
    if (pt[2] < (double)lo[1] + ground)
      cams.push_back(SnavelyCamera::from_position_direction(pt, from_angle_y(rng.range(0.0, 2.0 * 3.141592653589793))));
  }
  return cams;
}

// src/generate.rs:484-527: translate all models so that the minimum corner of their bounding box is the origin
inline std::vector<tobj::Model> move_to_origin(std::vector<tobj::Model> models) {
  float mn[3] = {INFINITY, INFINITY, INFINITY};
  bool any = false;
  for (const auto &m : models)
    for (size_t i = 0; i + 2 < m.mesh.positions.size(); i += 3) {
      any = true;
      for (int k = 0; k < 3; ++k) mn[k] = std::fmin(mn[k], m.mesh.positions[i + k]);
    }
  detail::require(any, "called `Option::unwrap()` on a `None` value");  // fold1 of nothing
  for (auto &m : models)
    for (size_t i = 0; i + 2 < m.mesh.positions.size(); i += 3)
      for (int k = 0; k < 3; ++k) m.mesh.positions[i + k] -= mn[k];
  return models;
}

// src/generate.rs:530-544: intrinsics uniform in [intrinsic_start, intrinsic_end)
inline void modify_intrinsics(std::vector<SnavelyCamera> &cameras, const Vector3 &intrinsic_start,
                              const Vector3 &intrinsic_end, uint64_t seed) {
  detail::Rng rng(seed);
  for (auto &c : cameras)
    for (int k = 0; k < 3; ++k) {
      const double v = rng.uniform();
      c.rec[12 + k] = intrinsic_start[k] + v * (intrinsic_end[k] - intrinsic_start[k]);
    }
}
}  // namespace generate

// ---- BAProblem, src/baproblem.rs:256-801 --------------------------------------------------------------
struct BAProblem {
  std::vector<SnavelyCamera> cameras;
  std::vector<Point3> points;
  VisGraph vis_graph;

  // src/baproblem.rs:360-376
  static BAProblem from_visibility(std::vector<SnavelyCamera> cams, std::vector<Point3> points, VisGraph obs) {
    detail::require(cams.size() == obs.size(), "assertion failed: cams.len() == obs.len()");
    for (const auto &o : obs)
      for (const auto &e : o) detail::require(e.first < points.size(), "assertion failed: ci < &points.len()");
    return BAProblem{std::move(cams), std::move(points), std::move(obs)};
  }
  size_t num_points() const { return points.size(); }
  size_t num_cameras() const { return cameras.size(); }
  size_t num_observations() const {
    size_t n = 0;
    for (const auto &v : vis_graph) n += v.size();
    return n;
  }

  // src/baproblem.rs:265-279
  double total_reprojection_error(double norm) const {
    double total = 0.0;
    for (size_t c = 0; c < cameras.size(); ++c) {
      double s = 0.0;
      for (const auto &[o, uv] : vis_graph[c]) {
        const auto p = cameras[c].project(cameras[c].project_world(points[o]));
        s += std::pow(std::fabs(p[0] - uv.first), norm) + std::pow(std::fabs(p[1] - uv.second), norm);
      }
      total += s;
    }
    return std::pow(total, 1.0 / norm);
  }

  // src/baproblem.rs:282-304 (sequential folds over camera centres, then points)
  Vector3 mean() const {
    const double num = (double)(cameras.size() + points.size());
    Vector3 a{0, 0, 0};
    auto add = [&](const Point3 &b) {
      for (int k = 0; k < 3; ++k) a[k] = a[k] + b[k] / num;
    };
    for (const auto &c : cameras) add(c.center());
    for (const auto &p : points) add(p);
    return a;
  }
  Vector3 std() const {
    const double num = (double)(cameras.size() + points.size());
    const Vector3 m = mean();
    Vector3 a{0, 0, 0};
    auto add = [&](const Point3 &x) {
      for (int k = 0; k < 3; ++k) a[k] = a[k] + (x[k] - m[k]) * (x[k] - m[k]);
    };
    for (const auto &c : cameras) add(c.center());
    for (const auto &p : points) add(p);
    return {std::sqrt(a[0] / num), std::sqrt(a[1] / num), std::sqrt(a[2] / num)};
  }
  // src/baproblem.rs:307-337
  std::pair<Vector3, Vector3> extent() const {
    Vector3 lo{INFINITY, INFINITY, INFINITY}, hi{-INFINITY, -INFINITY, -INFINITY};
    auto add = [&](const Point3 &x) {
      for (int k = 0; k < 3; ++k) {
        lo[k] = std::fmin(lo[k], x[k]);
        hi[k] = std::fmax(hi[k], x[k]);
      }
    };
    for (const auto &c : cameras) add(c.center());
    for (const auto &p : points) add(p);
    return {lo, hi};
  }
  Vector3 dimensions() const {
    const auto e = extent();
    return {e.second[0] - e.first[0], e.second[1] - e.first[1], e.second[2] - e.first[2]};
  }

  // src/baproblem.rs:394-423
  BAProblem subset(const std::vector<size_t> &ci, const std::vector<size_t> &pi) const {
    BAProblem out;
    for (size_t i : ci) out.cameras.push_back(cameras[i]);
    for (size_t i : pi) out.points.push_back(points[i]);
    std::vector<int64_t> point_indices(points.size(), -1);
    for (size_t i = 0; i < pi.size(); ++i) point_indices[pi[i]] = (int64_t)i;
    for (size_t i : ci) {
      std::vector<Observation> o;
      for (const auto &e : vis_graph[i])
        if (point_indices[e.first] >= 0) o.push_back({(size_t)point_indices[e.first], e.second});
      out.vis_graph.push_back(std::move(o));
    }
    return out;
  }
  // src/baproblem.rs:426-453: cameras need > 3 observations, points > 1
  BAProblem remove_singletons() const {
    std::vector<size_t> ci, pi;
    for (size_t i = 0; i < vis_graph.size(); ++i)
      if (vis_graph[i].size() > 3) ci.push_back(i);
    std::vector<int64_t> count(points.size(), 0);
    for (const auto &obs : vis_graph)
      for (const auto &e : obs) count[e.first] += 1;
    for (size_t i = 0; i < count.size(); ++i)
      if (count[i] > 1) pi.push_back(i);
    return subset(ci, pi);
  }
  // src/baproblem.rs:456-534.  Kept as written there, including the observation filter at :523 that
  // looks up sets[point index] WITHOUT the camera offset: an observation of point i by a camera of
  // the component is dropped when entity i of the combined (cameras, then points) numbering lies
  // outside the component.  Ties between equally large components: lowest set label here (hash-map
  // order in the reference, i.e. unspecified).
  BAProblem largest_connected_component() const {
    if (num_cameras() == 0) return *this;
    const size_t nc = num_cameras(), np = num_points();
    std::vector<size_t> parent(nc + np);
    std::iota(parent.begin(), parent.end(), 0);
    auto find = [&](size_t x) {
      while (parent[x] != x) {
        parent[x] = parent[parent[x]];
        x = parent[x];
      }
      return x;
    };
    for (size_t i = 0; i < nc; ++i)
      for (const auto &e : vis_graph[i]) {
        const size_t a = find(i), b = find(e.first + nc);
        if (a != b) parent[std::max(a, b)] = std::min(a, b);
      }
    std::vector<size_t> sets(nc + np);
    std::unordered_map<size_t, size_t> size_of;
    for (size_t i = 0; i < nc + np; ++i) size_of[sets[i] = find(i)] += 1;
    size_t lcc = 0, best = 0;
    for (const auto &[label, n] : size_of)
      if (n > best || (n == best && label < lcc)) {
        best = n;
        lcc = label;
      }
    BAProblem out;
    std::unordered_map<size_t, size_t> point_map;
    for (size_t i = 0; i < np; ++i)
      if (sets[nc + i] == lcc) {
        point_map[i] = out.points.size();
        out.points.push_back(points[i]);
      }
    for (size_t i = 0; i < nc; ++i) {
      if (sets[i] != lcc) continue;
      out.cameras.push_back(cameras[i]);
      std::vector<Observation> o;
      for (const auto &e : vis_graph[i])
        if (sets[e.first] == lcc) o.push_back({point_map.at(e.first), e.second});
      out.vis_graph.push_back(std::move(o));
    }
    return out;
  }
  // src/baproblem.rs:538-549
  BAProblem cull() const {
    size_t nc = num_cameras(), np = num_points();
    BAProblem culled = largest_connected_component().remove_singletons();
    while (culled.num_cameras() != nc || culled.num_points() != np) {
      nc = culled.num_cameras();
      np = culled.num_points();
      culled = culled.largest_connected_component().remove_singletons();
    }
    return culled;
  }
  // the same on the GPU (c2b_cull_problem): identical result, bit for bit.  stats (optional) receives the
  // call's sizes, iteration count and device times.
  BAProblem cull(const Context &ctx, c2b_cull_stats *stats = nullptr) const {
    const size_t nc = num_cameras();
    std::vector<double> cams(nc * C2B_CAM_STRIDE);
    for (size_t i = 0; i < nc; ++i) std::memcpy(&cams[i * C2B_CAM_STRIDE], cameras[i].rec, sizeof cameras[i].rec);
    std::vector<double> pts(points.size() * 3);
    for (size_t i = 0; i < points.size(); ++i) std::memcpy(&pts[3 * i], points[i].data(), 3 * sizeof(double));
    std::vector<uint64_t> offsets(nc + 1, 0);
    for (size_t i = 0; i < nc; ++i) offsets[i + 1] = offsets[i] + vis_graph[i].size();
    std::vector<uint32_t> idx(offsets[nc]);
    std::vector<double> uv(2 * offsets[nc]);
    for (size_t i = 0, k = 0; i < nc; ++i)
      for (const auto &e : vis_graph[i]) {
        detail::require(e.first <= 0xffffffffull, "point index does not fit 32 bits");
        idx[k] = (uint32_t)e.first;
        uv[2 * k] = e.second.first;
        uv[2 * k + 1] = e.second.second;
        ++k;
      }
    c2b_cull_stats st;
    detail::check(c2b_cull_problem(ctx.handle(), cams.data(), nc, pts.data(), points.size(), offsets.data(), idx.data(),
                                   uv.data(), &st));
    if (stats) *stats = st;
    BAProblem out;
    out.cameras.resize(st.n_cameras);
    for (size_t i = 0; i < st.n_cameras; ++i) std::memcpy(out.cameras[i].rec, &cams[i * C2B_CAM_STRIDE], sizeof out.cameras[i].rec);
    out.points.resize(st.n_points);
    for (size_t i = 0; i < st.n_points; ++i) std::memcpy(out.points[i].data(), &pts[3 * i], 3 * sizeof(double));
    out.vis_graph.resize(st.n_cameras);
    for (size_t i = 0; i < st.n_cameras; ++i) {
      out.vis_graph[i].reserve(offsets[i + 1] - offsets[i]);
      for (uint64_t k = offsets[i]; k < offsets[i + 1]; ++k) out.vis_graph[i].push_back({(size_t)idx[k], {uv[2 * k], uv[2 * k + 1]}});
    }
    return out;
  }

  // ---- BAL I/O, src/baproblem.rs:580-785 ----
  // Rust's `{}` for f64: shortest digits that round-trip, positional (never an exponent)
  static std::string fmt(double x) {
    char buf[400];
    const auto r = std::to_chars(buf, buf + sizeof buf, x, std::chars_format::fixed);
    return std::string(buf, r.ptr);
  }
  // src/baproblem.rs:709-733
  void write_text(const std::string &path) const {
    std::ofstream f(path);
    if (!f) throw Error(Error::IOError, "cannot create " + path);
    f << num_cameras() << ' ' << num_points() << ' ' << num_observations() << '\n';
    for (size_t c = 0; c < vis_graph.size(); ++c)
      for (const auto &[p, uv] : vis_graph[c]) f << c << ' ' << p << ' ' << fmt(uv.first) << ' ' << fmt(uv.second) << '\n';
    for (const auto &c : cameras) {
      const auto v = c.to_vec();
      for (int k = 0; k < 9; ++k) f << (k ? " " : "") << fmt(v[k]);
      f << '\n';
    }
    for (const auto &p : points) f << fmt(p[0]) << ' ' << fmt(p[1]) << ' ' << fmt(p[2]) << '\n';
    if (!f) throw Error(Error::IOError, "write failed: " + path);
  }
  // src/baproblem.rs:736-764: big-endian u64 / f64, per-camera count-prefixed observation lists
  void write_binary(const std::string &path) const {
    std::ofstream f(path, std::ios::binary);
    if (!f) throw Error(Error::IOError, "cannot create " + path);
    auto put64 = [&](uint64_t v) {
      unsigned char b[8];
      for (int k = 0; k < 8; ++k) b[k] = (unsigned char)(v >> (56 - 8 * k));
      f.write(reinterpret_cast<const char *>(b), 8);
    };
    auto putf = [&](double d) {
      uint64_t v;
      std::memcpy(&v, &d, 8);
      put64(v);
    };
    put64(num_cameras());
    put64(num_points());
    put64(num_observations());
    for (const auto &obs : vis_graph) {
      put64(obs.size());
      for (const auto &[p, uv] : obs) {
        put64(p);
        putf(uv.first);
        putf(uv.second);
      }
    }
    for (const auto &c : cameras)
      for (double v : c.to_vec()) putf(v);
    for (const auto &p : points)
      for (double v : p) putf(v);
    if (!f) throw Error(Error::IOError, "write failed: " + path);
  }
  // src/baproblem.rs:768-785: the extension picks the format
  static c2b_bal_format bal_format(const std::string &path) {
    const auto dot = path.rfind('.');
    const std::string ext = dot == std::string::npos ? "" : path.substr(dot + 1);
    if (ext == "bal") return C2B_BAL_TEXT;
    if (ext == "bbal") return C2B_BAL_BINARY;
    throw Error(Error::IOError, "unknown file extension: " + path);
  }
  void write(const std::string &path) const {
    if (bal_format(path) == C2B_BAL_TEXT)
      write_text(path);
    else
      write_binary(path);
  }
  // the same file encoded on the GPU and streamed to disk (c2b_write_bal).  The bytes are the reference's, which
  // write_text's std::to_chars does not give for |values| >= 2^53 and NaN (DESIGN.md, BAL files); the camera vectors
  // are to_vec's, bit for bit.  stats (optional) receives bytes, chunks and the encode / D2H / write times.
  void write(const Context &ctx, const std::string &path, c2b_bal_stats *stats = nullptr) const {
    const c2b_bal_format format = bal_format(path);
    const size_t nc = num_cameras();
    std::vector<double> cams(nc * C2B_CAM_STRIDE);
    for (size_t i = 0; i < nc; ++i) std::memcpy(&cams[i * C2B_CAM_STRIDE], cameras[i].rec, sizeof cameras[i].rec);
    std::vector<double> pts(points.size() * 3);
    for (size_t i = 0; i < points.size(); ++i) std::memcpy(&pts[3 * i], points[i].data(), 3 * sizeof(double));
    std::vector<uint64_t> offsets(nc + 1, 0);
    for (size_t i = 0; i < nc; ++i) offsets[i + 1] = offsets[i] + vis_graph[i].size();
    std::vector<uint32_t> idx(offsets[nc]);
    std::vector<double> uv(2 * offsets[nc]);
    for (size_t i = 0, k = 0; i < nc; ++i)
      for (const auto &e : vis_graph[i]) {
        detail::require(e.first <= 0xffffffffull, "point index does not fit 32 bits");
        idx[k] = (uint32_t)e.first;
        uv[2 * k] = e.second.first;
        uv[2 * k + 1] = e.second.second;
        ++k;
      }
    c2b_bal_stats st;
    detail::check(c2b_write_bal(ctx.handle(), path.c_str(), format, cams.data(), nc, pts.data(), points.size(),
                                offsets.data(), idx.data(), uv.data(), &st));
    if (stats) *stats = st;
  }
  // src/baproblem.rs:580-706
  static BAProblem from_file(const std::string &path) {
    const auto dot = path.rfind('.');
    const std::string ext = dot == std::string::npos ? "" : path.substr(dot + 1);
    BAProblem ba;
    if (ext == "bal") {
      std::ifstream f(path);
      if (!f) throw Error(Error::IOError, "cannot open " + path);
      // file size bounds every count (a camera takes >= 18 bytes, a point >= 6, an observation >= 8): a
      // malformed header is a ParseError (src/baproblem.rs:580-628 fails in nom), never a huge allocation
      f.seekg(0, std::ios::end);
      const uint64_t fsize = (uint64_t)f.tellg();
      f.seekg(0);
      // nom's digit1 takes digits only: a sign ("-1" would wrap in operator>>) is a parse error
      auto getu = [&](size_t &out) {
        f >> std::ws;
        const int ch = f.peek();
        if (ch < '0' || ch > '9') return false;
        if (!(f >> out)) return false;
        const int next = f.peek();  // "1.5" or "1e3" is not an index
        return next == std::char_traits<char>::eof() || std::isspace(next);
      };
      size_t nc, np, no;
      if (!(getu(nc) && getu(np) && getu(no))) throw Error(Error::ParseError, "bad BAL header");
      if (nc > fsize / 18 || np > fsize / 6 || no > fsize / 8)
        throw Error(Error::ParseError, "BAL header counts exceed the file size");
      ba.vis_graph.assign(nc, {});
      for (size_t i = 0; i < no; ++i) {
        size_t c, p;
        double u, v;
        if (!(getu(c) && getu(p) && (f >> u >> v))) throw Error(Error::ParseError, "bad observation line");
        detail::require(c < nc && p < np, "observation index out of range");
        ba.vis_graph[c].push_back({p, {u, v}});
      }
      for (size_t i = 0; i < nc; ++i) {
        std::array<double, 9> x;
        for (auto &t : x)
          if (!(f >> t)) throw Error(Error::ParseError, "bad camera line");
        ba.cameras.push_back(SnavelyCamera::from_vec(x));
      }
      for (size_t i = 0; i < np; ++i) {
        Point3 p;
        for (auto &t : p)
          if (!(f >> t)) throw Error(Error::ParseError, "bad point line");
        ba.points.push_back(p);
      }
    } else if (ext == "bbal") {
      std::ifstream f(path, std::ios::binary);
      if (!f) throw Error(Error::IOError, "cannot open " + path);
      auto get64 = [&]() {
        unsigned char b[8];
        if (!f.read(reinterpret_cast<char *>(b), 8)) throw Error(Error::ParseError, "truncated binary BAL file");
        uint64_t v = 0;
        for (int k = 0; k < 8; ++k) v = (v << 8) | b[k];
        return v;
      };
      auto getf = [&]() {
        const uint64_t v = get64();
        double d;
        std::memcpy(&d, &v, 8);
        return d;
      };
      f.seekg(0, std::ios::end);
      const uint64_t fsize = (uint64_t)f.tellg();
      f.seekg(0);
      const uint64_t nc = get64(), np = get64(), no = get64();
      // 8 + 72 bytes per camera, 24 per point, 24 per observation (src/baproblem.rs:736-764)
      if (nc > fsize / 80 || np > fsize / 24 || no > fsize / 24)
        throw Error(Error::ParseError, "binary BAL header counts exceed the file size");
      size_t seen = 0;
      ba.vis_graph.assign(nc, {});
      for (uint64_t c = 0; c < nc; ++c) {
        const uint64_t n = get64();
        if (n > no - seen) throw Error(Error::ParseError, "observation count does not match the header");
        for (uint64_t i = 0; i < n; ++i) {
          const uint64_t p = get64();
          const double u = getf(), v = getf();
          detail::require(p < np, "observation index out of range");
          ba.vis_graph[c].push_back({(size_t)p, {u, v}});
        }
        seen += n;
      }
      if (seen != no) throw Error(Error::ParseError, "observation count does not match the header");
      for (uint64_t i = 0; i < nc; ++i) {
        std::array<double, 9> x;
        for (auto &t : x) t = getf();
        ba.cameras.push_back(SnavelyCamera::from_vec(x));
      }
      for (uint64_t i = 0; i < np; ++i) {
        Point3 p;
        for (auto &t : p) t = getf();
        ba.points.push_back(p);
      }
    } else {
      throw Error(Error::IOError, "unknown file extension: " + path);
    }
    return ba;  // possibly empty, like the reference's from_file; EmptyProblem is run_generate's (src/bin/city2ba.rs:550-554)
  }
  // the same file parsed on the GPU (c2b_read_bal_resident): it becomes the ctx's resident problem, then the cameras,
  // points and CSR are downloaded.  Errors as above: Error::ParseError, Error::IOError, std::logic_error for an
  // observation index out of range.  stats (optional) receives sizes, chunks, slow tokens and the read / copy / parse
  // times.
  static BAProblem from_file(const Context &ctx, const std::string &path, c2b_bal_read_stats *stats = nullptr) {
    const c2b_bal_format format = bal_format(path);
    c2b_bal_read_stats st;
    const int rc = c2b_read_bal_resident(ctx.handle(), path.c_str(), format, &st);
    if (rc == C2B_ERR_INVALID && std::strstr(c2b_last_error(), "index out of range"))
      throw std::logic_error(c2b_last_error());
    detail::check(rc);
    if (stats) *stats = st;
    BAProblem ba;
    std::vector<double> cams(st.n_cameras * C2B_CAM_STRIDE), pts(st.n_points * 3);
    detail::check(c2b_download_problem(ctx.handle(), cams.data(), pts.data()));
    ba.cameras.resize(st.n_cameras);
    for (size_t i = 0; i < st.n_cameras; ++i) std::memcpy(ba.cameras[i].rec, &cams[i * C2B_CAM_STRIDE], sizeof ba.cameras[i].rec);
    ba.points.resize(st.n_points);
    for (size_t i = 0; i < st.n_points; ++i) std::memcpy(ba.points[i].data(), &pts[3 * i], 3 * sizeof(double));
    c2b_obs obs;
    detail::check(c2b_download_obs(ctx.handle(), &obs));
    ba.vis_graph.resize(st.n_cameras);
    for (size_t i = 0; i < st.n_cameras; ++i) {
      ba.vis_graph[i].reserve(obs.offsets[i + 1] - obs.offsets[i]);
      for (uint64_t k = obs.offsets[i]; k < obs.offsets[i + 1]; ++k)
        ba.vis_graph[i].push_back({(size_t)obs.point_idx[k], {obs.uv[2 * k], obs.uv[2 * k + 1]}});
    }
    return ba;
  }
  // impl Display, src/baproblem.rs:788-801
  std::string to_string() const {
    std::ostringstream s;
    s << "Bundle Adjustment Problem with " << num_cameras() << " cameras, " << num_points() << " points, "
      << "and " << num_observations() << " observations";
    return s.str();
  }
};

namespace synthetic {
// src/synthetic.rs:163-300.  Occlusion by the analytic 2-D wall test of the reference (src/synthetic.rs:52-124),
// or — mesh_occlusion, the north star's configuration, not in the reference — by rays against one box of
// height building_height per city block (c2b_city_mesh).
inline BAProblem synthetic_grid(const Context &ctx, size_t num_cameras_per_block, size_t num_points_per_block,
                                size_t num_blocks, double block_length, double block_inset, double camera_height,
                                double point_height, double max_dist, bool /*verbose*/, bool mesh_occlusion = false,
                                double building_height = 10.0) {
  detail::require(block_inset * 2.0 < block_length,
                  "Block inset must be less than half the block length, to not violate physical constraints.");
  std::vector<SnavelyCamera> cams(c2b_grid_num_cameras(num_cameras_per_block, num_blocks));
  std::vector<Point3> pts(c2b_grid_num_points(num_points_per_block, num_blocks));
  static_assert(sizeof(SnavelyCamera) == sizeof(double) * C2B_CAM_STRIDE, "camera records must be contiguous");
  detail::check(c2b_grid_cameras(num_cameras_per_block, num_blocks, block_length, camera_height,
                                 cams.empty() ? nullptr : cams[0].rec));
  detail::check(c2b_grid_points(num_points_per_block, num_blocks, block_length, block_inset, point_height,
                                pts.empty() ? nullptr : pts[0].data()));
  VisGraph g;
  if (mesh_occlusion) {
    std::vector<float> xyz(3 * 8 * num_blocks * num_blocks);
    std::vector<uint32_t> tri(3 * 12 * num_blocks * num_blocks);
    detail::check(c2b_city_mesh(num_blocks, block_length, block_inset, building_height, xyz.data(), tri.data()));
    const Scene scene(ctx, xyz, tri);
    g = detail::run_visibility(ctx, &scene, cams, pts, max_dist, C2B_OCC_MESH, block_length, block_inset);
  } else {
    g = detail::run_visibility(ctx, nullptr, cams, pts, max_dist, C2B_OCC_ANALYTIC, block_length, block_inset);
  }
  return BAProblem::from_visibility(std::move(cams), std::move(pts), std::move(g)).cull();
}

// src/synthetic.rs:313-381 (no occlusion test)
inline BAProblem synthetic_line(const Context &ctx, size_t num_cameras, size_t num_points, double length,
                                double point_offset, double camera_height, double point_height, double max_dist,
                                bool /*verbose*/) {
  std::vector<SnavelyCamera> cams(num_cameras);
  std::vector<Point3> pts(num_points);
  detail::check(c2b_line_cameras(num_cameras, length, camera_height, cams.empty() ? nullptr : cams[0].rec));
  detail::check(c2b_line_points(num_points, length, point_offset, point_height, pts.empty() ? nullptr : pts[0].data()));
  VisGraph g = detail::run_visibility(ctx, nullptr, cams, pts, max_dist, C2B_OCC_NONE, 20.0, 1.0);
  return BAProblem::from_visibility(std::move(cams), std::move(pts), std::move(g)).cull();
}
}  // namespace synthetic

namespace noise {
namespace detail_n {
struct Flat {
  std::vector<double> cams, pts, uv;
  explicit Flat(const BAProblem &ba) : cams(detail::flatten(ba.cameras)) {
    pts.reserve(ba.points.size() * 3);
    for (const auto &p : ba.points) pts.insert(pts.end(), p.begin(), p.end());
    for (const auto &o : ba.vis_graph)
      for (const auto &e : o) {
        uv.push_back(e.second.first);
        uv.push_back(e.second.second);
      }
  }
  BAProblem rebuild(const BAProblem &ba) const {
    BAProblem out = ba;
    for (size_t i = 0; i < out.cameras.size(); ++i) std::memcpy(out.cameras[i].rec, &cams[i * C2B_CAM_STRIDE], sizeof out.cameras[i].rec);
    for (size_t i = 0; i < out.points.size(); ++i) out.points[i] = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    size_t k = 0;
    for (auto &o : out.vis_graph)
      for (auto &e : o) {
        e.second = {uv[2 * k], uv[2 * k + 1]};
        ++k;
      }
    return out;
  }
};
}  // namespace detail_n

// src/noise.rs:68-116
inline BAProblem add_drift(const Context &ctx, const BAProblem &ba, double strength, double angle_strength, double std_,
                           const Vector3 &dir, uint64_t seed) {
  // the reference's nearest-to-origin fold1(..).unwrap() (src/noise.rs:75-87) panics on an empty problem
  detail::require(ba.num_cameras() + ba.num_points() > 0, "called `Option::unwrap()` on a `None` value");
  detail_n::Flat f(ba);
  detail::check(c2b_add_drift(ctx.handle(), f.cams.data(), ba.num_cameras(), f.pts.data(), ba.num_points(), strength,
                              angle_strength, std_, dir.data(), seed));
  return f.rebuild(ba);
}
// src/noise.rs:47-56
inline BAProblem add_drift_normalized(const Context &ctx, const BAProblem &ba, double strength, double angle_strength,
                                      double std_, uint64_t seed) {
  detail::require(ba.num_cameras() + ba.num_points() > 0, "called `Option::unwrap()` on a `None` value");
  detail_n::Flat f(ba);
  detail::check(c2b_add_drift_normalized(ctx.handle(), f.cams.data(), ba.num_cameras(), f.pts.data(), ba.num_points(),
                                         strength, angle_strength, std_, seed));
  return f.rebuild(ba);
}
// src/noise.rs:119-177
inline BAProblem add_noise(const Context &ctx, const BAProblem &ba, double translation_std, double rotation_std,
                           double point_std, double observations_std, uint64_t seed) {
  detail_n::Flat f(ba);
  detail::check(c2b_add_noise(ctx.handle(), f.cams.data(), ba.num_cameras(), f.pts.data(), ba.num_points(), f.uv.data(),
                              f.uv.size() / 2, translation_std, rotation_std, point_std, observations_std, seed));
  return f.rebuild(ba);
}
// src/noise.rs:388-416
inline BAProblem add_sin_noise(const Context &ctx, const BAProblem &ba, const Vector3 &dir, const Vector3 &noise_dir,
                               double strength, double frequency) {
  detail_n::Flat f(ba);
  detail::check(c2b_add_sin_noise(ctx.handle(), f.cams.data(), ba.num_cameras(), f.pts.data(), ba.num_points(),
                                  dir.data(), noise_dir.data(), strength, frequency));
  return f.rebuild(ba);
}

// ---- graph-editing noise (src/noise.rs:180-378): sequential, data-dependent edits of the observation
// graph, host side like the reference's (they are O(observations) and not on the data-parallel path).
// Seeded; parity with the reference's thread_rng() draws is distributional.

// src/noise.rs:180-226: with probability mismatch_chance an observation trades its point index with
// another observation of the same camera, chosen with weight (largest image distance) - (its image
// distance) — as written there, which also gives the observation itself the largest weight.
inline BAProblem add_incorrect_correspondences(const BAProblem &bal, double mismatch_chance, uint64_t seed) {
  BAProblem out = bal;
  detail::Rng rng(seed);
  for (auto &obs : out.vis_graph) {
    if (obs.size() <= 1) continue;
    for (size_t i = 0; i < obs.size(); ++i) {
      if (!(rng.uniform() <= mismatch_chance)) continue;
      std::vector<double> weights(obs.size());
      for (size_t j = 0; j < obs.size(); ++j) {
        const double dx = obs[i].second.first - obs[j].second.first, dy = obs[i].second.second - obs[j].second.second;
        weights[j] = -std::sqrt(dx * dx + dy * dy);
      }
      weights[i] = 0.0;
      double m = INFINITY;
      for (double w : weights) m = std::fmin(m, w);
      for (double &w : weights) w -= m;
      const size_t j = rng.weighted(weights);
      std::swap(obs[i].first, obs[j].first);
    }
  }
  return out;
}
// the same on the GPU (c2b_add_incorrect_correspondences), with the library's deterministic draws: a pure function
// of seed, not the draws of the host form above.  Throws std::logic_error with the host form's text when a selected
// observation's weights are invalid.  stats (optional) receives the call's counts and device times.
inline BAProblem add_incorrect_correspondences(const Context &ctx, const BAProblem &bal, double mismatch_chance,
                                               uint64_t seed, c2b_mismatch_stats *stats = nullptr) {
  const size_t nc = bal.num_cameras();
  std::vector<uint64_t> offsets(nc + 1, 0);
  for (size_t i = 0; i < nc; ++i) offsets[i + 1] = offsets[i] + bal.vis_graph[i].size();
  std::vector<uint32_t> idx(offsets[nc]);
  std::vector<double> uv(2 * offsets[nc]);
  for (size_t i = 0, k = 0; i < nc; ++i)
    for (const auto &e : bal.vis_graph[i]) {
      detail::require(e.first <= 0xffffffffull, "point index does not fit 32 bits");
      idx[k] = (uint32_t)e.first;
      uv[2 * k] = e.second.first;
      uv[2 * k + 1] = e.second.second;
      ++k;
    }
  c2b_mismatch_stats st;
  const int rc = c2b_add_incorrect_correspondences(ctx.handle(), offsets.data(), nc, idx.data(), uv.data(),
                                                   mismatch_chance, seed, &st);
  if (rc == C2B_ERR_INVALID) {
    const std::string m = c2b_last_error();
    for (const char *kind : {"AllWeightsZero", "NegativeWeight"})
      if (m.size() >= std::strlen(kind) && m.compare(m.size() - std::strlen(kind), std::string::npos, kind) == 0)
        throw std::logic_error(std::string("called `Result::unwrap()` on an `Err` value: ") + kind);
  }
  detail::check(rc);
  if (stats) *stats = st;
  BAProblem out = bal;
  size_t k = 0;
  for (auto &o : out.vis_graph)
    for (auto &e : o) e.first = idx[k++];
  return out;
}

// src/noise.rs:229-250: every camera keeps floor(len * drop_percent) of its observations, chosen by a shuffle
inline BAProblem drop_features(const BAProblem &bal, double drop_percent, uint64_t seed) {
  BAProblem out = bal;
  detail::Rng rng(seed);
  for (auto &o : out.vis_graph) {
    const size_t l = (size_t)((double)o.size() * drop_percent);
    rng.shuffle(o);
    if (l < o.size()) o.resize(l);
  }
  return out;
}

// src/noise.rs:254-288: floor(split_percent * points) landmarks get a copy at the same location; each of
// their observations moves to the copy with probability 1/2
inline BAProblem split_landmarks(const BAProblem &bal, double split_percent, uint64_t seed) {
  BAProblem out = bal;
  detail::Rng rng(seed);
  const size_t l = bal.points.size();
  const size_t n = (size_t)(split_percent * (double)l);
  const std::vector<size_t> inds = rng.choose_multiple(l, n);
  std::unordered_map<size_t, size_t> split_inds;
  for (size_t k = 0; k < inds.size(); ++k) {
    out.points.push_back(bal.points[inds[k]]);
    split_inds[inds[k]] = l + k;
  }
  for (auto &obs : out.vis_graph)
    for (auto &e : obs) {
      const auto it = split_inds.find(e.first);
      if (it != split_inds.end() && rng.coin()) e.first = it->second;
    }
  return out;
}

namespace detail_n {
// k nearest neighbours over the points (the reference's rstar R-tree, nearest_neighbor_iter): a k-d tree
struct KdTree {
  const std::vector<Point3> &pts;
  std::vector<uint32_t> order;
  explicit KdTree(const std::vector<Point3> &p) : pts(p), order(p.size()) {
    std::iota(order.begin(), order.end(), 0u);
    build(0, order.size(), 0);
  }
  void build(size_t lo, size_t hi, int axis) {
    if (hi - lo <= 1) return;
    const size_t mid = (lo + hi) / 2;
    std::nth_element(order.begin() + lo, order.begin() + mid, order.begin() + hi,
                     [&](uint32_t a, uint32_t b) { return pts[a][axis] < pts[b][axis]; });
    build(lo, mid, (axis + 1) % 3);
    build(mid + 1, hi, (axis + 1) % 3);
  }
  // (squared distance, index) of the k nearest points to q, ascending (ties by index)
  std::vector<std::pair<double, uint32_t>> nearest(const Point3 &q, size_t k) const {
    std::vector<std::pair<double, uint32_t>> heap;  // max-heap on (distance, index)
    search(0, order.size(), 0, q, k, heap);
    std::sort_heap(heap.begin(), heap.end());
    return heap;
  }
  void search(size_t lo, size_t hi, int axis, const Point3 &q, size_t k,
              std::vector<std::pair<double, uint32_t>> &heap) const {
    if (lo >= hi) return;
    const size_t mid = (lo + hi) / 2;
    const uint32_t id = order[mid];
    const Vector3 d = detail::sub(pts[id], q);
    const std::pair<double, uint32_t> cand{detail::dot(d, d), id};
    if (heap.size() < k) {
      heap.push_back(cand);
      std::push_heap(heap.begin(), heap.end());
    } else if (cand < heap.front()) {
      std::pop_heap(heap.begin(), heap.end());
      heap.back() = cand;
      std::push_heap(heap.begin(), heap.end());
    }
    const double delta = q[axis] - pts[id][axis];
    const int next = (axis + 1) % 3;
    if (delta < 0.0) {
      search(lo, mid, next, q, k, heap);
      if (heap.size() < k || delta * delta <= heap.front().first) search(mid + 1, hi, next, q, k, heap);
    } else {
      search(mid + 1, hi, next, q, k, heap);
      if (heap.size() < k || delta * delta <= heap.front().first) search(lo, mid, next, q, k, heap);
    }
  }
};
}  // namespace detail_n

// src/noise.rs:323-378: floor(join_percent * points) observations (drawn over ALL observations) are
// re-pointed at one of the 10 nearest other landmarks of the landmark they see
inline BAProblem join_landmarks(const BAProblem &bal, double join_percent, uint64_t seed) {
  BAProblem out = bal;
  detail::Rng rng(seed);
  const detail_n::KdTree tree(bal.points);
  const size_t n = (size_t)(join_percent * (double)bal.points.size());
  const std::vector<size_t> inds = rng.choose_multiple(bal.num_observations(), n);
  std::vector<size_t> starts(bal.vis_graph.size() + 1, 0);  // linear observation index -> (camera, slot)
  for (size_t c = 0; c < bal.vis_graph.size(); ++c) starts[c + 1] = starts[c] + bal.vis_graph[c].size();
  for (size_t i : inds) {
    const size_t c = (size_t)(std::upper_bound(starts.begin(), starts.end(), i) - starts.begin()) - 1;
    auto &e = out.vis_graph[c][i - starts[c]];
    const auto near = tree.nearest(bal.points[e.first], 11);  // .skip(1).take(10)
    detail::require(near.size() > 1, "No neighbors?!");
    e.first = near[1 + rng.below(near.size() - 1)].second;
  }
  return out;
}
// the same on the GPU (c2b_join_landmarks), with the library's deterministic draws: a pure function of seed, not the
// draws of the host form above; the neighbours are exact, ties by index.  Throws the host form's std::logic_error
// ("No neighbors?!") when observations are selected among fewer than two points.  stats (optional) receives the
// call's counts and device times.
inline BAProblem join_landmarks(const Context &ctx, const BAProblem &bal, double join_percent, uint64_t seed,
                                c2b_join_stats *stats = nullptr) {
  const size_t nc = bal.num_cameras(), np = bal.num_points();
  std::vector<uint64_t> offsets(nc + 1, 0);
  for (size_t i = 0; i < nc; ++i) offsets[i + 1] = offsets[i] + bal.vis_graph[i].size();
  std::vector<uint32_t> idx(offsets[nc]);
  for (size_t i = 0, k = 0; i < nc; ++i)
    for (const auto &e : bal.vis_graph[i]) {
      detail::require(e.first <= 0xffffffffull, "point index does not fit 32 bits");
      idx[k++] = (uint32_t)e.first;
    }
  std::vector<double> pts(3 * np);
  for (size_t i = 0; i < np; ++i)
    for (int k = 0; k < 3; ++k) pts[3 * i + k] = bal.points[i][k];
  c2b_join_stats st;
  const int rc = c2b_join_landmarks(ctx.handle(), pts.data(), np, offsets.data(), nc, idx.data(), join_percent, seed,
                                    &st);
  if (rc == C2B_ERR_INVALID) {
    const std::string m = c2b_last_error(), tail = "No neighbors?!";
    if (m.size() >= tail.size() && m.compare(m.size() - tail.size(), std::string::npos, tail) == 0)
      throw std::logic_error(tail);
  }
  detail::check(rc);
  if (stats) *stats = st;
  BAProblem out = bal;
  size_t k = 0;
  for (auto &o : out.vis_graph)
    for (auto &e : o) e.first = idx[k++];
  return out;
}
}  // namespace noise

}  // namespace city2ba
