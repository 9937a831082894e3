// tests/cpp/test_bal_read.cpp — the BAL reader against the C++ mirror of include/city2ba.hpp.
//   host part (always):    c2b_camera_from_vec equals SnavelyCamera::from_vec bit for bit on random 9-vectors that
//                          cover both branches of from_rodrigues, with theta2 at and around 2.220446049250313e-16
//   GPU part (no --host-only): BAProblem::from_file(ctx, path) equals BAProblem::from_file(path) bit for bit on
//                          files the mirror's write_text / write_binary wrote, and maps errors as from_file does
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <random>
#include <string>

#include "city2ba.hpp"

using namespace city2ba;

static int failures = 0;
#define CHECK(cond)                                                        \
  do {                                                                     \
    if (!(cond)) {                                                         \
      std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond);        \
      std::fflush(stdout);                                                 \
      ++failures;                                                          \
    }                                                                      \
  } while (0)

static bool same_bits(const double *a, const double *b, size_t n) { return std::memcmp(a, b, n * sizeof(double)) == 0; }

static void host_part() {
  std::mt19937_64 rng(11);
  std::normal_distribution<double> N(0.0, 1.0);
  std::uniform_real_distribution<double> U(-1.0, 1.0);
  const double eps = 2.220446049250313e-16;
  int small = 0, large = 0;
  for (int i = 0; i < 100000; ++i) {
    std::array<double, 9> v;
    for (auto &t : v) t = N(rng) * std::pow(10.0, (double)(int)(rng() % 7) - 3.0);
    const int kind = i % 4;
    double d[3] = {N(rng), N(rng), N(rng)};
    const double n = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    double scale;
    if (kind == 0) scale = U(rng) * 3.2;                                       // ordinary rotations
    else if (kind == 1) scale = std::sqrt(eps) * (1.0 + U(rng) * 1e-6);       // theta2 around the threshold
    else if (kind == 2) scale = std::sqrt(eps) * std::nextafter(1.0, (double)(rng() % 2) * 2.0);  // within an ulp
    else scale = std::sqrt(eps) * U(rng) * 1e-3;                              // far below it
    for (int k = 0; k < 3; ++k) v[k] = d[k] / n * scale;
    if (i == 1) v[0] = std::sqrt(eps), v[1] = v[2] = 0.0;
    if (i == 2) v[0] = v[1] = v[2] = 0.0;
    const double theta2 = (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2];
    (theta2 > eps ? large : small)++;
    const SnavelyCamera ref = SnavelyCamera::from_vec(v);
    double got[C2B_CAM_STRIDE];
    c2b_camera_from_vec(v.data(), got);
    if (!same_bits(ref.rec, got, C2B_CAM_STRIDE)) {
      CHECK(same_bits(ref.rec, got, C2B_CAM_STRIDE));
      if (failures > 5) return;
    }
  }
  CHECK(small > 20000 && large > 20000);
}

static BAProblem random_problem(std::mt19937_64 &rng, size_t C, size_t P, size_t max_obs) {
  std::normal_distribution<double> N(0.0, 1.0);
  BAProblem ba;
  for (size_t c = 0; c < C; ++c) {
    std::array<double, 9> v;
    for (auto &t : v) t = N(rng);
    ba.cameras.push_back(SnavelyCamera::from_vec(v));
  }
  for (size_t p = 0; p < P; ++p) ba.points.push_back({N(rng) * 100.0, N(rng), N(rng) * 1e-3});
  ba.vis_graph.assign(C, {});
  for (size_t c = 0; c < C; ++c) {
    const size_t n = P ? rng() % (max_obs + 1) : 0;
    for (size_t k = 0; k < n; ++k) ba.vis_graph[c].push_back({(size_t)(rng() % P), {N(rng), N(rng)}});
  }
  return ba;
}

static void same_problem(const BAProblem &a, const BAProblem &b, const char *what) {
  bool ok = a.cameras.size() == b.cameras.size() && a.points.size() == b.points.size() &&
            a.vis_graph.size() == b.vis_graph.size();
  for (size_t i = 0; ok && i < a.cameras.size(); ++i) ok = same_bits(a.cameras[i].rec, b.cameras[i].rec, C2B_CAM_STRIDE);
  for (size_t i = 0; ok && i < a.points.size(); ++i) ok = same_bits(a.points[i].data(), b.points[i].data(), 3);
  for (size_t c = 0; ok && c < a.vis_graph.size(); ++c) {
    ok = a.vis_graph[c].size() == b.vis_graph[c].size();
    for (size_t k = 0; ok && k < a.vis_graph[c].size(); ++k) {
      const auto &x = a.vis_graph[c][k], &y = b.vis_graph[c][k];
      ok = x.first == y.first && same_bits(&x.second.first, &y.second.first, 1) &&
           same_bits(&x.second.second, &y.second.second, 1);
    }
  }
  if (!ok) std::printf("problem differs: %s\n", what);
  CHECK(ok);
}

static void gpu_part(const std::string &dir) {
  const Context ctx(0);
  std::mt19937_64 rng(12);
  const size_t sizes[][3] = {{1, 1, 3}, {9, 40, 12}, {70, 900, 60}, {0, 5, 0}, {4, 0, 0}};
  for (const auto &s : sizes) {
    const BAProblem ba = random_problem(rng, s[0], s[1], s[2]);
    for (const char *ext : {".bal", ".bbal"}) {
      const std::string path = dir + "/cpp_read" + ext;
      ba.write(path);
      c2b_bal_read_stats st;
      const BAProblem gpu = BAProblem::from_file(ctx, path, &st);
      same_problem(BAProblem::from_file(path), gpu, ext);
      CHECK(st.n_cameras == s[0] && st.n_points == s[1] && st.regrouped == 0);
    }
  }
  // errors: the kinds from_file throws
  {
    std::ofstream(dir + "/bad.bal") << "2 1 1\n0 0 1.0 x\n";
    bool parse = false;
    try {
      BAProblem::from_file(ctx, dir + "/bad.bal");
    } catch (const Error &e) {
      parse = e.kind == Error::ParseError;
    }
    CHECK(parse);
    std::ofstream(dir + "/range.bal") << "1 1 1\n0 3 1 2\n" << std::string(9, '1') << " 0 0 0 0 0 0 0 0\n1 2 3\n";
    bool logic = false;
    try {
      BAProblem::from_file(ctx, dir + "/range.bal");
    } catch (const std::logic_error &) {
      logic = true;
    }
    CHECK(logic);
    bool io = false;
    try {
      BAProblem::from_file(ctx, dir + "/missing.bal");
    } catch (const Error &e) {
      io = e.kind == Error::IOError;
    }
    CHECK(io);
  }
}

int main(int argc, char **argv) {
  host_part();
  if (!(argc > 1 && !std::strcmp(argv[1], "--host-only"))) gpu_part(argc > 1 ? argv[1] : ".");
  std::printf("%s\n", failures ? "FAILURES" : "OK");
  return failures ? 1 : 0;
}
