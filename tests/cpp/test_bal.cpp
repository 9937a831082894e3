// tests/cpp/test_bal.cpp — the BAL writer against the C++ mirror of include/city2ba.hpp.
//   host part (always):    c2b_camera_to_vec equals SnavelyCamera::to_vec bit for bit on random rotations that
//                          cover the four branches of quat_from_mat, the identity, half turns and d < eps
//   GPU part (no --host-only): BAProblem::write(ctx, path) equals write_text / write_binary byte for byte, on seeded
//                          random problems whose values are all below 2^53 in magnitude (where std::to_chars(fixed)
//                          prints the shortest digits too) and on the culled synthetic_grid(10, 20, 3, 5, 1, 1, 1, 10)
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>
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

static std::string slurp(const std::string &path) {
  std::ifstream f(path, std::ios::binary);
  return std::string(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
}

// which quat_from_mat branch a rotation takes (0: trace >= 0, 1-3: the largest diagonal entry)
static int branch(const Basis3 &m) {
  auto M = [&](int c, int r) { return m[c * 3 + r]; };
  if ((M(0, 0) + M(1, 1)) + M(2, 2) >= 0.0) return 0;
  if (M(0, 0) > M(1, 1) && M(0, 0) > M(2, 2)) return 1;
  return M(1, 1) > M(2, 2) ? 2 : 3;
}

static void host_part() {
  std::mt19937_64 rng(7);
  std::normal_distribution<double> nd;
  std::uniform_real_distribution<double> ud(-1.0, 1.0);
  int hits[4] = {0, 0, 0, 0}, zero_branch = 0;
  auto one = [&](const Basis3 &R) {
    SnavelyCamera c;
    std::copy(R.begin(), R.end(), c.rec);
    for (int k = 9; k < 15; ++k) c.rec[k] = ud(rng) * 100.0;
    const auto ref = c.to_vec();
    double got[9];
    c2b_camera_to_vec(c.rec, got);
    CHECK(std::memcmp(ref.data(), got, sizeof got) == 0);
    ++hits[branch(R)];
    if (ref[0] == 0.0 && ref[1] == 0.0 && ref[2] == 0.0) ++zero_branch;
  };
  for (int i = 0; i < 100000; ++i) {
    Vector3 a{nd(rng), nd(rng), nd(rng)};
    a = detail::normalize(a);
    const int kind = i % 4;
    const double angle = kind == 0 ? ud(rng) * 3.141592653589793          // anywhere
                         : kind == 1 ? 3.141592653589793 - 1e-3 * std::fabs(ud(rng))  // near a half turn
                         : kind == 2 ? 1e-9 * ud(rng)                      // d < eps
                                     : 2.0 + std::fabs(ud(rng));           // trace < 0
    one(from_axis_angle(a, angle));
  }
  one(basis_one());
  for (int k = 0; k < 3; ++k) {  // exact half turns about the axes and a diagonal
    Vector3 a{0, 0, 0};
    a[(size_t)k] = 1.0;
    one(from_axis_angle(a, 3.141592653589793));
  }
  one(from_axis_angle(detail::normalize({1, 1, 1}), 3.141592653589793));
  one(from_angle_y(3.141592653589793));
  for (int b = 0; b < 4; ++b) CHECK(hits[b] > 1000);
  CHECK(zero_branch > 1000);
  std::printf("to_vec: branches %d %d %d %d, d < eps %d\n", hits[0], hits[1], hits[2], hits[3], zero_branch);
}

static BAProblem random_problem(std::mt19937_64 &rng, size_t C, size_t P, size_t max_obs) {
  std::uniform_real_distribution<double> u(-1.0, 1.0);
  std::uniform_int_distribution<int> ex(-30, 40);
  auto val = [&]() {
    const double x = u(rng) * std::ldexp(1.0, ex(rng));  // |x| < 2^40
    return (rng() % 16 == 0) ? std::round(x) : x;         // integers now and then, signed zeros among them
  };
  BAProblem ba;
  for (size_t c = 0; c < C; ++c) {
    Vector3 a{u(rng), u(rng), u(rng) + 2.0};
    SnavelyCamera cam;
    const Basis3 R = from_axis_angle(detail::normalize(a), u(rng) * 3.0);
    std::copy(R.begin(), R.end(), cam.rec);
    for (int k = 9; k < 15; ++k) cam.rec[k] = val();
    ba.cameras.push_back(cam);
  }
  for (size_t p = 0; p < P; ++p) ba.points.push_back({val(), val(), val()});
  ba.vis_graph.resize(C);
  for (size_t c = 0; c < C && P; ++c) {
    const size_t k = rng() % (max_obs + 1);
    for (size_t j = 0; j < k; ++j) ba.vis_graph[c].push_back({(size_t)(rng() % P), {val(), val()}});
  }
  return ba;
}

static void same_files(const Context &ctx, const BAProblem &ba, const std::string &dir, const char *what) {
  for (const char *ext : {".bal", ".bbal"}) {
    const std::string host = dir + "/host" + ext, gpu = dir + "/gpu" + ext;
    ba.write(host);
    c2b_bal_stats st;
    ba.write(ctx, gpu, &st);
    const std::string a = slurp(host), b = slurp(gpu);
    if (a != b) std::printf("%s%s: %zu host bytes, %zu GPU bytes\n", what, ext, a.size(), b.size());
    CHECK(a == b);
    CHECK(st.bytes == b.size());
  }
}

int main(int argc, char **argv) {
  host_part();
  if (argc > 1 && !std::strcmp(argv[1], "--host-only")) {
    if (failures) return 1;
    std::printf("test_bal (host) ok\n");
    return 0;
  }
  const std::string dir = argc > 1 ? argv[1] : ".";
  const Context ctx(0);
  std::mt19937_64 rng(11);
  same_files(ctx, random_problem(rng, 0, 0, 0), dir, "empty");
  same_files(ctx, random_problem(rng, 5, 0, 0), dir, "no points");
  for (int t = 0; t < 20; ++t) same_files(ctx, random_problem(rng, 1 + rng() % 50, 1 + rng() % 500, 40), dir, "random");
  same_files(ctx, random_problem(rng, 300, 20000, 400), dir, "larger");
  {
    const BAProblem ba = synthetic::synthetic_grid(ctx, 10, 20, 3, 5., 1., 1., 1., 10., false);
    CHECK(ba.num_observations() > 0);
    same_files(ctx, ba, dir, "synthetic_grid");
  }
  {  // an unwritable path is Error::IOError
    bool io = false;
    try {
      random_problem(rng, 2, 3, 2).write(ctx, dir + "/no/such/dir/x.bal");
    } catch (const Error &e) {
      io = e.kind == Error::IOError;
    }
    CHECK(io);
  }
  if (failures) return 1;
  std::printf("test_bal ok\n");
  return 0;
}
