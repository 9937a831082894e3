// tests/cpp/test_cull.cpp — BAProblem::cull(ctx) (c2b_cull_problem on the GPU) against the host BAProblem::cull()
// of include/city2ba.hpp: identical cameras, points and observations, bit for bit, on seeded random graphs and on
// the un-culled graph of synthetic_grid(10, 20, 3, 5, 1, 1, 1, 10) (analytic occlusion, as test_host.cpp uses it).
#include <cstdio>
#include <cstring>
#include <random>

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

static bool same_bits(const void *a, const void *b, size_t n) { return std::memcmp(a, b, n) == 0; }

static bool same_problem(const BAProblem &a, const BAProblem &b) {
  if (a.num_cameras() != b.num_cameras() || a.num_points() != b.num_points()) return false;
  for (size_t i = 0; i < a.num_cameras(); ++i)
    if (!same_bits(a.cameras[i].rec, b.cameras[i].rec, sizeof a.cameras[i].rec)) return false;
  for (size_t i = 0; i < a.num_points(); ++i)
    if (!same_bits(a.points[i].data(), b.points[i].data(), 3 * sizeof(double))) return false;
  for (size_t c = 0; c < a.num_cameras(); ++c) {
    if (a.vis_graph[c].size() != b.vis_graph[c].size()) return false;
    for (size_t k = 0; k < a.vis_graph[c].size(); ++k) {
      const auto &x = a.vis_graph[c][k], &y = b.vis_graph[c][k];
      if (x.first != y.first || !same_bits(&x.second.first, &y.second.first, 8) ||
          !same_bits(&x.second.second, &y.second.second, 8))
        return false;
    }
  }
  return true;
}

// several components over disjoint point groups, duplicates, unsorted lists, 0..8 observations per camera
static BAProblem random_problem(std::mt19937_64 &rng) {
  std::uniform_real_distribution<double> u(-1.0, 1.0);
  const size_t C = rng() % 40, P = rng() % 60, groups = 1 + rng() % 4;
  BAProblem ba;
  ba.cameras.resize(C);
  for (auto &c : ba.cameras)
    for (double &v : c.rec) v = u(rng);
  ba.points.resize(P);
  for (auto &p : ba.points)
    for (double &v : p) v = u(rng);
  ba.vis_graph.resize(C);
  for (size_t c = 0; c < C && P; ++c) {
    const size_t g = rng() % groups, k = rng() % 9;
    for (size_t j = 0; j < k; ++j) {
      size_t p = rng() % P;
      p -= p % groups;  // group g owns the points congruent to g
      p += g;
      if (p >= P) continue;
      ba.vis_graph[c].push_back({p, {u(rng), u(rng)}});
    }
  }
  return ba;
}

int main() {
  const Context ctx(0);
  std::mt19937_64 rng(99);
  for (int t = 0; t < 200; ++t) {
    const BAProblem ba = random_problem(rng);
    c2b_cull_stats st;
    const BAProblem gpu = ba.cull(ctx, &st);
    const BAProblem host = ba.cull();
    CHECK(same_problem(gpu, host));
    CHECK(st.n_cameras == host.num_cameras() && st.n_points == host.num_points() &&
          st.n_obs == host.num_observations());
  }
  {  // the graph synthetic::synthetic_grid builds before its .cull()
    const size_t cpb = 10, ppb = 20, n = 3;
    const double L = 5.0, inset = 1.0;
    std::vector<SnavelyCamera> cams(c2b_grid_num_cameras(cpb, n));
    std::vector<Point3> pts(c2b_grid_num_points(ppb, n));
    detail::check(c2b_grid_cameras(cpb, n, L, 1.0, cams[0].rec));
    detail::check(c2b_grid_points(ppb, n, L, inset, 1.0, pts[0].data()));
    VisGraph g = detail::run_visibility(ctx, nullptr, cams, pts, 10.0, C2B_OCC_ANALYTIC, L, inset);
    const BAProblem ba = BAProblem::from_visibility(std::move(cams), std::move(pts), std::move(g));
    const BAProblem host = ba.cull();
    CHECK(host.num_observations() > 0);
    CHECK(same_problem(ba.cull(ctx), host));
    CHECK(same_problem(synthetic::synthetic_grid(ctx, 10, 20, 3, 5., 1., 1., 1., 10., false), host));
  }
  if (failures) return 1;
  std::printf("test_cull ok\n");
  return 0;
}
