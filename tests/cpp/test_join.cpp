// tests/cpp/test_join.cpp — noise::join_landmarks(ctx, ...) (c2b_join_landmarks on the GPU): the reference's library
// property (tests/main.rs:155-190) on synthetic_grid(10, 20, 3, 5, 1, 1, 1, 10), the host form's error, and the point
// indices before and after the call written to argv[1] (u32, native order) so that the Python test can compare them
// with noise.join_landmarks_gpu on the same seed.
#include <cstdio>
#include <stdexcept>
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

int main(int argc, char **argv) {
  if (argc != 2) return 2;
  const Context ctx(0);
  const BAProblem ba = synthetic::synthetic_grid(ctx, 10, 20, 3, 5., 1., 1., 1., 10., false);
  CHECK(ba.num_observations() > 0);
  c2b_join_stats st;
  const BAProblem out = noise::join_landmarks(ctx, ba, 0.01, 7, &st);
  CHECK(out.total_reprojection_error(2.0) > ba.total_reprojection_error(2.0));
  CHECK(st.n_selected == (uint64_t)(0.01 * (double)ba.num_points()) && st.n_changed > 0 &&
        st.n_changed <= st.n_selected);
  FILE *f = std::fopen(argv[1], "wb");
  CHECK(f != nullptr);
  if (!f) return 1;
  for (const BAProblem *p : {&ba, &out})
    for (const auto &o : p->vis_graph)
      for (const auto &e : o) {
        const uint32_t v = (uint32_t)e.first;
        std::fwrite(&v, 4, 1, f);
      }
  std::fclose(f);
  // the host form's error, with its text: observations selected among fewer than two points
  BAProblem one = ba;
  one.points.resize(1);
  for (auto &o : one.vis_graph)
    for (auto &e : o) e.first = 0;
  std::string what;
  try {
    noise::join_landmarks(ctx, one, 1.0, 3);
  } catch (const std::logic_error &e) {
    what = e.what();
  }
  CHECK(what == "No neighbors?!");
  // the ctx stays usable and the result is a function of the seed
  CHECK(noise::join_landmarks(ctx, ba, 0.01, 7).vis_graph == out.vis_graph);
  if (failures) return 1;
  std::printf("test_join ok\n");
  return 0;
}
