// tests/cpp/test_mismatch.cpp — noise::add_incorrect_correspondences(ctx, ...) (c2b_add_incorrect_correspondences on
// the GPU): the reference's library property (tests/main.rs:155-190) on synthetic_grid(10, 20, 3, 5, 1, 1, 1, 10),
// the host form's error text, and the point indices before and after the call written to argv[1] (u32, native
// order) so that the Python test can compare them with noise.add_incorrect_correspondences_gpu on the same seed.
#include <cmath>
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

static std::string error_of(const Context &ctx, const BAProblem &ba) {
  try {
    noise::add_incorrect_correspondences(ctx, ba, 1.0, 3);
  } catch (const std::logic_error &e) {
    return e.what();
  }
  return "";
}

int main(int argc, char **argv) {
  if (argc != 2) return 2;
  const Context ctx(0);
  const BAProblem ba = synthetic::synthetic_grid(ctx, 10, 20, 3, 5., 1., 1., 1., 10., false);
  CHECK(ba.num_observations() > 0);
  c2b_mismatch_stats st;
  const BAProblem out = noise::add_incorrect_correspondences(ctx, ba, 0.01, 4, &st);
  CHECK(out.total_reprojection_error(2.0) > ba.total_reprojection_error(2.0));
  CHECK(st.n_selected > 0 && st.n_swapped > 0 && st.n_swapped <= st.n_selected);
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
  // the host form's errors, with its text
  BAProblem same = ba;
  for (auto &e : same.vis_graph[0]) e.second = same.vis_graph[0][0].second;
  CHECK(error_of(ctx, same) == "called `Result::unwrap()` on an `Err` value: AllWeightsZero");
  BAProblem nan = ba;
  nan.vis_graph[1][2].second.first = std::nan("");
  CHECK(error_of(ctx, nan) == "called `Result::unwrap()` on an `Err` value: NegativeWeight");
  // the ctx stays usable and the result is a function of the seed
  CHECK(noise::add_incorrect_correspondences(ctx, ba, 0.01, 4).vis_graph == out.vis_graph);
  if (failures) return 1;
  std::printf("test_mismatch ok\n");
  return 0;
}
