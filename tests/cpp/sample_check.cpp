// sample_check.cpp -- the C++ shim's sampling overload (include/ractip_prob.hpp), for tests/test_sampling.py:
//   sample_check gpu S1 S2 PROBLEM NUM SEED   one pair's samples of one problem (RP_SAMPLE_* bit), one table per line
#include <cstdio>
#include <cstdlib>
#include <exception>
#include <string>
#include <vector>

#include "ractip_prob.hpp"

int main(int argc, char** argv) {
  if (argc != 7) {
    std::printf("usage: sample_check gpu S1 S2 PROBLEM NUM SEED\n");
    return 2;
  }
  try {
    rp::ProbabilityStage stage;
    rp::PairProbabilities pp;
    std::vector<std::vector<int16_t> > samples;
    stage.solve_probabilities(argv[2], argv[3], "", "", {}, {}, std::atoi(argv[4]), std::atoi(argv[5]),
                              std::strtoull(argv[6], nullptr, 10), pp, samples);
    std::printf("samples %zu sum_hp_rows %zu\n", samples.size(), pp.hp.size());
    for (const auto& t : samples) {
      for (size_t k = 0; k < t.size(); k++) std::printf(k ? " %d" : "%d", t[k]);
      std::printf("\n");
    }
  } catch (const std::exception& e) {
    std::printf("error: %s\n", e.what());
    return 1;
  }
  return 0;
}
