// sample_shim.cpp -- the sampling side of the host planner (ractip_b200/csrc/plan.cpp) on a CPU, for
// tests/test_sampling.py: rp::check_samples and what rp::plan_batch derives from the sampling options (each problem's
// flags and kernel, the constraint keys the emulator binds) on the device facts of a B200, next to the plan of the same
// pairs without samples.
#include <cstring>
#include <string>

#include "plan.h"

namespace {
rp::DeviceFacts b200() {
  rp::DeviceFacts dev;
  dev.sm_count = 148;
  dev.smem_optin = 232448;
  dev.ctas_per_sm = 2;
  dev.ctas_per_sm1 = 1;
  dev.up_ctas_per_sm = 1;
  dev.band_occupancy = [](int threads, size_t) { return threads == rp::BAND_THREADS[0] ? 1 : 2; };
  dev.memory = []() { return (size_t)170 << 30; };
  return dev;
}
}  // namespace

// rc of check_samples (its message to msg), else of plan_batch(cons, se, so).  key: the plan's constraint keys
// (key_len entries, at most cap copied).  probs: per problem (seq_off, n, constrained, on the general kernel).
// same_as_soft: whether the plan equals that of the same pairs without samples (buffers, problems, queue, launch shapes).
extern "C" int sample_shim(const rp_pair* pairs, const rp_constraint* cons, const rp_stack_energy* se, int n_pairs,
                           const rp_opts* opts, const rp_sample_opts* so, char* msg, int msg_cap, uint16_t* key,
                           long long* key_len, int cap, long long* probs, int* same_as_soft) {
  std::string m;
  int rc = rp::check_samples(pairs, n_pairs, opts, so, &m);
  std::snprintf(msg, (size_t)msg_cap, "%s", m.c_str());
  if (rc) return rc;
  const rp::DeviceFacts dev = b200();
  rp::BatchPlan p, q;
  rc = rp::plan_batch(pairs, n_pairs, opts, dev, rp::RouteSettings{}, &p, cons, se, so);
  if (rc) return rc;
  rc = rp::plan_batch(pairs, n_pairs, opts, dev, rp::RouteSettings{}, &q, cons, se);
  *key_len = (long long)p.key.size();
  std::memcpy(key, p.key.data(), sizeof(uint16_t) * std::min<size_t>(p.key.size(), (size_t)cap));
  const size_t g0 = (size_t)p.n_band[0] + p.n_band[1];
  for (size_t k = 0; k < p.probs.size(); k++) {
    bool general = false;
    for (size_t x = g0; x < g0 + (size_t)p.n_general; x++) general |= p.order[x] == (int)k;
    probs[4 * k] = p.probs[k].seq_off;
    probs[4 * k + 1] = p.probs[k].n;
    probs[4 * k + 2] = p.probs[k].constrained;
    probs[4 * k + 3] = general;
  }
  bool same = p.seq == q.seq && p.key == q.key && p.stack == q.stack && p.probs.size() == q.probs.size() &&
              p.order == q.order && p.n_band[0] == q.n_band[0] && p.n_band[1] == q.n_band[1] &&
              p.n_general == q.n_general && p.up_mode == q.up_mode && p.mcc_minb == q.mcc_minb && p.grid == q.grid &&
              p.cluster == q.cluster && p.band_grid[0] == q.band_grid[0] && p.band_grid[1] == q.band_grid[1] &&
              p.ws_doubles == q.ws_doubles && p.split_fetch == q.split_fetch && p.sample_total == q.sample_total;
  for (size_t k = 0; same && k < p.probs.size(); k++) same = std::memcmp(&p.probs[k], &q.probs[k], sizeof(rp::Problem)) == 0;
  *same_as_soft = same;
  return rc;
}
