// constraint_shim.cpp -- the structure-constraint side of the host planner (ractip_b200/csrc/plan.cpp) on a CPU, for
// tests/test_constraints.py: rp::check_constraints and what rp::plan_batch derives from the constraints (the key
// buffer, each problem's flag and kernel) on the device facts of a B200.
#include <cstring>
#include <string>

#include "plan.h"

// rc of check_constraints (its message to msg), else of plan_batch.  key: the plan's key buffer (key_len entries,
// 0 when the plan has none; at most cap copied).  probs: per problem (seq_off, n, constrained, on the general kernel).
extern "C" int constraint_shim(const rp_pair* pairs, const rp_constraint* cons, int n_pairs, const rp_opts* opts,
                               char* msg, int msg_cap, unsigned short* key, long long* key_len, int cap, long long* probs) {
  std::string m;
  int rc = rp::check_constraints(pairs, cons, n_pairs, &m);
  std::snprintf(msg, (size_t)msg_cap, "%s", m.c_str());
  if (rc) return rc;
  rp::DeviceFacts dev;
  dev.sm_count = 148;
  dev.smem_optin = 232448;
  dev.ctas_per_sm = 2;
  dev.ctas_per_sm1 = 1;
  dev.up_ctas_per_sm = 1;
  dev.band_occupancy = [](int threads, size_t) { return threads == rp::BAND_THREADS[0] ? 1 : 2; };
  dev.memory = []() { return (size_t)170 << 30; };
  rp::BatchPlan p;
  rc = rp::plan_batch(pairs, n_pairs, opts, dev, rp::RouteSettings{}, &p, cons);
  *key_len = (long long)p.key.size();
  std::memcpy(key, p.key.data(), sizeof(unsigned short) * std::min<size_t>(p.key.size(), (size_t)cap));
  const size_t g0 = (size_t)p.n_band[0] + p.n_band[1];
  for (size_t k = 0; k < p.probs.size(); k++) {
    bool general = false;
    for (size_t x = g0; x < g0 + (size_t)p.n_general; x++) general |= p.order[x] == (int)k;
    probs[4 * k] = p.probs[k].seq_off;
    probs[4 * k + 1] = p.probs[k].n;
    probs[4 * k + 2] = p.probs[k].constrained;
    probs[4 * k + 3] = general;
  }
  return rc;
}
