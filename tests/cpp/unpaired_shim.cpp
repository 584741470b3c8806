// unpaired_shim.cpp -- the unpaired-pseudo-energy side of the host planner (ractip_b200/csrc/plan.cpp) on a CPU, for
// tests/test_unpaired.py: rp::check_unpaired_energies and what rp::plan_batch derives from the energies (the pair
// factors, the log-Z terms, each problem's flags and kernel) on the device facts of a B200, next to the plan of the same
// pairs without them.
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

// rc of check_unpaired_energies (its message to msg), else of plan_batch(cons, se, so = none, ue).  unp: the plan's
// pair factors (unp_len entries, 0 when the plan has none; at most cap copied); lz: its log-Z terms (3 per pair, or
// none).  probs: per problem (seq_off, n, constrained, on the general kernel).  same_as_plain: whether the whole plan
// without the unpaired data (buffers, problems, queue, launch shapes) equals the plan of the same pairs, constraints
// and stacking energies without unpaired energies.
extern "C" int unpaired_shim(const rp_pair* pairs, const rp_constraint* cons, const rp_stack_energy* se,
                             const rp_unpaired_energy* ue, int n_pairs, const rp_opts* opts, char* msg, int msg_cap,
                             double* unp, long long* unp_len, double* lz, int cap, long long* probs, int* same_as_plain) {
  std::string m;
  int rc = rp::check_unpaired_energies(pairs, ue, n_pairs, opts, &m);
  std::snprintf(msg, (size_t)msg_cap, "%s", m.c_str());
  if (rc) return rc;
  const rp::DeviceFacts dev = b200();
  rp::BatchPlan p, q;
  rc = rp::plan_batch(pairs, n_pairs, opts, dev, rp::RouteSettings{}, &p, cons, se, nullptr, ue);
  if (rc) return rc;
  rc = rp::plan_batch(pairs, n_pairs, opts, dev, rp::RouteSettings{}, &q, cons, se, nullptr);
  *unp_len = (long long)p.unpaired.size();
  std::memcpy(unp, p.unpaired.data(), sizeof(double) * std::min<size_t>(p.unpaired.size(), (size_t)cap));
  std::memcpy(lz, p.unpaired_lz.data(), sizeof(double) * std::min<size_t>(p.unpaired_lz.size(), (size_t)cap));
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
              p.n_general == q.n_general && p.n_mcc == q.n_mcc && p.up_mode == q.up_mode && p.mcc_minb == q.mcc_minb &&
              p.grid == q.grid && p.cluster == q.cluster && p.band_grid[0] == q.band_grid[0] &&
              p.band_grid[1] == q.band_grid[1] && p.band_smem[0] == q.band_smem[0] && p.band_smem[1] == q.band_smem[1] &&
              p.ws_doubles == q.ws_doubles && p.slot_doubles == q.slot_doubles && p.split_fetch == q.split_fetch &&
              p.alg_flops == q.alg_flops && p.total_floats == q.total_floats;
  for (size_t k = 0; same && k < p.probs.size(); k++) same = std::memcmp(&p.probs[k], &q.probs[k], sizeof(rp::Problem)) == 0;
  *same_as_plain = same;
  return rc;
}
