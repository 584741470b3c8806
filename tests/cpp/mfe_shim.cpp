// mfe_shim.cpp -- TEST INFRASTRUCTURE.  The host side of rp_run_mfe (check_mfe, plan_mfe) on a CPU, for tests/test_mfe.py:
// device facts as arguments, the plan's layout, jobs and per-base arrays out.
#include <cstring>

#include "plan.h"

// facts: sm_count, mfe_ctas_per_sm, ws_bytes, memory.  out_layout: 6 per pair (s1, s2, co, len_s1, len_s2, len_co);
// out_jobs: 8 per job (seq_off, n, cp, flags, out, energy_at, eu_const, 0) up to cap_jobs; scal: total, jobs, grid,
// slot_ints; es / eu / key: the per-base arrays (length in scal[4]; empty ones left alone), up to cap_seq.
extern "C" int mfe_shim(const rp_pair* pairs, const rp_constraint* cons, const rp_stack_energy* se,
                        const rp_unpaired_energy* ue, int n_pairs, int problems, const long long* facts, char* msg,
                        int msg_cap, long long* out_layout, long long* out_jobs, int cap_jobs, long long* scal,
                        int* es, int* eu, unsigned short* key, int cap_seq) {
  std::string m;
  int rc = rp::check_mfe(pairs, n_pairs, cons, se, ue, problems, &m);
  rp::MfePlan plan;
  if (rc == RP_OK) {
    rp::DeviceFacts dev;
    dev.sm_count = (int)facts[0];
    dev.mfe_ctas_per_sm = (int)facts[1];
    dev.ws_bytes = (size_t)facts[2];
    dev.memory = [&]() { return (size_t)facts[3]; };
    rc = rp::plan_mfe(pairs, n_pairs, cons, se, ue, problems, dev, &plan, &m);
  }
  std::snprintf(msg, msg_cap, "%s", m.c_str());
  if (rc != RP_OK) return rc;
  for (int p = 0; p < n_pairs; p++) {
    const rp_sample_layout& L = plan.layout[p];
    const long long v[6] = {(long long)L.s1, (long long)L.s2, (long long)L.co, (long long)L.len_s1, (long long)L.len_s2, (long long)L.len_co};
    std::memcpy(out_layout + 6 * p, v, sizeof v);
  }
  for (size_t k = 0; k < plan.jobs.size() && (int)k < cap_jobs; k++) {
    const rp::MfeJob& j = plan.jobs[k];
    const long long v[8] = {j.seq_off, j.n, j.cp, j.flags, j.out, j.energy_at, j.eu_const, 0};
    std::memcpy(out_jobs + 8 * k, v, sizeof v);
  }
  scal[0] = (long long)plan.total;
  scal[1] = (long long)plan.jobs.size();
  scal[2] = plan.grid;
  scal[3] = (long long)plan.slot_ints;
  scal[4] = (long long)plan.seq.size();
  for (size_t x = 0; x < plan.seq.size() && (int)x < cap_seq; x++) {
    if (!plan.es.empty()) es[x] = plan.es[x];
    if (!plan.eu.empty()) eu[x] = plan.eu[x];
    if (!plan.key.empty()) key[x] = plan.key[x];
  }
  return RP_OK;
}
