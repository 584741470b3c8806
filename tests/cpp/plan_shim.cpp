// plan_shim.cpp -- rp::plan_batch (ractip_b200/csrc/plan.cpp) on stubbed device facts, its decisions as one flat
// array for tests/test_plan.py.
#include "plan.h"

namespace {
enum {
  S_N_PROBS, S_N_ORDER, S_N_BAND0, S_N_BAND1, S_N_GENERAL, S_N_MCC, S_N_DUPLEX, S_UP_MODE, S_N_DEFER, S_MCC_MINB,
  S_GRID, S_CLUSTER, S_BAND_GRID0, S_BAND_GRID1, S_UP_GRID, S_DOM_KIND, S_SPLIT_FETCH, S_N_SECT_LONG, S_N_SECT_SHORT,
  S_MEMORY_CALLS, S_TOTAL_FLOATS, S_WS_DOUBLES, S_DEFER_SLOT, S_SLOT_DOUBLES, S_COUNT = 32
};
}

// facts: sm_count, smem_optin, ctas_per_sm, ctas_per_sm1, up_ctas_per_sm, ws_bytes, band occupancy of class L and S,
//        memory (what DeviceFacts::memory returns)
// settings: band, mcc_long_n, cluster, split_fetch
// out: S_COUNT scalars, then the queue, then per problem (kind, n, defer_up, ws_off), then the long and the short
//      sections as (offset, length).  Returns the plan's code, or -1 when `cap` entries do not hold it.
extern "C" int plan_shim(const rp_pair* pairs, int n_pairs, const rp_opts* opts, const long long* facts,
                         const int* settings, long long* out, int cap) {
  rp::DeviceFacts dev;
  dev.sm_count = (int)facts[0];
  dev.smem_optin = (size_t)facts[1];
  dev.ctas_per_sm = (int)facts[2];
  dev.ctas_per_sm1 = (int)facts[3];
  dev.up_ctas_per_sm = (int)facts[4];
  dev.ws_bytes = (size_t)facts[5];
  dev.band_occupancy = [&](int threads, size_t) { return (int)(threads == rp::BAND_THREADS[0] ? facts[6] : facts[7]); };
  long long memory_calls = 0;
  dev.memory = [&]() { memory_calls++; return (size_t)facts[8]; };
  rp::RouteSettings rs;
  rs.band = settings[0] != 0;
  rs.mcc_long_n = settings[1];
  rs.cluster = settings[2];
  rs.split_fetch = settings[3] != 0;
  rp::BatchPlan p;
  const int rc = rp::plan_batch(pairs, n_pairs, opts, dev, rs, &p);
  const size_t need = S_COUNT + p.order.size() + 4 * p.probs.size() + 2 * (p.sect_long.size() + p.sect_short.size());
  if (need > (size_t)cap) return -1;
  long long* s = out;
  s[S_N_PROBS] = (long long)p.probs.size();
  s[S_N_ORDER] = (long long)p.order.size();
  s[S_N_BAND0] = p.n_band[0];
  s[S_N_BAND1] = p.n_band[1];
  s[S_N_GENERAL] = p.n_general;
  s[S_N_MCC] = p.n_mcc;
  s[S_N_DUPLEX] = p.n_duplex;
  s[S_UP_MODE] = p.up_mode;
  s[S_N_DEFER] = p.n_defer;
  s[S_MCC_MINB] = p.mcc_minb;
  s[S_GRID] = p.grid;
  s[S_CLUSTER] = p.cluster;
  s[S_BAND_GRID0] = p.band_grid[0];
  s[S_BAND_GRID1] = p.band_grid[1];
  s[S_UP_GRID] = p.up_grid;
  s[S_DOM_KIND] = p.dom_kind;
  s[S_SPLIT_FETCH] = p.split_fetch;
  s[S_N_SECT_LONG] = (long long)p.sect_long.size();
  s[S_N_SECT_SHORT] = (long long)p.sect_short.size();
  s[S_MEMORY_CALLS] = memory_calls;
  s[S_TOTAL_FLOATS] = (long long)p.total_floats;
  s[S_WS_DOUBLES] = (long long)p.ws_doubles;
  s[S_DEFER_SLOT] = (long long)p.defer_slot;
  s[S_SLOT_DOUBLES] = (long long)p.slot_doubles;
  long long* o = out + S_COUNT;
  for (int x : p.order) *o++ = x;
  for (const rp::Problem& q : p.probs) {
    *o++ = q.kind; *o++ = q.n; *o++ = q.defer_up; *o++ = q.ws_off;
  }
  for (const auto* v : {&p.sect_long, &p.sect_short})
    for (const auto& sc : *v) { *o++ = (long long)sc.first; *o++ = (long long)sc.second; }
  return rc;
}
