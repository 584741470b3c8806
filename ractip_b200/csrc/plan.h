// plan.h -- how a batch runs: every host-side routing decision of rp_batch_create / rp_batch_run, as one pure
// function of the pairs, the device's facts and the route settings.  Plain C++ (no CUDA headers): api.cu executes
// the plan, tests/test_plan.py checks it on a CPU.
#ifndef RP_PLAN_H
#define RP_PLAN_H

#include <stddef.h>
#include <stdint.h>

#include <functional>
#include <string>
#include <utility>
#include <vector>

#include "mcc_core.h"
#include "ractip_prob.h"

namespace rp {

// problems at least this long run the 128-register build of the general kernel (RouteSettings::mcc_long_n)
constexpr int MCC_LONG_N = 700;
// CTA widths of the band kernel's two launch shapes: class L (one CTA per SM), class S (two CTAs per SM)
constexpr int BAND_THREADS[2] = {512, 256};

// Read from the environment once per context (rp_create); they exist for tests and A/B comparisons.
struct RouteSettings {
  bool band = true;              // RP_BAND=0: every problem goes to the general kernel
  int mcc_long_n = MCC_LONG_N;   // RP_MCC_LONG_N
  int cluster = -1;              // RP_CLUSTER: -1 chosen by batch size, 0 one CTA per problem, 8 / 16 forced
  bool split_fetch = true;       // RP_NO_SPLIT_FETCH: fetch the dense outputs in one copy
};

struct DeviceFacts {
  int sm_count = 0;
  size_t smem_optin = 0;   // max dynamic shared memory per CTA
  int ctas_per_sm = 0;     // occupancy of the general kernel, 64-register build
  int ctas_per_sm1 = 0;    // ... 128-register build
  int up_ctas_per_sm = 0;  // ... of unstru_kernel
  size_t ws_bytes = 0;     // workspace the context already holds
  // CTAs per SM of the band kernel with `threads` threads and `smem` bytes of dynamic shared memory
  std::function<int(int threads, size_t smem)> band_occupancy;
  // free device memory + ws_bytes + cached pool buffers.  Slow (cudaMemGetInfo): asked at most once per plan, and
  // only when a workspace the plan wants exceeds ws_bytes.
  std::function<size_t()> memory;
};

struct BatchPlan {
  std::vector<uint8_t> seq;              // encoded sequences, per pair  0 s1 0 s2 0 s1s2 0
  // structure-constraint keys of the constrained problems, laid out like seq (pair (i,j) of a problem is allowed iff
  // its two bases carry the same key); empty when no problem of the batch is constrained
  std::vector<uint16_t> key;
  std::vector<Problem> probs;            // three per pair: s1, s2, s1&s2
  std::vector<rp_dense_layout> layout;
  size_t total_floats = 0;
  bool has_single = false;               // some pair has n2 == 0: its unused output sections are zero-filled once
  double alg_flops = 0;
  // Work queue: [class L | class S | general | unstru_kernel (mode 1)].  Entries are problem indices, + RP_JOB_UNPAIRED
  // for an unpaired-window job (mode 2).
  std::vector<int> order;
  int n_band[2] = {0, 0};
  int n_general = 0;                     // general-kernel + duplex entries
  int n_mcc = 0, n_duplex = 0;
  // Unpaired-window passes of the band classes: 0 fused with the wavefronts, 1 unstru_kernel after them, 2 jobs of
  // their own inside the band kernel.  Modes 1 and 2 keep each deferred problem's tables in a private workspace.
  int up_mode = 0;
  int n_defer = 0;
  size_t defer_slot = 0;                 // doubles per private workspace
  // launch shapes
  int mcc_minb = 2;                      // register budget of the general kernel (kernels.h)
  int grid = 0;                          // general kernel (and duplex kernel): CTAs = workspace slots
  int cluster = 0;                       // CTAs per problem of the multi-CTA wavefront (0: one CTA per problem)
  int band_grid[2] = {0, 0};
  size_t band_smem[2] = {0, 0};
  int up_grid = 0;
  // workspace, in doubles: [general slots | class L slots | class S slots | private workspaces]
  size_t slot_doubles = 0;               // general kernel
  size_t band_slot[2] = {0, 0};
  size_t ws_band[2] = {0, 0};            // offsets of the band classes' slots
  size_t ws_up = 0;                      // offset of the private workspaces
  size_t ws_doubles = 0;
  // launch timed by itself for the roofline: the one with most of the algorithmic flops (0 / 1 band class,
  // 2 general), -1 when nothing carries any
  int dom_kind = -1;
  double dom_flops = 0;
  // Split fetch (uniform batches whose problems fall into both band classes, nothing else launched): sections of a
  // pair's dense block written by the long class / by the short class, as (offset, length) in floats within pair 0's
  // block; every pair has the same block layout, `pair_stride` floats apart.
  bool split_fetch = false;
  size_t pair_stride = 0;
  std::vector<std::pair<size_t, size_t>> sect_long, sect_short;
};

size_t bp_len(int L);
int check_pairs(const rp_pair* pairs, int n_pairs, const rp_opts* opts);
// The structure constraints of pairs that pass check_pairs (cons may be null: none).  RP_OK, or RP_ERR_ARG with a
// message in *msg that names the pair, the string and the (1-based) position.
int check_constraints(const rp_pair* pairs, const rp_constraint* cons, int n_pairs, std::string* msg);

// The pairs must pass check_pairs and the constraints check_constraints (cons == null: none).  A problem that a
// constraint restricts runs on the general kernel.  Returns RP_OK, or RP_ERR_CUDA when a band launch shape fits no SM.
int plan_batch(const rp_pair* pairs, int n_pairs, const rp_opts* opts, const DeviceFacts& dev, const RouteSettings& rs,
               BatchPlan* plan, const rp_constraint* cons = nullptr);

}  // namespace rp
#endif
