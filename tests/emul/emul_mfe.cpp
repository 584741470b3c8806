// emul_mfe.cpp -- TEST INFRASTRUCTURE.  The MFE kernel's phase functions (ractip_b200/csrc/mfe_core.h) on the host:
// thread after thread with lane 0 of each warp walking the candidates alone (the reference form), or warp by warp in
// lockstep with the device's shuffle reductions (warp_emul.h).  Per-base data are bound as mfe_kernel binds them.
// Built by tests/test_mfe.py.
#include <cstring>
#include <vector>

#include "warp_emul.h"   // first: the host stand-ins for the CUDA intrinsics

#include "dev_model.h"
#include "mfe_core.h"
#include "seq_encode.h"

namespace {
struct SerialMfeExec {
  static constexpr bool kShfl = false;
  int T;
  int nthreads() const { return T; }
  template <class F>
  void phase(int, F f) {
    for (int t = 0; t < T; t++) f(t);
  }
  int error() const { return 0; }
};

rp::DevModel g_model;   // large

template <class Exec>
int mfe_run(Exec&& ex, const char* seq, int n, int cp, const uint16_t* key, const int* es, const int* eu, int16_t* pt,
            int* energy) {
  std::vector<uint8_t> S(n + 16, 0);
  for (int i = 1; i <= n; i++) S[i] = rp::encode_base(seq[i - 1]);
  std::vector<int> ws(rp::mfe_slot_ints(n), 0x5a5a5a5a);   // poison: stale data must never be read
  std::vector<int> red(ex.nthreads(), 0x5a5a5a5a);
  rp::MfeCtx c;
  rp::bind_mfe(c, &g_model, S.data(), n, cp, ws.data());
  c.key = key;
  c.es = es;
  c.eu = eu;
  int e = rp::MFE_INF;
  rp::solve_mfe(ex, c, red.data(), pt, &e);
  if (int err = ex.error()) return err;
  int eu_const = 0;
  for (int i = 1; eu && i <= n; i++) eu_const += eu[i];
  *energy = e >= rp::MFE_BIG ? RP_INF : e + eu_const;
  return 0;
}
}  // namespace

// One problem of length n (cp > 0: the co-fold with strand 2 from cp) with keys, stacking and unpaired pseudo-energies
// at [1..n] (null: none) on T threads.  pt: n int16; energy: 0.01 kcal/mol, the unpaired constant included.
extern "C" int emul_mfe_problem(int lockstep, int T, const rp_model* m, const char* seq, int n, int cp,
                                const uint16_t* key, const int* es, const int* eu, int16_t* pt, int* energy) {
  int rc = rp::build_dev_model(*m, &g_model);
  if (rc) return rc;
  if (lockstep) return mfe_run(wemu::WarpExecT<1, 4, 10>(T), seq, n, cp, key, es, eu, pt, energy);
  return mfe_run(SerialMfeExec{T}, seq, n, cp, key, es, eu, pt, energy);
}
