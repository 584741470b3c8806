// emul_constrained.cpp -- TEST INFRASTRUCTURE.  The routes of the general kernel (solve_mcc, solve_mcc_wide, the
// cluster schedule) on the host, as emul.cpp runs them, for a problem with a structure constraint: its keys are bound
// to Ctx::key as mcc_persistent / mcc_cluster_kernel bind them.  Built by tests/test_constraints.py.
#include "emul.cpp"

namespace {
template <class Exec>
int keyed_run(Exec&& ex, int W, bool wide, bool lockstep, const uint16_t* key, const rp_model* m, const char* seq,
              int n, int cp, int kind, int max_w, int n1, int n2, float th_hy, int T, float* bp, float* up, float* hp,
              double* logz) {
  int rc = rp::build_dev_model(*m, &g_model);
  if (rc) return rc;
  std::vector<uint8_t> S(n + 16, 0);
  for (int i = 1; i <= n; i++) S[i] = rp::encode_base(seq[i - 1]);
  rp::Problem p;
  std::memset(&p, 0, sizeof p);
  p.n = n; p.cp = cp; p.kind = kind; p.max_w = max_w; p.n1 = n1; p.n2 = n2; p.th_hy = th_hy; p.constrained = key != nullptr;
  size_t nbp, nup, nhp;
  layout(n, max_w, n1, n2, nbp, nup, nhp);
  std::vector<float> dense(nbp + nup + nhp + 8, 0.f);
  p.out_bp = (kind == rp::KIND_LINEAR && bp) ? 0 : -1;
  p.out_up = (kind == rp::KIND_LINEAR && up && max_w > 0) ? (long long)nbp : -1;
  p.out_hp = (kind == rp::KIND_COFOLD && hp) ? (long long)(nbp + nup) : -1;
  std::vector<double> ws(rp::slot_doubles(n), 1e300);
  std::vector<double> smem(rp::shared_bytes(T, W) / sizeof(double) + 2, lockstep ? 1e300 : 0.0);
  rp::Shared sh;
  rp::carve_shared(sh, smem.data(), T, W);
  double lz[3] = {0, 0, 0};
  rp::Ctx c;
  rp::bind_ctx(c, &g_model, S.data(), p, ws.data());
  c.key = key;
  if (!wide) rp::solve_mcc(ex, c, p, dense.data(), lz, sh);
  else rp::solve_mcc_wide(ex, c, p, dense.data(), lz, sh);
  if (int err = ex.error()) return err;
  if (p.out_bp >= 0) std::memcpy(bp, dense.data(), nbp * sizeof(float));
  if (p.out_up >= 0) std::memcpy(up, dense.data() + nbp, nup * sizeof(float));
  if (p.out_hp >= 0) std::memcpy(hp, dense.data() + nbp + nup, nhp * sizeof(float));
  if (logz) *logz = lz[0];
  return 0;
}
}  // namespace

// One problem of the general kernel with constraint keys key[1..n] (pair (i,j) allowed iff key[i] == key[j]; null: no
// constraint).  route 0: solve_mcc; 5, 10, 15: solve_mcc_wide with split-sum bands of that width; G = 8, 16 (route 10
// only): the cluster schedule.  lockstep: the warp-lockstep executor (the device's shuffle forms, kBatch 2 for
// solve_mcc, 4 otherwise), else the serial one.  Returns -1 for a route it does not run.
extern "C" int emul_constrained_problem(int route, int G, int lockstep, const uint16_t* key, const rp_model* m,
                                        const char* seq, int n, int cp, int kind, int max_w, int n1, int n2, float th_hy,
                                        int T, float* bp, float* up, float* hp, double* logz) {
  auto run = [&](auto&& ex, int W, bool wide) {
    return keyed_run(ex, W, wide, lockstep != 0, key, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
  };
  if (G == 8 || G == 16) {
    if (route != 10) return -1;
    if (lockstep) return G == 8 ? run(wemu::WarpExecT<8, 4, 10>(T), 10, true) : run(wemu::WarpExecT<16, 4, 10>(T), 10, true);
    return G == 8 ? run(SerialExecT<10, 8>{T}, 10, true) : run(SerialExecT<10, 16>{T}, 10, true);
  }
  if (G != 1) return -1;
  switch (route) {
    case 0: return lockstep ? run(wemu::WarpExecT<1, 2, rp::BAND>(T), rp::BAND, false) : run(SerialExec{T}, rp::BAND, false);
    case 5: return lockstep ? run(wemu::WarpExecT<1, 4, 5>(T), 5, true) : run(SerialExecT<5>{T}, 5, true);
    case 10: return lockstep ? run(wemu::WarpExecT<1, 4, 10>(T), 10, true) : run(SerialExecT<10>{T}, 10, true);
    case 15: return lockstep ? run(wemu::WarpExecT<1, 4, 15>(T), 15, true) : run(SerialExecT<15>{T}, 15, true);
    default: return -1;
  }
}
