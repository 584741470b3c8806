// emul_sampled.cpp -- TEST INFRASTRUCTURE.  The sampling phase of the general kernel (mcc_sample.h) on the host, on each
// of its routes (solve_mcc, solve_mcc_wide, the cluster schedule), serial or warp-lockstep as emul.cpp runs them.  The
// sample buffer, seed and count are bound to Ctx::smp* as bind_per_base (kernels.cu) binds them, and so are the
// stacking factors and constraint keys.  Built by tests/test_sampling.py.
#include "emul.cpp"

namespace {
template <class Exec>
int sampled_run(Exec&& ex, int W, bool wide, bool lockstep, const double* stk, const uint16_t* key, const rp_model* m,
                const char* seq, int n, int cp, int kind, int pair, int which, unsigned long long seed, int num, int T,
                int16_t* out, double* logz) {
  int rc = rp::build_dev_model(*m, &g_model);
  if (rc) return rc;
  std::vector<uint8_t> S(n + 16, 0);
  for (int i = 1; i <= n; i++) S[i] = rp::encode_base(seq[i - 1]);
  rp::Problem p;
  std::memset(&p, 0, sizeof p);
  p.n = n; p.cp = cp; p.kind = kind; p.pair = pair; p.which = which;
  p.out_bp = p.out_up = p.out_hp = -1;   // samples only
  p.constrained = (key ? rp::CON_KEYS : 0) | (stk ? rp::CON_STACK : 0) | rp::CON_SAMPLE;
  std::vector<double> ws(rp::slot_doubles(n), 1e300);
  std::vector<double> smem(rp::shared_bytes(T, W) / sizeof(double) + 2, lockstep ? 1e300 : 0.0);
  std::vector<int16_t> buf((size_t)num * n + 1, -1);   // the phase clears it
  rp::Shared sh;
  rp::carve_shared(sh, smem.data(), T, W);
  std::vector<double> lz(3 * (size_t)pair + 3, 0.);   // emit_logz writes lz[3 pair + which]
  rp::Ctx c;
  rp::bind_ctx(c, &g_model, S.data(), p, ws.data());
  c.key = key;
  c.stk = stk;
  c.smp = buf.data();
  c.smp_seed = seed;
  c.smp_num = num;
  if (!wide) rp::solve_mcc(ex, c, p, nullptr, lz.data(), sh);
  else rp::solve_mcc_wide(ex, c, p, nullptr, lz.data(), sh);
  if (int err = ex.error()) return err;
  std::memcpy(out, buf.data(), (size_t)num * n * sizeof(int16_t));
  if (logz) *logz = lz[3 * (size_t)pair + which];
  return 0;
}
}  // namespace

// `num` samples of one problem (pair `pair`, problem `which` for the random numbers) into out[num][n], with stacking
// factors stk[1..n] and constraint keys key[1..n] (null: none).  route and G as emul_shaped_problem; lockstep: the
// warp-lockstep executor (the shuffle form of the decisions), else the serial one (the direct form).  Returns -1 for a
// route it does not run.
extern "C" int emul_sampled_problem(int route, int G, int lockstep, const double* stk, const uint16_t* key,
                                    const rp_model* m, const char* seq, int n, int cp, int kind, int pair, int which,
                                    unsigned long long seed, int num, int T, int16_t* out, double* logz) {
  auto run = [&](auto&& ex, int W, bool wide) {
    return sampled_run(ex, W, wide, lockstep != 0, stk, key, m, seq, n, cp, kind, pair, which, seed, num, T, out, logz);
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
