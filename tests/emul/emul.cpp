// emul.cpp -- TEST INFRASTRUCTURE.  Runs the kernels' per-thread phase
// functions (ractip_b200/csrc/mcc_core.h, mcc_driver.h) on the host, one
// emulated thread after another, so that the CUDA kernels' logic can be checked
// against the oracle on a CPU-only box.  Never loaded by the product.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "dev_model.h"
#include "mcc_driver.h"
#include "seq_encode.h"

namespace {
// The executor (contract at the top of mcc_driver.h) of G CTAs that share one problem, run as one serial flow with one
// copy of shared memory: it runs the work of every rank, rank after rank, as the device deals it out.
template <int W, int G = 1>
struct SerialExecT {
  static constexpr int kCtas = G;
  static constexpr int kWide = W;   // width of the wide split-sum bands (solve_mcc_wide)
  int T;
  int nthreads() const { return T; }
  template <class F>
  void phase(int, F f) {
    for (int t = 0; t < T; t++) f(t);
  }
  int rank_begin() const { return 0; }
  int rank_end() const { return G; }
  void sync() {}
};
using SerialExec = SerialExecT<rp::BAND>;

rp::DevModel g_model;  // large

void layout(int n, int max_w, int n1, int n2, size_t& nbp, size_t& nup, size_t& nhp) {
  nbp = (size_t)(n + 1) * (n + 2) / 2;
  nup = (size_t)n * (max_w > 0 ? max_w : 0);
  nhp = (size_t)(n1 + 1) * (n2 + 1);
}
}  // namespace

// one problem; band = 0: general kernel (solve_mcc), band = 1: shared-memory band kernel (solve_band),
// band = 5, 8, 10, 15: general kernel with wide split-sum bands of that width (solve_mcc_wide);
// G = 8, 16 (band = 10 only): solve_mcc_wide on a cluster of G CTAs
static int run_problem(int band, int G, const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1, int n2,
                       float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  int rc = rp::build_dev_model(*m, &g_model);
  if (rc) return rc;
  std::vector<uint8_t> S(n + 16, 0);
  for (int i = 1; i <= n; i++) S[i] = rp::encode_base(seq[i - 1]);
  rp::Problem p;
  std::memset(&p, 0, sizeof p);
  p.seq_off = 0; p.n = n; p.cp = cp; p.kind = kind; p.pair = 0; p.which = 0; p.max_w = max_w;
  p.n1 = n1; p.n2 = n2; p.th_hy = th_hy;
  size_t nbp, nup, nhp;
  layout(n, max_w, n1, n2, nbp, nup, nhp);
  std::vector<float> dense(nbp + nup + nhp + 8, 0.f);
  p.out_bp = (kind == rp::KIND_LINEAR && bp) ? 0 : -1;
  p.out_up = (kind == rp::KIND_LINEAR && up && max_w > 0) ? (long long)nbp : -1;
  p.out_hp = (kind == rp::KIND_COFOLD && hp) ? (long long)(nbp + nup) : -1;
  std::vector<double> ws(rp::slot_doubles(n), 1e300);  // poison: stale data must never be read
  const int W = band >= rp::BAND ? band : rp::BAND;
  std::vector<double> smem(rp::shared_bytes(T, W) / sizeof(double) + 2, 0.0);
  rp::Shared sh;
  rp::carve_shared(sh, smem.data(), T, W);
  double lz[3] = {0, 0, 0};
  rp::Ctx c;
  rp::bind_ctx(c, &g_model, S.data(), p, ws.data());
  SerialExec ex{T};
  if (G == 8) {
    SerialExecT<10, 8> wx{T};
    rp::solve_mcc_wide(wx, c, p, dense.data(), lz, sh);
  } else if (G == 16) {
    SerialExecT<10, 16> wx{T};
    rp::solve_mcc_wide(wx, c, p, dense.data(), lz, sh);
  } else if (band == 5) {
    SerialExecT<5> wx{T};
    rp::solve_mcc_wide(wx, c, p, dense.data(), lz, sh);
  } else if (band == 8) {
    SerialExecT<8> wx{T};
    rp::solve_mcc_wide(wx, c, p, dense.data(), lz, sh);
  } else if (band == 10) {
    SerialExecT<10> wx{T};
    rp::solve_mcc_wide(wx, c, p, dense.data(), lz, sh);
  } else if (band == 15) {
    SerialExecT<15> wx{T};
    rp::solve_mcc_wide(wx, c, p, dense.data(), lz, sh);
  } else if (band) {
    std::vector<double> bsm(rp::band_shared_doubles(n, T) + 2, 1e300);  // poison
    rp::solve_band(ex, c, p, dense.data(), lz, bsm.data());
  } else {
    rp::solve_mcc(ex, c, p, dense.data(), lz, sh);
  }
  if (p.out_bp >= 0) std::memcpy(bp, dense.data(), nbp * sizeof(float));
  if (p.out_up >= 0) std::memcpy(up, dense.data() + nbp, nup * sizeof(float));
  if (p.out_hp >= 0) std::memcpy(hp, dense.data() + nbp + nup, nhp * sizeof(float));
  if (logz) *logz = lz[0];
  return 0;
}

extern "C" int emul_problem(const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1, int n2,
                            float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  return run_problem(0, 1, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
extern "C" int emul_wide_problem(int W, const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1,
                                 int n2, float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  if (W != 5 && W != 8 && W != 10 && W != 15) return -1;
  return run_problem(W, 1, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
extern "C" int emul_band_problem(const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1, int n2,
                                 float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  return run_problem(1, 1, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
extern "C" int emul_cluster_problem(int G, const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1,
                                    int n2, float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  if (G != 8 && G != 16) return -1;
  return run_problem(10, G, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
