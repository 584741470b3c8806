// emul.cpp -- TEST INFRASTRUCTURE.  Runs the kernels' per-thread phase
// functions (ractip_b200/csrc/mcc_core.h, mcc_driver.h) on the host so that the
// CUDA kernels' logic can be checked against the oracle on a CPU-only box: one
// emulated thread after another (SerialExecT, the direct forms of the split
// sums), or warp by warp in lockstep (wemu::WarpExecT, warp_emul.h: the
// device's warp-shuffle forms).  Never loaded by the product.
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include "warp_emul.h"   // first: the host stand-ins for the CUDA intrinsics

#include "dev_model.h"
#include "mcc_driver.h"
#include "seq_encode.h"

namespace {
// The executor (contract at the top of mcc_driver.h) of G CTAs that share one problem, run as one serial flow with one
// copy of shared memory: it runs the work of every rank, rank after rank, as the device deals it out.
template <int W, int G = 1>
struct SerialExecT {
  static constexpr int kCtas = G;
  static constexpr bool kShfl = false;   // the direct forms of the split sums, thread by thread
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
  int error() const { return 0; }
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
// G = 8, 16 (band = 10 only): solve_mcc_wide on a cluster of G CTAs.
// lockstep: run with the warp-lockstep executor as the device build does -- the shuffle forms of the split sums,
// kBatch 2 for solve_mcc (mcc_persistent<2,5>), 4 otherwise -- in shared memory of the device's sizes, poisoned;
// returns its hazard code (warp_emul.h) if it reports one.
static int run_problem(int band, int G, bool lockstep, const rp_model* m, const char* seq, int n, int cp, int kind,
                       int max_w, int n1, int n2, float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
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
  // shared memory: the serial runs zero it; the lockstep runs poison it, as the device leaves it undefined
  std::vector<double> smem(rp::shared_bytes(T, W) / sizeof(double) + 2, lockstep ? 1e300 : 0.0);
  rp::Shared sh;
  rp::carve_shared(sh, smem.data(), T, W);
  double lz[3] = {0, 0, 0};
  rp::Ctx c;
  rp::bind_ctx(c, &g_model, S.data(), p, ws.data());
  int err = 0;
  auto wide = [&](auto&& ex) {
    rp::solve_mcc_wide(ex, c, p, dense.data(), lz, sh);
    err = ex.error();
  };
  auto band_kernel = [&](auto&& ex) {
    // the band kernel's dynamic shared memory as its build sizes it, poisoned
    std::vector<double> bsm(rp::band_shared_doubles(n, T, ex.kShfl) + 2, 1e300);
    rp::solve_band(ex, c, p, dense.data(), lz, bsm.data());
    err = ex.error();
  };
  if (lockstep) {
    if (G == 8) wide(wemu::WarpExecT<8, 4, 10>(T));
    else if (G == 16) wide(wemu::WarpExecT<16, 4, 10>(T));
    else if (band == 10) wide(wemu::WarpExecT<1, 4, 10>(T));
    else if (band == 1) band_kernel(wemu::WarpExecT<1, 4, rp::BAND>(T));
    else if (band == 0) {
      wemu::WarpExecT<1, 2, rp::BAND> ex(T);
      rp::solve_mcc(ex, c, p, dense.data(), lz, sh);
      err = ex.error();
    } else {
      return -1;
    }
  } else if (G == 8) {
    wide(SerialExecT<10, 8>{T});
  } else if (G == 16) {
    wide(SerialExecT<10, 16>{T});
  } else if (band == 5) {
    wide(SerialExecT<5>{T});
  } else if (band == 8) {
    wide(SerialExecT<8>{T});
  } else if (band == 10) {
    wide(SerialExecT<10>{T});
  } else if (band == 15) {
    wide(SerialExecT<15>{T});
  } else if (band) {
    band_kernel(SerialExec{T});
  } else {
    SerialExec ex{T};
    rp::solve_mcc(ex, c, p, dense.data(), lz, sh);
  }
  if (err) return err;
  if (p.out_bp >= 0) std::memcpy(bp, dense.data(), nbp * sizeof(float));
  if (p.out_up >= 0) std::memcpy(up, dense.data() + nbp, nup * sizeof(float));
  if (p.out_hp >= 0) std::memcpy(hp, dense.data() + nbp + nup, nhp * sizeof(float));
  if (logz) *logz = lz[0];
  return 0;
}

extern "C" int emul_problem(const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1, int n2,
                            float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  return run_problem(0, 1, false, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
extern "C" int emul_wide_problem(int W, const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1,
                                 int n2, float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  if (W != 5 && W != 8 && W != 10 && W != 15) return -1;
  return run_problem(W, 1, false, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
extern "C" int emul_band_problem(const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1, int n2,
                                 float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  return run_problem(1, 1, false, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
extern "C" int emul_cluster_problem(int G, const rp_model* m, const char* seq, int n, int cp, int kind, int max_w, int n1,
                                    int n2, float th_hy, int T, float* bp, float* up, float* hp, double* logz) {
  if (G != 8 && G != 16) return -1;
  return run_problem(10, G, false, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}
// one problem on the warp-lockstep executor, as a device route runs it: route 0 solve_mcc (mcc_persistent<2,5>),
// 1 solve_band (mcc_band_kernel), 10 solve_mcc_wide<10> (mcc_persistent<1,10>; G = 8, 16: mcc_cluster_kernel)
extern "C" int emul_lockstep_problem(int route, int G, const rp_model* m, const char* seq, int n, int cp, int kind,
                                     int max_w, int n1, int n2, float th_hy, int T, float* bp, float* up, float* hp,
                                     double* logz) {
  if (!(route == 0 || route == 1 || route == 10) || !(G == 1 || (route == 10 && (G == 8 || G == 16)))) return -1;
  return run_problem(route, G, true, m, seq, n, cp, kind, max_w, n1, n2, th_hy, T, bp, up, hp, logz);
}

// ---- one split-sum band on dense random tables, shuffle form against direct form

namespace {
// Fills every table the A phases of the split sums read as prologue2 leaves diagonals 0..TURN -- q = a scale factor
// on the cells of the triangle, every other table 0 -- and with seeded values in [0.5, 1.5) on diagonals > TURN
// (the whole row, cells past the triangle's edge too).  Everything else stays poisoned.
void fill_split_tables(const rp::Ctx& c, unsigned seed) {
  std::mt19937_64 g(seed);
  std::uniform_real_distribution<double> u(0.5, 1.5);
  const int n = c.n;
  for (int t : {rp::T_Q, rp::T_QQ, rp::T_QM, rp::T_QM1, rp::T_MC, rp::T_QB, rp::T_PRML})
    for (int d = 0; d < n; d++)
      for (int i = 0; i <= n; i++) {
        const double v = u(g);
        TB(c, t, d, i) = d > rp::TURN ? v : (t == rp::T_Q && i >= 1 && i + d <= n) ? v : 0.;
      }
  for (int t : {rp::T_QMR, rp::T_PRMLR})
    for (int i = 1; i <= n; i++)
      for (int j = 0; j <= n; j++) {
        const double v = u(g);
        *c.rptr(t, i, j) = j - i > rp::TURN ? v : 0.;
      }
}

template <int W, class Exec>
int run_split(Exec&& ex, const rp::Ctx& c0, int T, int d, int side, double* ws) {
  std::vector<double> smem(rp::shared_bytes(T, W) / sizeof(double) + 2, 1e300);
  rp::Shared sh;
  rp::carve_shared(sh, smem.data(), T, W);
  rp::Ctx c = c0;
  c.ws = ws;
  if (side == 0) rp::split_sums_inside<W>(ex, c, sh, d);
  else rp::split_sums_outside<W>(ex, c, sh, d);
  return ex.error();
}

template <int W, int NB, int G>
int split_pair(const rp::Ctx& c, int T, int d, int side, double* ws_lock, double* ws_serial) {
  const int e = run_split<W>(wemu::WarpExecT<G, NB, W>(T), c, T, d, side, ws_lock);
  run_split<W>(SerialExecT<W, G>{T}, c, T, d, side, ws_serial);
  return e;
}
}  // namespace

// The split sums of the band that starts at diagonal d (side 0: inside, d .. d+W-1; side 1: outside, d .. d-W+1) of
// a problem of length n (cp > 0: two strands), W = BAND or 10, on G = 1 or 8 CTAs of T threads, kBatch NB (BAND only):
// the workspace is filled by fill_split_tables(seed) and copied to ws_init, then the band's split sums run from
// those bytes once on the warp-lockstep executor (result in ws_lock) and once on the serial one (ws_serial).  Each
// buffer holds rp::slot_doubles(n) doubles (emul_slot_doubles).  Returns the lockstep executor's hazard code, or -1.
extern "C" int emul_split_sums(const rp_model* m, int W, int NB, int G, int T, const char* seq, int n, int cp, int d,
                               int side, unsigned seed, double* ws_init, double* ws_lock, double* ws_serial) {
  static const rp_model* built = nullptr;   // (called hundreds of times in a row with one model)
  if (m != built) {
    int rc = rp::build_dev_model(*m, &g_model);
    if (rc) return rc;
    built = m;
  }
  if (d <= rp::TURN || d >= n) return -1;
  std::vector<uint8_t> S(n + 16, 0);
  for (int i = 1; i <= n; i++) S[i] = rp::encode_base(seq[i - 1]);
  rp::Problem p;
  std::memset(&p, 0, sizeof p);
  p.n = n; p.cp = cp;
  p.kind = cp > 0 ? rp::KIND_COFOLD : rp::KIND_LINEAR;
  p.max_w = cp > 0 ? 0 : 15;   // a linear problem keeps PR for the unpaired-window pass (T_XX)
  const size_t nd = rp::slot_doubles(n);
  std::fill(ws_init, ws_init + nd, 1e300);
  rp::Ctx c;
  rp::bind_ctx(c, &g_model, S.data(), p, ws_init);
  fill_split_tables(c, seed);
  std::memcpy(ws_lock, ws_init, nd * sizeof(double));
  std::memcpy(ws_serial, ws_init, nd * sizeof(double));
  const int key = W * 1000 + NB * 100 + G;
  switch (key) {
    case rp::BAND * 1000 + 200 + 1: return split_pair<rp::BAND, 2, 1>(c, T, d, side, ws_lock, ws_serial);
    case rp::BAND * 1000 + 400 + 1: return split_pair<rp::BAND, 4, 1>(c, T, d, side, ws_lock, ws_serial);
    case rp::BAND * 1000 + 200 + 8: return split_pair<rp::BAND, 2, 8>(c, T, d, side, ws_lock, ws_serial);
    case rp::BAND * 1000 + 400 + 8: return split_pair<rp::BAND, 4, 8>(c, T, d, side, ws_lock, ws_serial);
    case 10 * 1000 + 200 + 1: return split_pair<10, 2, 1>(c, T, d, side, ws_lock, ws_serial);
    case 10 * 1000 + 400 + 1: return split_pair<10, 4, 1>(c, T, d, side, ws_lock, ws_serial);
    case 10 * 1000 + 200 + 8: return split_pair<10, 2, 8>(c, T, d, side, ws_lock, ws_serial);
    case 10 * 1000 + 400 + 8: return split_pair<10, 4, 8>(c, T, d, side, ws_lock, ws_serial);
    default: return -1;
  }
}
extern "C" long long emul_slot_doubles(int n) { return (long long)rp::slot_doubles(n); }
// Marks (1) the elements of a workspace slot the rest of the outside pass can read after the split sums of the band
// d0 .. d0-W+1, leaving 0 on the PRB / MLB cells of a two-strand problem (cp > 0) that do not join the strands: the
// outside pass finishes only inter-strand cells (cross_lo .. cross_hi), so the shuffle forms skip the others.
extern "C" void emul_outside_read_mask(int n, int cp, int d0, int W, uint8_t* mask) {
  const size_t nd = rp::slot_doubles(n);
  std::memset(mask, 1, nd);
  if (cp <= 0) return;
  rp::Problem p;
  std::memset(&p, 0, sizeof p);
  p.n = n; p.cp = cp;
  rp::Ctx c;
  rp::bind_ctx(c, &g_model, nullptr, p, nullptr);
  for (int d = d0; d > d0 - W && d >= 1; d--)
    for (int k = 1; k + d <= n; k++)
      if (!(k >= rp::cross_lo(c, d) && k <= rp::cross_hi(c, d)))
        for (int t : {rp::T_PRB, rp::T_MLB}) mask[c.off(t, d, k)] = 0;
}
