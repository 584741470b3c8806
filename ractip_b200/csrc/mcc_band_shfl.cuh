// mcc_band_shfl.cuh -- the device's variants of the split-sum band phases
// (inside_band_A / outside_band_A of mcc_core.h) that fetch every element of the streamed
// table ONCE per warp and pass it along the lanes with warp shuffles.
//
// In the band formulation a thread keeps BAND accumulators (one per diagonal e of the band)
// for its row and needs, at every step, BAND elements B(e) of the second operand.  Those
// elements are shared with the neighbouring rows:
//   inside   M/Q sums : B_a(i, e)   = B_{a-1}(i+1, e-1)     (previous step of the right neighbour)
//   outside  PR sum   : B_t(k, e)   = B_{t-1}(k+1, e+1)
//   outside  ML-left  : B_i(l, e)   = B_i(l+e, 0)           (same step, e lanes to the right)
// so a lane loads ONE new element per step and per sum instead of BAND; the L2 -> SM traffic of
// the phase drops ~2.5x.
// A warp owns 28 rows; its last 4 lanes shadow the next warp's first rows to feed the chain.
// Loads of 4 consecutive steps are issued together (the phase is latency-bound otherwise).
// Same sums in a different association order than the direct forms (a slice covers a contiguous
// run of steps instead of every S-th one).  For two strands the outside forms here and in
// mcc_wide_shfl.cuh skip the PR / ML-left terms of cells that do not join the strands (pr_live,
// ml_live, the nick test of cand) and leave other values than the direct forms in those PRB / MLB
// cells: the outside pass finishes only inter-strand cells (cross_lo .. cross_hi) and never reads them.  The host emulation runs these forms too, with each warp's
// lanes as fibers that meet at every shuffle (tests/emul/warp_emul.h).
#ifndef RP_MCC_BAND_SHFL_CUH
#define RP_MCC_BAND_SHFL_CUH

#include "mcc_core.h"

namespace rp {

__device__ __forceinline__ double shfl_down_f64(double v, int delta) { return __shfl_down_sync(0xffffffffu, v, delta); }
// starts the line of `p` towards the L2 (no register, no scoreboard slot); nothing in the host emulation
__device__ __forceinline__ void prefetch_l2(const void* p) {
#ifdef __CUDA_ARCH__
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#else
  (void)p;
#endif
}
// fine-grained probes (RP_PROFILE): thread 0 accumulates the cycles between two marks into slot k
#define RP_MARK(k)                                                                                       \
  do {                                                                                                   \
    if (RP_PROF(c) && tid == 0) {                                                                            \
      const long long now__ = clock64();                                                                 \
      atomicAdd(reinterpret_cast<unsigned long long*>(RP_PROF(c) + (k)), (unsigned long long)(now__ - tmark)); \
      atomicAdd(reinterpret_cast<unsigned long long*>(RP_PROF(c) + 32 + (k)), 1ull);                         \
      tmark = clock64();                                                                                 \
    }                                                                                                    \
  } while (0)

// Work split of the shuffle variants: a warp owns HW = 28 rows; lanes 28..31 shadow the first rows
// of the next warp and only feed the shuffle chain (a value needs BAND-1 = 4 hops to cross over).
constexpr int HW = 32 - (BAND - 1);
struct SplitW {
  int W;    // warps per slice
  int S;    // slices
  int CP;   // partial-sum stride per slice (>= C)
};
__device__ __forceinline__ SplitW make_split_w(int C, int T) {
  SplitW s;
  s.W = (C + HW - 1) / HW;
  s.S = (T / 32) / s.W;
  if (s.S < 1) s.S = 1;
  s.CP = s.W * HW;
  return s;
}
// partial (sum w, diagonal e, slice sl, row cell) at part[((w*BAND+e)*S + sl)*CP + cell]

// NB: steps whose loads are issued together (4 with 128 registers per thread, 2 in the 64-register build)
template <int NB = 4>
__device__ __forceinline__ void inside_band_A_shfl(const Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const SplitW sp = make_split_w(C, T);
  const int warp = tid >> 5, lane = tid & 31;
  const int slice = warp / sp.W, S = sp.S;
  if (slice >= S) return;
  const int cell = (warp - slice * sp.W) * HW + lane;
  const bool own = lane < HW && cell < C;          // this lane accumulates and writes
  const int i = i0 + cell;
  const bool rowok = i <= c.n - d0;                // the row exists on the band's first diagonal: its B(0) stream is real
  const int ds = c.dstep();
  double m[BAND], q[BAND];
#pragma unroll
  for (int e = 0; e < BAND; e++) m[e] = q[e] = 0.;
  long long tmark = (RP_PROF(c) && tid == 0) ? clock64() : 0;
  if (!(RP_DBG(c) & 2)) {
    const int amax = d0 - 1;
    const int lim = d0 - TURN - 2;
    const int askip = c.cp > 0 ? c.cp - 1 - i : -1;
    const long es = ds;
    if (own) {  // head of the q-split, a <= TURN
      for (int a = slice; a <= TURN && a <= amax; a += S) {
        const double A = TB(c, T_Q, a, i);
        const double* B = c.ptr(T_QQ, d0 - 1 - a, i + 1 + a);
        const int emin = a - lim;
#pragma unroll
        for (int e = 0; e < BAND; e++)
          if (e >= emin && e <= a) q[e] += A * B[e * es];
      }
    }
    RP_MARK(26);
    // main part, TURN < a <= lim: a contiguous run per slice, 4 steps' loads in flight at a time
    const int len = lim - TURN;
    if (len > 0) {
      const int per = (len + S - 1) / S;
      const int a_lo = TURN + 1 + slice * per;
      int a_hi = a_lo + per - 1;
      if (a_hi > lim) a_hi = lim;
      double bm[BAND], bq[BAND];
#pragma unroll
      for (int e = 0; e < BAND; e++) bm[e] = bq[e] = 0.;
      if (a_lo <= a_hi && rowok) {   // prime the chain: elements e >= 1 of the first step, loaded directly
        const double* Bm = c.ptr(T_QM1, d0 - 1 - a_lo, i + 1 + a_lo);
        const double* Bq = c.ptr(T_QQ, d0 - 1 - a_lo, i + 1 + a_lo);
#pragma unroll
        for (int e = 1; e < BAND; e++) { bm[e] = Bm[e * es]; bq[e] = Bq[e * es]; }
      }
      bool first = true;
#pragma unroll 1
      for (int a = a_lo; a <= a_hi; a += NB) {
        double Am[NB], Aq[NB], b0m[NB], b0q[NB];
#pragma unroll
        for (int u = 0; u < NB; u++) {
          const int au = a + u;
          const bool on = au <= a_hi;
          Am[u] = (on && own && au != askip) ? TB(c, T_QM, au, i) : 0.;
          Aq[u] = (on && own) ? TB(c, T_Q, au, i) : 0.;
          b0m[u] = (on && rowok) ? TB(c, T_QM1, d0 - 1 - au, i + 1 + au) : 0.;
          b0q[u] = (on && rowok) ? TB(c, T_QQ, d0 - 1 - au, i + 1 + au) : 0.;
        }
#pragma unroll
        for (int u = 0; u < NB; u++) {
          if (a + u <= a_hi) {
            if (!first) {
#pragma unroll
              for (int e = BAND - 1; e >= 1; e--) {
                bm[e] = shfl_down_f64(bm[e - 1], 1);
                bq[e] = shfl_down_f64(bq[e - 1], 1);
              }
            }
            first = false;
            bm[0] = b0m[u];
            bq[0] = b0q[u];
#pragma unroll
            for (int e = 0; e < BAND; e++) { m[e] += Am[u] * bm[e]; q[e] += Aq[u] * bq[e]; }
          }
        }
      }
    }
    RP_MARK(27);
    if (own) {  // tail, lim < a <= amax
      const int a0 = lim + 1 > TURN + 1 ? lim + 1 : TURN + 1;
      for (int a = a0 + slice; a <= amax; a += S) {
        const double Am = (a == askip) ? 0. : TB(c, T_QM, a, i);
        const double Aq = TB(c, T_Q, a, i);
        const double* Bm = c.ptr(T_QM1, d0 - 1 - a, i + 1 + a);
        const double* Bq = c.ptr(T_QQ, d0 - 1 - a, i + 1 + a);
        const int emin = a - lim;
#pragma unroll
        for (int e = 0; e < BAND; e++)
          if (e >= emin) { m[e] += Am * Bm[e * es]; q[e] += Aq * Bq[e * es]; }
      }
    }
  }
  RP_MARK(28);
  if (!own) return;
#pragma unroll
  for (int e = 0; e < BAND; e++) {
    sh.part[((size_t)e * S + slice) * sp.CP + cell] = m[e];
    sh.part[((size_t)(BAND + e) * S + slice) * sp.CP + cell] = q[e];
  }
}
__device__ __forceinline__ void inside_band_B_shfl(Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const SplitW sp = make_split_w(C, T);
  for (int x = tid; x < BAND * C; x += T) {
    const int e = x / C, cell = x % C, i = i0 + cell;
    if (i + d0 + e > c.n) continue;
    double m = 0., q = 0.;
    for (int s = 0; s < sp.S; s++) {
      m += sh.part[((size_t)e * sp.S + s) * sp.CP + cell];
      q += sh.part[((size_t)(BAND + e) * sp.S + s) * sp.CP + cell];
    }
    TB(c, T_QM2, d0 + e, i) = m;
    TB(c, T_QS, d0 + e, i) = q;
  }
}

template <int NB = 4>
__device__ __forceinline__ void outside_band_A_shfl(const Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T;
  const SplitW sp = make_split_w(C, T);
  const int warp = tid >> 5, lane = tid & 31;
  const int slice = warp / sp.W, S = sp.S;
  if (slice >= S) return;
  const int cell = (warp - slice * sp.W) * HW + lane;
  const bool own = lane < HW && cell < C;
  const int r = r0 + cell;
  const int n = c.n, ds = c.dstep(), ps = c.pstep();
  double pr[BAND], ml[BAND];
#pragma unroll
  for (int e = 0; e < BAND; e++) pr[e] = ml[e] = 0.;
  long long tmark = (RP_PROF(c) && tid == 0) ? clock64() : 0;
  if (!(RP_DBG(c) & 2)) {
    {  // the qb entries the ML part asks for below were written a whole pass ago: start them towards the L2 now
      // (a prefetch holds no register and no scoreboard slot, unlike the loads themselves)
      const int l = d0 - BAND + 2 + r, k0 = l - d0;
      if (own && l <= n) {
#pragma unroll
        for (int e = 0; e < BAND; e++) {
          const int k = k0 + e, d = d0 - e;
          if (k > 2 && d > TURN) prefetch_l2(c.ptr(T_QB, d, k));
        }
      }
    }
    {  // PR, row k; t = j - (k+d0+TURN+3)
      const int k = 1 + r;
      const int tmax = n - k - d0 - (TURN + 3);   // decreases along the lanes: a lane past its tmax feeds zeros
      int ecell = k + d0 - n;
      if (ecell < 0) ecell = 0;
      const long es = ds - ps;
      if (own) {
        for (int t = -(BAND - 1) + slice; t < 0 && t <= tmax; t += S) {
          const double A = TB(c, T_MC, d0 + TURN + 3 + t, k);
          const double* B = c.ptr(T_QM, TURN + 1 + t, k + d0 + 1);
          const int emin = -t > ecell ? -t : ecell;
#pragma unroll
          for (int e = 0; e < BAND; e++)
            if (e >= emin) pr[e] += A * B[e * es];
        }
      }
      // main part t = 0 .. tmax, a contiguous run per slice; the warp walks to lane 0's (largest) tmax
      const int tmax0 = __shfl_sync(0xffffffffu, tmax, 0);
      // two strands: only inter-strand cells are finished in the outside pass (cross_lo / cross_hi): a warp whose
      // rows all lie on strand 2 has nothing to sum
      const bool pr_live = c.cp <= 0 || 1 + r0 + (warp - slice * sp.W) * HW < c.cp;
      if (tmax0 >= 0 && pr_live) {
        const int per = (tmax0 + 1 + S - 1) / S;
        const int t_lo = slice * per;
        int t_hi = t_lo + per - 1;
        if (t_hi > tmax0) t_hi = tmax0;
        double bv[BAND];
#pragma unroll
        for (int e = 0; e < BAND; e++) bv[e] = 0.;
        if (t_lo <= t_hi && t_lo <= tmax) {  // prime the chain: elements e < BAND-1 of the first step
          const double* B = c.ptr(T_QM, TURN + 1 + t_lo, k + d0 + 1);
#pragma unroll
          for (int e = 0; e < BAND - 1; e++) bv[e] = B[e * es];
        }
        bool first = true;
#pragma unroll 1
        for (int t = t_lo; t <= t_hi; t += NB) {
          double A[NB], b4[NB];
#pragma unroll
          for (int u = 0; u < NB; u++) {
            const int tu = t + u;
            const bool on = tu <= t_hi && tu <= tmax;
            A[u] = (on && own) ? TB(c, T_MC, d0 + TURN + 3 + tu, k) : 0.;
            b4[u] = on ? *(c.ptr(T_QM, TURN + 1 + tu, k + d0 + 1) + (BAND - 1) * es) : 0.;
          }
#pragma unroll
          for (int u = 0; u < NB; u++) {
            if (t + u <= t_hi) {
              if (!first) {
#pragma unroll
                for (int e = 0; e < BAND - 1; e++) bv[e] = shfl_down_f64(bv[e + 1], 1);
              }
              first = false;
              bv[BAND - 1] = b4[u];
#pragma unroll
              for (int e = 0; e < BAND; e++)
                if (e >= ecell) pr[e] += A[u] * bv[e];
            }
          }
        }
      }
    }
    RP_MARK(29);
    {  // ML-left, column l; cells (k0+e, l), k0 = l-d0; i <= k0+e-TURN-3
      const int l = d0 - BAND + 2 + r, k0 = l - d0;
      unsigned need = 0;
      if (own && l <= n) {
        // the five qb look-ups in one round trip (a short-circuit chain would serialise them)
        double qbv[BAND];
        bool cand[BAND];
#pragma unroll
        for (int e = 0; e < BAND; e++) {
          const int k = k0 + e, d = d0 - e;
          cand[e] = k > 2 && d > TURN && pair_type(base(c, k), base(c, l)) != 0 && (c.cp <= 0 || (k < c.cp && l >= c.cp));
          qbv[e] = cand[e] ? TB(c, T_QB, d, k) : 0.;
        }
#pragma unroll
        for (int e = 0; e < BAND; e++)
          if (cand[e] && qbv[e] != 0.) need |= 1u << e;
      }
      RP_MARK(30);
      const int imax = k0 + (BAND - 1) - TURN - 3, imain = k0 - TURN - 3;
      // main part: B(e) = qm(i+1, k0+e-1) is the B(0) of the lane e places to the right, same step
      const int imain_hi = __shfl_sync(0xffffffffu, imain, HW - 1);   // largest among the owning lanes
      // (two strands: a warp whose columns all lie on strand 1 has no inter-strand cell)
      const bool ml_live = c.cp <= 0 || d0 - BAND + 2 + r0 + (warp - slice * sp.W) * HW + HW - 1 >= c.cp;
#pragma unroll 1
      for (int i = 1 + slice; ml_live && i <= imain_hi; i += NB * S) {
        double A[NB], b0[NB];
#pragma unroll
        for (int u = 0; u < NB; u++) {
          const int iu = i + u * S;
          const int row0 = k0 - 2 - iu;   // diagonal of B(0)
          A[u] = (need != 0 && iu <= imain) ? TB(c, T_PRML, l - iu, iu) : 0.;
          b0[u] = (iu <= imain_hi && row0 >= 0 && k0 - 1 <= n) ? *(c.ptr(T_QM, 0, iu + 1) + (long)row0 * ds) : 0.;   // qm(iu+1, k0-1)
        }
#pragma unroll
        for (int u = 0; u < NB; u++) {
          double bv[BAND];
          bv[0] = b0[u];
#pragma unroll
          for (int e = 1; e < BAND; e++) bv[e] = shfl_down_f64(b0[u], e);
#pragma unroll
          for (int e = 0; e < BAND; e++)
            if ((need >> e) & 1) ml[e] += A[u] * bv[e];
        }
      }
      if (need) {
        const int it0 = imain + 1 > 1 ? imain + 1 : 1;
        for (int i = it0 + slice; i <= imax; i += S) {   // tail: only the cells further right (larger k)
          const double A = TB(c, T_PRML, l - i, i);
          const double* B = c.ptr(T_QM, 0, i + 1) + (long)(k0 - 2 - i) * ds;
          const int emin = i - k0 + TURN + 3;
#pragma unroll
          for (int e = 0; e < BAND; e++)
            if (e >= emin && ((need >> e) & 1)) ml[e] += A * B[(long)e * ds];
        }
      }
    }
  }
  RP_MARK(31);
  if (!own) return;
#pragma unroll
  for (int e = 0; e < BAND; e++) {
    sh.part[((size_t)e * S + slice) * sp.CP + cell] = pr[e];
    sh.part[((size_t)(BAND + e) * S + slice) * sp.CP + cell] = ml[e];
  }
}
__device__ __forceinline__ void outside_band_B_shfl(Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T, n = c.n;
  const bool keep = c.kind == KIND_LINEAR && c.max_w > 0;
  const SplitW sp = make_split_w(C, T);
  for (int x = tid; x < BAND * C; x += T) {
    const int e = x / C, cell = x % C, r = r0 + cell, d = d0 - e;
    if (d < 1) continue;
    double a = 0., b = 0.;
    for (int s = 0; s < sp.S; s++) {
      a += sh.part[((size_t)e * sp.S + s) * sp.CP + cell];
      b += sh.part[((size_t)(BAND + e) * sp.S + s) * sp.CP + cell];
    }
    const int k = 1 + r;
    if (k + d <= n) {
      TB(c, T_PRB, d, k) = a;
      if (keep) RP_ST_STREAM(TB(c, T_XX, d, k), a);   // the unpaired-window pass reads PR again (unstru_windows)
    }
    const int l = d0 - BAND + 2 + r, k2 = l - d;
    if (l <= n && k2 >= 1) TB(c, T_MLB, d, k2) = b;
  }
}

}  // namespace rp
#endif
