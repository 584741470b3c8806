// mcc_wide_shfl.cuh -- the device's far passes of the WIDE split-sum bands (mcc_core.h, "Wide bands"),
// general kernel, long problems.
//
// Same scheme as mcc_band_shfl.cuh -- a thread keeps one accumulator per diagonal of the band for its
// row, loads ONE new element of each streamed table per step and receives the others from its lane
// neighbours -- but for W = 10..15 diagonals instead of 5, so every element fetched from HBM feeds W
// FMAs.  A warp owns 32-(W-1) rows; the last W-1 lanes shadow the next warp's first rows.  The two
// sums of a pass run one after the other (W accumulators + W chain values each: both at once would
// not fit 128 registers).
//
// No masks in the inner loops.  Which (step, diagonal) pairs belong to the far pass follows from the
// data: chain slots that would hold an operand of the band itself are primed with 0 and stay 0 as
// they travel, and operands on diagonals <= TURN are stored zeros (prologue2).  Values that reach a
// cell outside the triangle come from outside their table row; such cells are never written.
#ifndef RP_MCC_WIDE_SHFL_CUH
#define RP_MCC_WIDE_SHFL_CUH

#include "mcc_band_shfl.cuh"
#include "mcc_core.h"

namespace rp {

// The far passes stream tens of MB per call that will not be touched again before the next pass of the
// same problem, by which time 147 other problems have streamed theirs: evict-first loads keep them from
// pushing the recent diagonals (the interior-loop operands, re-read for 32 diagonals) out of the L2.
__device__ __forceinline__ double ld_stream(const double* p) { return __ldcs(p); }

template <int W>
struct WideSplit {
  static constexpr int HWW = 32 - (W - 1);   // rows a warp owns
  int NW;   // warps per slice
  int S;    // slices
  int CP;   // partial-sum stride per slice (>= C)
  __device__ __forceinline__ WideSplit(int C, int T) {
    NW = (C + HWW - 1) / HWW;
    S = (T / 32) / NW;
    if (S < 1) S = 1;
    CP = NW * HWW;
  }
};
// load-batch depth of the far passes: one sum at a time leaves registers for 8 steps' loads
constexpr int WIDE_NB = 8;
// partial (sum w, diagonal e, slice sl, row cell) at part[((w*W+e)*S + sl)*CP + cell]

template <int W, int NB>
__device__ __forceinline__ void wide_inside_A_shfl(const Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const WideSplit<W> sp(C, T);
  const int warp = tid >> 5, lane = tid & 31;
  const int slice = warp / sp.NW, S = sp.S;
  if (slice >= S) return;
  const int cell = (warp - slice * sp.NW) * WideSplit<W>::HWW + lane;
  const bool own = lane < WideSplit<W>::HWW && cell < C;
  const int i = i0 + cell;
  const bool rowok = i <= c.n - d0;   // the row exists on the band's first diagonal: its e = 0 stream is real
  const long es = c.dstep();
  const int amax = d0 - 1;
  const int askip = c.cp > 0 ? c.cp - 1 - i : -1;   // split on the nick (M only)
  const int per = (amax + 1 + S - 1) / S;
  const int s_lo = slice * per;
  int s_hi = s_lo + per - 1;
  if (s_hi > amax) s_hi = amax;
#pragma unroll
  for (int sum = 0; sum < 2; sum++) {   // unrolled: the table ids must be compile-time constants (ring masks fold away)
    const int tA = sum ? T_Q : T_QM, tB = sum ? T_QQ : T_QM1;
    const int a_lo = (!sum && s_lo < TURN + 1) ? TURN + 1 : s_lo;   // qm vanishes on diagonals <= TURN
    const int a_hi = s_hi;
    double acc[W], bv[W];
#pragma unroll
    for (int e = 0; e < W; e++) acc[e] = bv[e] = 0.;
    if (a_lo <= a_hi && !(RP_DBG(c) & 2)) {
      {  // prime the chain: elements e >= 1 of the first step that are final (diagonal < d0) and inside their row
        const double* B = c.ptr(tB, d0 - 1 - a_lo, i + 1 + a_lo);
#pragma unroll
        for (int e = 1; e < W; e++) bv[e] = (e <= a_lo && i + d0 + e <= c.n) ? B[e * es] : 0.;
      }
      bool first = true;
#pragma unroll 1
      for (int a = a_lo; a <= a_hi; a += NB) {
        double A[NB], b0[NB];
#pragma unroll
        for (int u = 0; u < NB; u++) {
          const int au = a + u;
          const bool on = au <= a_hi;
          A[u] = (on && own && (sum || au != askip)) ? ld_stream(c.ptr(tA, au, i)) : 0.;
          b0[u] = (on && rowok) ? ld_stream(c.ptr(tB, d0 - 1 - au, i + 1 + au)) : 0.;
        }
#pragma unroll
        for (int u = 0; u < NB; u++) {
          if (a + u <= a_hi) {
            if (!first) {
#pragma unroll
              for (int e = W - 1; e >= 1; e--) bv[e] = shfl_down_f64(bv[e - 1], 1);
            }
            first = false;
            bv[0] = b0[u];
#pragma unroll
            for (int e = 0; e < W; e++) acc[e] += A[u] * bv[e];
          }
        }
      }
    }
    if (own) {
#pragma unroll
      for (int e = 0; e < W; e++) sh.part[((size_t)(sum * W + e) * S + slice) * sp.CP + cell] = acc[e];
    }
  }
}
template <int W>
__device__ __forceinline__ void wide_inside_B_shfl(Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const WideSplit<W> sp(C, T);
  for (int x = tid; x < W * C; x += T) {
    const int e = x / C, cell = x % C, i = i0 + cell;
    if (i + d0 + e > c.n) continue;
    double m = 0., q = 0.;
    for (int s = 0; s < sp.S; s++) {
      m += sh.part[((size_t)e * sp.S + s) * sp.CP + cell];
      q += sh.part[((size_t)(W + e) * sp.S + s) * sp.CP + cell];
    }
    TB(c, T_QM2, d0 + e, i) = m;
    TB(c, T_QS, d0 + e, i) = q;
  }
}

template <int W, int NB>
__device__ __forceinline__ void wide_outside_A_shfl(const Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T;
  const WideSplit<W> sp(C, T);
  const int warp = tid >> 5, lane = tid & 31;
  const int slice = warp / sp.NW, S = sp.S;
  if (slice >= S) return;
  constexpr int HWW = WideSplit<W>::HWW;
  const int cell = (warp - slice * sp.NW) * HWW + lane;
  const bool own = lane < HWW && cell < C;
  const int r = r0 + cell;
  const int n = c.n, ds = c.dstep(), ps = c.pstep();
  {  // PR, row k: steps t = -(TURN+1) .. tmax; Mc(k, .) on diagonal d0+TURN+3+t, chain element e = qm on diagonal TURN+1+t+e
    const int k = 1 + r;
    const int tmax = n - k - d0 - (TURN + 3);   // decreases along the lanes: a lane past its tmax feeds zeros
    const long es = ds - ps;
    double acc[W], bv[W];
#pragma unroll
    for (int e = 0; e < W; e++) acc[e] = bv[e] = 0.;
    const int tmax0 = __shfl_sync(0xffffffffu, tmax, 0);
    const int tfirst = -(TURN + 1);
    // two strands: only inter-strand cells are finished in the outside pass (cross_lo / cross_hi), so a warp whose
    // rows all lie on strand 2 has nothing to sum (its zero partials are still written)
    const bool pr_live = c.cp <= 0 || 1 + r0 + (warp - slice * sp.NW) * HWW < c.cp;
    if (tmax0 >= tfirst && pr_live && !(RP_DBG(c) & 2)) {
      const int per = (tmax0 - tfirst + 1 + S - 1) / S;
      const int t_lo = tfirst + slice * per;
      int t_hi = t_lo + per - 1;
      if (t_hi > tmax0) t_hi = tmax0;
      if (t_lo <= t_hi && t_lo <= tmax) {   // prime the chain: elements e < W-1 of the first step
        const double* B = c.ptr(T_QM, TURN + 1 + t_lo, k + d0 + 1);
#pragma unroll
        for (int e = 0; e < W - 1; e++) bv[e] = (k + d0 + 1 - e >= 1) ? B[e * es] : 0.;
      }
      bool first = true;
#pragma unroll 1
      for (int t = t_lo; t <= t_hi; t += NB) {
        double A[NB], bn[NB];
#pragma unroll
        for (int u = 0; u < NB; u++) {
          const int tu = t + u;
          const bool on = tu <= t_hi && tu <= tmax;
          A[u] = (on && own) ? ld_stream(c.ptr(T_MC, d0 + TURN + 3 + tu, k)) : 0.;
          bn[u] = (on && k + d0 + 2 - W >= 1) ? ld_stream(c.ptr(T_QM, TURN + 1 + tu, k + d0 + 1) + (W - 1) * es) : 0.;
        }
#pragma unroll
        for (int u = 0; u < NB; u++) {
          if (t + u <= t_hi) {
            if (!first) {
#pragma unroll
              for (int e = 0; e < W - 1; e++) bv[e] = shfl_down_f64(bv[e + 1], 1);
            }
            first = false;
            bv[W - 1] = bn[u];
#pragma unroll
            for (int e = 0; e < W; e++) acc[e] += A[u] * bv[e];
          }
        }
      }
    }
    if (own) {
#pragma unroll
      for (int e = 0; e < W; e++) sh.part[((size_t)e * S + slice) * sp.CP + cell] = acc[e];
    }
  }
  {  // ML-left, column l: cells (k0+e, l); steps i = 1 .. k0-2 (PRML(i,l) final); element e = qm(i+1, k0+e-1) is the
     // e = 0 element of the lane e places to the right, same step
    const int l = d0 - W + 2 + r, k0 = l - d0;
    double acc[W];
#pragma unroll
    for (int e = 0; e < W; e++) acc[e] = 0.;
    unsigned need = 0;
    if (own && l <= n) {
      double qbv[W];
      bool cand[W];
#pragma unroll
      for (int e = 0; e < W; e++) {
        const int k = k0 + e, d = d0 - e;
        cand[e] = k > 2 && d > TURN && pair_type(base(c, k), base(c, l)) != 0 && (c.cp <= 0 || (k < c.cp && l >= c.cp));
        qbv[e] = cand[e] ? TB(c, T_QB, d, k) : 0.;
      }
#pragma unroll
      for (int e = 0; e < W; e++)
        if (cand[e] && qbv[e] != 0.) need |= 1u << e;
    }
    const int ifar = k0 - 2;
    const int ifar_hi = __shfl_sync(0xffffffffu, ifar, HWW - 1);   // largest among the owning lanes
    // (two strands: a warp whose columns all lie on strand 1 has no inter-strand cell)
    const bool ml_live = c.cp <= 0 || d0 - W + 2 + r0 + (warp - slice * sp.NW) * HWW + HWW - 1 >= c.cp;
    if (ml_live && !(RP_DBG(c) & 2)) {
#pragma unroll 1
      for (int i = 1 + slice; i <= ifar_hi; i += NB * S) {
        double A[NB], b0[NB];
#pragma unroll
        for (int u = 0; u < NB; u++) {
          const int iu = i + u * S;
          const int row0 = k0 - 2 - iu;   // diagonal of this lane's e = 0 element
          A[u] = (need != 0 && iu <= ifar) ? ld_stream(c.rptr(T_PRMLR, iu, l)) : 0.;   // (row-major copies: lanes are neighbours)
          b0[u] = (iu <= ifar_hi && row0 >= 0 && k0 - 1 <= n) ? ld_stream(c.rptr(T_QMR, iu + 1, k0 - 1)) : 0.;
        }
#pragma unroll
        for (int u = 0; u < NB; u++) {
          double bv[W];
          bv[0] = b0[u];
#pragma unroll
          for (int e = 1; e < W; e++) bv[e] = shfl_down_f64(b0[u], e);
#pragma unroll
          for (int e = 0; e < W; e++)
            if ((need >> e) & 1) acc[e] += A[u] * bv[e];
        }
      }
    }
    if (own) {
#pragma unroll
      for (int e = 0; e < W; e++) sh.part[((size_t)(W + e) * S + slice) * sp.CP + cell] = acc[e];
    }
  }
}
template <int W>
__device__ __forceinline__ void wide_outside_B_shfl(Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T, n = c.n;
  const WideSplit<W> sp(C, T);
  for (int x = tid; x < W * C; x += T) {
    const int e = x / C, cell = x % C, r = r0 + cell, d = d0 - e;
    if (d < 1) continue;
    double a = 0., b = 0.;
    for (int s = 0; s < sp.S; s++) {
      a += sh.part[((size_t)e * sp.S + s) * sp.CP + cell];
      b += sh.part[((size_t)(W + e) * sp.S + s) * sp.CP + cell];
    }
    const int k = 1 + r;
    if (k + d <= n) TB(c, T_PRB, d, k) = a;
    const int l = d0 - W + 2 + r, k2 = l - d;
    if (l <= n && k2 >= 1) TB(c, T_MLB, d, k2) = b;
  }
}

}  // namespace rp
#endif
