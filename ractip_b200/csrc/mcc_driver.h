// mcc_driver.h -- the phase schedules, written once against an "executor".  kernels.cu instantiates them with
// CtaExecT (one CTA, or the G CTAs of a thread-block cluster that share one problem); tests/emul with a serial one.
//
//   solve_mcc        one problem per CTA, tables in HBM (the 64-register build)
//   solve_mcc_wide   one problem per CTA or per cluster, tables in HBM (long problems)
//   solve_band       one problem per CTA, interior-loop operands in shared memory
//
// An executor provides
//   nthreads()      threads per CTA
//   phase(id, f)    f(tid) on every thread of this CTA, then a CTA barrier
//   kWide           diagonals per split-sum band of solve_mcc_wide
//   kBatch          load-batch depth of the BAND-wide shuffle far passes (device only, mcc_band_shfl.cuh)
// and, when G = kCtas > 1 CTAs share one problem (a thread-block cluster), also
//   rank_begin(), rank_end()   the ranks of the CTAs whose work this flow of control runs: its own on the device,
//                              all G in the serial host emulation
//   sync()                     a barrier over the whole problem
// An executor without kCtas runs each problem on one CTA.  On top of these, chunks() deals a range of items out over
// the CTAs and flat() runs a pass over all threads of the problem (below).
#ifndef RP_MCC_DRIVER_H
#define RP_MCC_DRIVER_H

#include <type_traits>

#include "mcc_band.h"
#include "mcc_core.h"
#ifdef __CUDACC__
#include "mcc_band_shfl.cuh"
#include "mcc_wide_shfl.cuh"
#endif

namespace rp {

enum {
  PH_STAGE = 0, PH_PROLOGUE, PH_PROLOGUE2, PH_INSIDE_A, PH_INSIDE_B, PH_GENERIC_IN, PH_GENERIC_OUT, PH_OUTSIDE_A, PH_OUTSIDE_B,
  PH_WRITE_BP, PH_UN_ITEMS, PH_UN_DOMROWS, PH_UN_DOMCOLS, PH_UN_WINDOWS,
  PH_WRITE_HP, PH_LOGZ, PH_BAND_A, PH_BAND_B, PH_CFAC, PH_COUNT
};

// number of CTAs that share one problem under executor Exec
template <class Exec, class = void>
struct CtasOf { static constexpr int value = 1; };
template <class Exec>
struct CtasOf<Exec, std::void_t<decltype(Exec::kCtas)>> { static constexpr int value = Exec::kCtas; };

// chunk size of chunks(): `total` items spread over G CTAs, at most `cap` per chunk
RP_HD int deal_chunk(int total, int G, int cap) {
  int ch = (total + G - 1) / G;
  if (ch > cap) ch = cap;
  return ch < 1 ? 1 : ch;
}

// Deals [first, end) in chunks of deal_chunk(end - first, G, cap) over the G CTAs of the problem -- CTA r takes the
// chunks at first + r*chunk, stride G*chunk -- and calls body(i0, C) on each chunk's owner; then, for G > 1, a barrier
// over the problem (for G = 1 the CTA barrier the body's last phase ended with is one).
template <class Exec, class F>
RP_HD void chunks(Exec& ex, int first, int end, int cap, F body) {
  constexpr int G = CtasOf<Exec>::value;
  const int ch = deal_chunk(end - first, G, cap);
  if constexpr (G == 1) {
    for (int i0 = first; i0 < end; i0 += ch) body(i0, end - i0 < ch ? end - i0 : ch);
  } else {
    for (int r = ex.rank_begin(); r < ex.rank_end(); r++)
      for (int i0 = first + r * ch; i0 < end; i0 += G * ch) body(i0, end - i0 < ch ? end - i0 : ch);
    ex.sync();
  }
}

// f(tid, gt, GT) on all GT = G*nthreads() threads of the problem, gt = r*nthreads() + tid, then a barrier over the problem
template <class Exec, class F>
RP_HD void flat(Exec& ex, int id, F f) {
  constexpr int G = CtasOf<Exec>::value;
  const int T = ex.nthreads();
  if constexpr (G == 1) {
    ex.phase(id, [&](int tid) { f(tid, tid, T); });
  } else {
    for (int r = ex.rank_begin(); r < ex.rank_end(); r++) ex.phase(id, [&](int tid) { f(tid, r * T + tid, G * T); });
    ex.sync();
  }
}

// copies the sequence into shared memory `S` in one phase, together with the per-thread work `with(tid)`
template <class Exec, class F>
RP_HD void stage_sequence(Exec& ex, Ctx& c, uint8_t* S, F with) {
  const uint8_t* gS = c.S;
  const int n = c.n, T = ex.nthreads();
  ex.phase(PH_STAGE, [&](int tid) {
    for (int x = tid; x <= n + 1; x += T) S[x] = gS[x];
    with(tid);
  });
  c.S = S;
}

// log Z of the finished inside pass: 3 doubles per pair (s1, s2, s1&s2)
template <class Exec>
RP_HD void emit_logz(Exec& ex, Ctx& c, const Problem& p, double* logz) {
  if (!logz) return;
  if constexpr (CtasOf<Exec>::value > 1) {
    if (ex.rank_begin() != 0) return;   // the CTA of rank 0 writes it
  }
  ex.phase(PH_LOGZ, [&](int tid) {
    if (tid == 0) logz[(size_t)p.pair * 3 + p.which] = log(TB(c, T_Q, c.n - 1, 1)) + c.n * log(c.M->pf_scale);
  });
}

// Split sums of the band of W diagonals d .. d+W-1 (inside) / d .. d-W+1 (outside): inside_band_* / outside_band_*
// for W = BAND, the far pass wide_* for W > BAND; the shuffle forms on the device, the reference forms on the host.
// Rows are dealt in chunks of at most wide_chunk<W>(T), the rows one shuffle-form call takes.
template <int W, class Exec>
RP_HD void split_sums_inside(Exec& ex, Ctx& c, const Shared& sh, int d) {
  chunks(ex, 1, c.n - d + 1, wide_chunk<W>(sh.T), [&](int i0, int C) {
    ex.phase(PH_BAND_A, [&](int tid) {
#ifdef __CUDA_ARCH__
      if constexpr (W == BAND) inside_band_A_shfl<Exec::kBatch>(c, sh, d, i0, C, tid);
      else wide_inside_A_shfl<W, WIDE_NB>(c, sh, d, i0, C, tid);
#else
      if constexpr (W == BAND) inside_band_A(c, sh, d, i0, C, tid);
      else wide_inside_A<W>(c, sh, d, i0, C, tid);
#endif
    });
    ex.phase(PH_BAND_B, [&](int tid) {
#ifdef __CUDA_ARCH__
      if constexpr (W == BAND) inside_band_B_shfl(c, sh, d, i0, C, tid);
      else wide_inside_B_shfl<W>(c, sh, d, i0, C, tid);
#else
      if constexpr (W == BAND) inside_band_B(c, sh, d, i0, C, tid);
      else wide_inside_B<W>(c, sh, d, i0, C, tid);
#endif
    });
  });
}
template <int W, class Exec>
RP_HD void split_sums_outside(Exec& ex, Ctx& c, const Shared& sh, int d) {
  chunks(ex, 0, c.n - d + W - 1, wide_chunk<W>(sh.T), [&](int r0, int C) {
    ex.phase(PH_BAND_A, [&](int tid) {
#ifdef __CUDA_ARCH__
      if constexpr (W == BAND) outside_band_A_shfl<Exec::kBatch>(c, sh, d, r0, C, tid);
      else wide_outside_A_shfl<W, WIDE_NB>(c, sh, d, r0, C, tid);
#else
      if constexpr (W == BAND) outside_band_A(c, sh, d, r0, C, tid);
      else wide_outside_A<W>(c, sh, d, r0, C, tid);
#endif
    });
    ex.phase(PH_BAND_B, [&](int tid) {
#ifdef __CUDA_ARCH__
      if constexpr (W == BAND) outside_band_B_shfl(c, sh, d, r0, C, tid);
      else wide_outside_B_shfl<W>(c, sh, d, r0, C, tid);
#else
      if constexpr (W == BAND) outside_band_B(c, sh, d, r0, C, tid);
      else wide_outside_B<W>(c, sh, d, r0, C, tid);
#endif
    });
  });
}

// the unpaired-window pass of a finished single-strand problem (pf_unstru, src/ractip.cpp:371-375): reads the tables
// the two wavefronts left in the problem's workspace.  Run right after them (emit_outputs) or, for the band-kernel
// classes, later by unstru_kernel / solve_band_unpaired.
// `SM`: the model the table-driven gap loops read (DevModel, or the band kernel's shared-memory copy);
// `gfull`: DevModel::gfull or a shared-memory copy of it
template <class Exec, class MT>
RP_HD void emit_unpaired(Exec& ex, Ctx& c, const Problem& p, float* dense, const MT& SM, const double* gfull) {
  flat(ex, PH_UN_ITEMS, [&](int, int gt, int GT) { unstru_items(c, SM, gfull, gt, GT); });
  flat(ex, PH_UN_DOMROWS, [&](int, int gt, int GT) { unstru_dom_rows(c, gt, GT); });
  flat(ex, PH_UN_DOMCOLS, [&](int, int gt, int GT) { unstru_dom_cols(c, gt, GT); });
  if (p.out_up >= 0) flat(ex, PH_UN_WINDOWS, [&](int, int gt, int GT) { unstru_windows(c, dense + p.out_up, gt, GT); });
}

// outputs of a finished problem.  dense: base of the dense float output.  The barrier of the last phase also
// keeps a cluster's next problem out of the workspace slot until every CTA is done with this one.
template <class Exec, class MT>
RP_HD void emit_outputs(Exec& ex, Ctx& c, const Problem& p, float* dense, const MT& SM, const double* gfull) {
  if (p.kind == KIND_LINEAR) {
    if (p.out_bp >= 0) {
      flat(ex, PH_WRITE_BP, [&](int, int gt, int GT) { write_bp(c, dense + p.out_bp, gt, GT); });
      flat(ex, PH_WRITE_BP, [&](int, int gt, int GT) { write_bp2(c, dense + p.out_bp, gt, GT); });
    }
    if (p.max_w > 0 && !p.defer_up) emit_unpaired(ex, c, p, dense, SM, gfull);
  } else if (p.kind == KIND_COFOLD) {
    if (p.out_hp >= 0)
      flat(ex, PH_WRITE_HP, [&](int, int gt, int GT) { write_hp(c, dense + p.out_hp, p.n1, p.n2, p.th_hy, gt, GT); });
  }
}

// ---------------------------------------------------------------------------
// general kernel, one problem per CTA, sliced cells (the 64-register build).  logz: 3 doubles per pair or nullptr.
// ---------------------------------------------------------------------------
template <class Exec>
RP_HD void solve_mcc(Exec& ex, Ctx& c, const Problem& p, float* dense, double* logz, const Shared& sh) {
  const int T = sh.T;
  const int n = c.n;
  if (n + 2 <= RP_SMEM_SEQ) stage_sequence(ex, c, sh.S, [](int) {});
  ex.phase(PH_PROLOGUE, [&](int tid) {
    load_shared_model(*c.M, sh, tid);
    prologue_vectors(c, tid, T);
    prologue_lists(c, tid, T);
  });
  ex.phase(PH_PROLOGUE2, [&](int tid) { prologue2(c, tid, T); });

  // ---- inside: anti-diagonal wavefront, shortest spans first; split sums one band ahead
  // (The cells of a diagonal are dealt by plain loops rather than chunks(): in this spill-bound build the latter ran
  // 296 pairs of 300 x 250 nt 0.2 % slower, 101.55 against 101.32 ms, on a B200 at its 1000 W limit.)
  for (int d = TURN + 1; d <= n - 1; d++) {
    if (d == band_start_inside(d)) split_sums_inside<BAND>(ex, c, sh, d);
    const int cells = n - d;
    const int chunk = cells < T ? cells : T;
    for (int i0 = 1; i0 <= cells; i0 += chunk) {
      const int C = cells - i0 + 1 < chunk ? cells - i0 + 1 : chunk;
      ex.phase(PH_INSIDE_A, [&](int tid) { inside_A(c, sh, d, i0, C, tid); });
      ex.phase(PH_INSIDE_B, [&](int tid) { inside_B(c, sh, d, i0, C, tid); });
    }
  }
  inside_end(c);
  emit_logz(ex, c, p, logz);

  // ---- outside: longest spans first
  // (two strands: only the inter-strand cells of a diagonal, no nick sums -- cross_lo / cross_hi in mcc_core.h)
  for (int d = n - 1; d >= TURN + 1; d--) {
    if ((n - 1 - d) % BAND == 0) split_sums_outside<BAND>(ex, c, sh, d);   // a band of diagonals d .. d-BAND+1 starts here
    const int lo = cross_lo(c, d), hi = cross_hi(c, d), cells = hi - lo + 1;
    const int chunk = cells < T ? cells : T;
    for (int i0 = lo; i0 <= hi; i0 += chunk) {
      const int C = hi - i0 + 1 < chunk ? hi - i0 + 1 : chunk;
      ex.phase(PH_OUTSIDE_A, [&](int tid) { outside_A(c, sh, d, i0, C, tid); });
      ex.phase(PH_OUTSIDE_B, [&](int tid) { outside_B(c, sh, d, i0, C, tid); });
    }
  }
  emit_outputs(ex, c, p, dense, *c.M, &c.M->gfull[0][0]);
}

// ---------------------------------------------------------------------------
// general kernel, wide-band schedule (long problems), on one CTA or on the CTAs of a cluster (a single long pair
// instead of a shuffle batch): as solve_mcc, but the split sums are computed W = Exec::kWide diagonals at a time
// (far pass, "Wide bands" in mcc_core.h) and the finishing phase of a diagonal adds the few terms the far pass could
// not see.  `sh` must be carved with W.  A chunk's two phases (partial sums, then the reduction / the finish of its
// cells) stay inside one CTA; what crosses CTAs -- every table in the problem's HBM workspace -- is ordered by the
// problem-wide barrier of chunks() / flat() (for a cluster: release/acquire at cluster scope, which also drops the
// L1): after the far pass of a band and after the finishing phase of every diagonal.
// ---------------------------------------------------------------------------
template <class Exec>
RP_HD void solve_mcc_wide(Exec& ex, Ctx& c, const Problem& p, float* dense, double* logz, const Shared& sh) {
  constexpr int W = Exec::kWide;
  // Only a problem on one CTA stages the generic tile (and splits a diagonal's cells into the strand segments the tile
  // needs): a cluster deals each diagonal out in chunks of 1/G of it, and the tile's 38-column halo would dominate.
  constexpr bool tile = CtasOf<Exec>::value == 1;
  const int T = sh.T;
  const int n = c.n;
  if (n + 2 <= RP_SMEM_SEQ) stage_sequence(ex, c, sh.S, [](int) {});
  flat(ex, PH_PROLOGUE, [&](int tid, int gt, int GT) {
    load_shared_model(*c.M, sh, tid);
    prologue_vectors(c, gt, GT);
    prologue_lists(c, gt, GT);
  });
  flat(ex, PH_PROLOGUE2, [&](int, int gt, int GT) {
    prologue2(c, gt, GT);
    prologue_rowmajor(c, gt, GT);
  });

  for (int d = TURN + 1; d <= n - 1; d++) {
    if (d == wide_start_inside<W>(d)) split_sums_inside<W>(ex, c, sh, d);
    // Chunks of up to T cells that do not straddle a strand segment (both ends on strand 1 / joining the strands /
    // both on strand 2): the generic-class taps of a chunk are summed densely out of a shared-memory tile
    // (stage_generic_tile + generic_items), the ends and the table-driven shapes per cell (inside_A).
    const int cells = n - d;
    int sb[4] = {1, cells + 1, cells + 1, cells + 1};
    if (tile && c.cp > 0) {
      int b1 = c.cp - d, b2 = c.cp;
      if (b1 < 1) b1 = 1;
      if (b1 > cells + 1) b1 = cells + 1;
      if (b2 > cells + 1) b2 = cells + 1;
      if (b2 < b1) b2 = b1;
      sb[1] = b1; sb[2] = b2;
    }
    const bool staged = tile && W > BAND && gs_smax(n, d, 1) >= GS_ROW0;   // (the tile lives in the wide builds' partial-sum buffer)
    for (int sgm = 0; sgm < (tile ? 3 : 1); sgm++) {
      chunks(ex, sb[sgm], sb[sgm + 1], T, [&](int i0, int C) {
        const bool crossing = c.cp > 0 && sgm == 1;
        ex.phase(PH_INSIDE_A, [&](int tid) {
          if (staged) {
            stage_generic_tile<1>(c, sh, d, i0, C, crossing, tid);
            ends_items<1>(c, sh, d, i0, C, tid);
          } else {
            inside_A(c, sh, d, i0, C, tid);
          }
        });
        if (staged) ex.phase(PH_GENERIC_IN, [&](int tid) { generic_items<1>(c, sh, d, i0, C, tid); });
        ex.phase(PH_INSIDE_B, [&](int tid) { wide_inside_finish<W>(c, sh, d, i0, C, tid, staged); });
      });
    }
  }
  inside_end(c);
  emit_logz(ex, c, p, logz);

  for (int d = n - 1; d >= TURN + 1; d--) {
    if (d == wide_start_outside<W>(n, d)) split_sums_outside<W>(ex, c, sh, d);
    const bool staged = tile && W > BAND && gs_smax(n, d, -1) >= GS_ROW0;
    chunks(ex, cross_lo(c, d), cross_hi(c, d) + 1, T, [&](int i0, int C) {
      ex.phase(PH_OUTSIDE_A, [&](int tid) {
        if (staged) {
          stage_generic_tile<-1>(c, sh, d, i0, C, false, tid);   // (enclosing pairs of inter-strand cells join the strands anyway)
          ends_items<-1>(c, sh, d, i0, C, tid);
        } else {
          outside_A(c, sh, d, i0, C, tid);
        }
      });
      if (staged) ex.phase(PH_GENERIC_OUT, [&](int tid) { generic_items<-1>(c, sh, d, i0, C, tid); });
      ex.phase(PH_OUTSIDE_B, [&](int tid) { wide_outside_finish<W>(c, sh, d, i0, C, tid, staged); });
    });
  }
  emit_outputs(ex, c, p, dense, *c.M, &c.M->gfull[0][0]);
}

// the band ring is free once the wavefronts are done: it takes a copy of the gap-sum weights when they fit
template <class Exec>
RP_HD const double* stage_gap_weights(Exec& ex, const Ctx& c, const BandShared& bs) {
  const double* gfull = &c.M->gfull[0][0];
  if ((size_t)3 * BSLOTS * bs.LDB < (size_t)(MAXLOOP + 1) * GROW_LD) return gfull;
  const int T = ex.nthreads();
  ex.phase(PH_STAGE, [&](int tid) {
    for (int x = tid; x < (MAXLOOP + 1) * GROW_LD; x += T) bs.TI[x] = gfull[x];
  });
  return bs.TI;
}

// ---------------------------------------------------------------------------
// band kernel: one problem per CTA, interior-loop operands in a shared-memory
// ring of the last 32 diagonals (mcc_band.h); split sums, nick sums, unpaired
// windows and outputs as in solve_mcc.  `smem` is the CTA's dynamic shared
// memory (band_shared_bytes(n, T) bytes).
// ---------------------------------------------------------------------------
template <class Exec>
RP_HD void solve_band(Exec& ex, Ctx& c, const Problem& p, float* dense, double* logz, void* smem) {
  const int T = ex.nthreads();
  const int n = c.n;
  Shared sh;
  BandShared bs;
  carve_band(sh, bs, smem, n, T);
  const bool wide = c.kind == KIND_LINEAR && c.max_w > 0;  // the unpaired-window pass reads the class tables' full history
  stage_sequence(ex, c, sh.S, [&](int tid) {
    load_band_weights(*c.M, bs, tid, T);
    prologue_vectors(c, tid, T);
  });
  ex.phase(PH_PROLOGUE2, [&](int tid) {
    prologue2(c, tid, T);
    if (tid == T - 1 && TURN + 1 <= n - 1) band_make_desc(bs.desc[(TURN + 1) & (NDESC - 1)], n, c.cp, TURN + 1, T);
  });

  // Per-diagonal descriptors (strand segments, item schedule, thread roles: DiagDesc) are worked out by ONE
  // thread during the long phase of the step before their first use.
  // Schedule: the completion ("finish") of diagonal d runs one step late, in the same long phase
  // as the interior items of the next diagonal, so that its HBM/L2 round trips and the nick sums
  // hide behind the items' arithmetic.  Per diagonal: one long phase, then one quick phase that
  // collects the items' partial sums (freeing the partial buffer for the split-sum band phases,
  // which follow every BAND diagonals) and sets up the next diagonal's closing factors.
  // ---- inside: diagonals TURN+1 .. n-1
  ex.phase(PH_CFAC, [&](int tid) { band_collect<1>(c, bs, -1, TURN + 1 <= n - 1 ? TURN + 1 : -1, tid, T); });
  for (int d = TURN + 1; d <= n; d++) {
    const int dfin = d - 1 >= TURN + 1 ? d - 1 : -1;   // diagonal to complete in this step
    const int dnew = d <= n - 1 ? d : -1;              // diagonal whose items run in this step
    ex.phase(PH_INSIDE_A, [&](int tid) {
      if (dfin >= 0) band_inside_B(c, sh, bs, dfin, wide, tid);
      if (dnew >= 0) band_interior_A<1>(c, bs, dnew, tid, T);
      if (tid == T - 1 && d + 1 <= n - 1) band_make_desc(bs.desc[(d + 1) & (NDESC - 1)], n, c.cp, d + 1, T);
    });
    if (dnew < 0) break;
    ex.phase(PH_CFAC, [&](int tid) { band_collect<1>(c, bs, dnew, d + 1 <= n - 1 ? d + 1 : -1, tid, T); });
    // split sums of diagonals d .. d+BAND-1: every operand lies on a diagonal < d, complete now
    if (d == band_start_inside(d)) split_sums_inside<BAND>(ex, c, sh, d);
  }
  inside_end(c);
  emit_logz(ex, c, p, logz);

  // ---- outside: diagonals n-1 .. TURN+1; step d completes diagonal d+1 and runs the items of d.
  if (n - 1 >= TURN + 1)
    ex.phase(PH_CFAC, [&](int tid) { if (tid == 0) band_make_desc(bs.desc[(n - 1) & (NDESC - 1)], n, c.cp, n - 1, T, true); });
  ex.phase(PH_CFAC, [&](int tid) { band_collect<-1>(c, bs, -1, n - 1 >= TURN + 1 ? n - 1 : -1, tid, T); });
  for (int d = n - 1; d >= TURN; d--) {
    const int dfin = d + 1 <= n - 1 ? d + 1 : -1;
    const int dnew = d >= TURN + 1 ? d : -1;
    // split sums of diagonals d .. d-BAND+1: operands on diagonals >= d+2, complete after the previous step
    if (dnew >= 0 && (n - 1 - d) % BAND == 0) split_sums_outside<BAND>(ex, c, sh, d);
    ex.phase(PH_OUTSIDE_A, [&](int tid) {
      if (dfin >= 0) band_outside_B(c, sh, bs, dfin, wide, tid);
      if (dnew >= 0) band_interior_A<-1>(c, bs, dnew, tid, T);
      if (tid == T - 1 && d - 1 >= TURN + 1) band_make_desc(bs.desc[(d - 1) & (NDESC - 1)], n, c.cp, d - 1, T, true);
    });
    if (dnew < 0) break;
    ex.phase(PH_CFAC, [&](int tid) {
      band_collect<-1>(c, bs, dnew, d - 1 >= TURN + 1 ? d - 1 : -1, tid, T);
    });
  }
  const double* gfull = wide && !p.defer_up ? stage_gap_weights(ex, c, bs) : &c.M->gfull[0][0];
  emit_outputs(ex, c, p, dense, *bs.sm, gfull);
}

// the unpaired-window pass of a problem the band kernel finished earlier, run as a job of its own inside that kernel
template <class Exec>
RP_HD void solve_band_unpaired(Exec& ex, Ctx& c, const Problem& p, float* dense, void* smem) {
  const int T = ex.nthreads(), n = c.n;
  Shared sh;
  BandShared bs;
  carve_band(sh, bs, smem, n, T);
  stage_sequence(ex, c, sh.S, [&](int tid) { load_band_weights(*c.M, bs, tid, T); });
  inside_end(c);
  emit_unpaired(ex, c, p, dense, *bs.sm, stage_gap_weights(ex, c, bs));
}

}  // namespace rp
#endif