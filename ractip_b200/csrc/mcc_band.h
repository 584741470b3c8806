// mcc_band.h -- the shared-memory "band" formulation of the McCaskill wavefront
// (same recurrences and reference call sites as mcc_core.h; this file only
// changes WHERE the operands of the interior-loop sums live and HOW they are
// summed).
//
// The interior-loop sum of cell (i,j) on anti-diagonal d reaches back at most
// MAXLOOP+2 = 32 diagonals:  inner pair (i+1+u1, j-1-u2) lies on diagonal
// d-2-s, s = u1+u2 <= 30, at position i+1+u1.  Seen along one earlier
// diagonal ("row" s) the sum is a 1-D correlation of that row with the weights
// g(u1, s-u1): neighbouring cells use overlapping windows of the same row.
// So:
//   * the three factorised class tables (generic / 1xn / bulge, see
//     dev_model.h) of the last 32 diagonals live in a shared-memory ring
//     (3 x 32 rows), written by the thread that finishes a cell;
//   * a thread owns a GROUP of 8 neighbouring cells and walks a row with a
//     sliding 8-wide register window: one shared load + one weight per 8 DFMA;
//   * rows are stored "mod-8 transposed" (position p at (p&7)*LD8 + (p>>3)), so
//     the 16 lanes of a half-warp, which own 16 consecutive groups, read 16
//     consecutive doubles although every lane strides by 8 (conflict-free for the
//     window walk; measured over the whole kernel, ncu: 0.23 G conflicts on 1.81 G
//     shared-load wavefronts, 13 %, from the two half-warps of a warp working on
//     different rows and from the per-cell finish / small-loop reads);
//   * the sum is DENSE (cells that cannot pair are computed and multiplied by
//     a zero closing factor): no compaction lists, no divergence;
//   * the 31 rows are dealt out as 16 balanced row pairs (q, 30-q) = 16 slices;
//     a work item is (slice, block of 16 groups) on one half-warp;
//   * two-strand problems: cells of a diagonal are grouped per strand segment
//     (both ends on strand 1 / crossing the nick / both on strand 2), so the
//     strand guard of a whole group is ONE interval of valid row positions,
//     applied when a row element is loaded.
// The outside pass is the mirror image (enclosing pairs lie on later diagonals
// d+2+s at positions k-1-u1) and runs through the same code with the same
// ring, now holding out*factor rows.
//
// Everything else of a diagonal step (split sums over finished diagonals, nick
// sums, unpaired windows, outputs) is shared with mcc_core.h.
#ifndef RP_MCC_BAND_H
#define RP_MCC_BAND_H

#include "mcc_core.h"

namespace rp {

constexpr int BR = 8;            // cells per group
constexpr int BSLOTS = 32;       // ring slots = MAXLOOP + 2
constexpr int NSLICE = 16;       // row pairs (q, 30-q)

// Shared-memory copy of the small Boltzmann tables (same member names as DevModel, so that
// ext_stem / ml_stem / special_loop work on either).  With ~225 KB of shared memory carved out the
// L1 has no room left and every DevModel access would be an L2 round trip on the critical path.
struct SmallModel {
  double scale1, mlb1, expMLclosing, expMLintern, expTermAU, inv_expTermAU;
  double scale_small[10];
  double mmI[8][5][5], mmH[8][5][5], mmM[8][5][5], mmExt[8][5][5], mm1n[8][5][5];
  double dangle5[8][5], dangle3[8][5];
  const double* spw;                      // finished weights of the table-driven small loops: stay in HBM/L2
  int special_hp, pad;
};
constexpr int SM_DOUBLES = (int)((sizeof(SmallModel) + 7) / 8);

struct DiagDesc;
struct BandShared {
  int LDB, LD8;   // ring row stride in doubles (multiple of 8) and sub-row length LDB/8
  int NGP;        // stride of the group-transposed arrays (>= max number of groups of a diagonal)
  double *TI, *T1, *TA;    // [BSLOTS][LDB] generic / 1xn / bulge class rows
  double* ipart;           // [NSLICE+1][BR*NGP] partial interior sums, element (r, g) at r*NGP+g; aliases Shared::part
  double *cI, *c1, *cA;    // [BR*NGP] closing-pair factors of the diagonal whose interior sums are being built
  double* G;               // generic weights, packed: G[s*(s+1)/2 + t] = g(t, s-t), 0 where (t, s-t) is not generic
  double *gA, *g1;         // [32] bulge weight g(0,s), 1xn weight g(1,s-1)
  double* sIv;             // [n+2] finished interior sums of the diagonal that is being completed (by cell)
  SmallModel* sm;
  DiagDesc* desc;          // [NDESC] per-diagonal descriptors
};
constexpr int GPACK = (MAXLOOP + 1) * (MAXLOOP + 2) / 2;   // 496
constexpr int DESC_DOUBLES = 4 * 6;                        // NDESC descriptors of 12 ints (DiagDesc, below)

RP_HD int band_ldb(int n) { return ((n + 1 + 7) / 8) * 8; }
RP_HD int band_ngp(int n) { return (n + 7) / 8 + 3; }
// partial sums of the split-sum band phases / of the interior items (they alias).  The CUDA build runs the
// shuffle form of the band phases (mcc_band_shfl.cuh), where a warp owns 32-(BAND-1) rows: 2*BAND partials for
// 28 rows per warp.  The direct form takes 2*BAND partials per thread.  Host code that sizes a launch of the CUDA
// build (plan.cpp) asks for the shuffle form: shfl = true; solve_band carves the form its executor runs (kShfl).
#ifdef __CUDACC__
constexpr bool BAND_SHFL = true;
#else
constexpr bool BAND_SHFL = false;
#endif
RP_HD size_t band_part_doubles(int n, int T, bool shfl = BAND_SHFL) {
  const size_t a = shfl ? (size_t)2 * BAND * (32 - (BAND - 1)) * (T / 32) : (size_t)2 * BAND * T;
  const size_t b = (size_t)(NSLICE + 1) * BR * band_ngp(n);
  return a > b ? a : b;
}
RP_HD size_t band_shared_doubles(int n, int T, bool shfl = BAND_SHFL) {
  return band_part_doubles(n, T, shfl) + 128 /*red*/ + (size_t)3 * BSLOTS * band_ldb(n) + (size_t)3 * BR * band_ngp(n) +
         GPACK + 64 + (size_t)(n + 2) + SM_DOUBLES + DESC_DOUBLES + (size_t)(n + 2 + 7) / 8 + 2;
}
RP_HD size_t band_shared_bytes(int n, int T, bool shfl = BAND_SHFL) { return band_shared_doubles(n, T, shfl) * sizeof(double); }

RP_HD void carve_band(Shared& sh, BandShared& bs, void* base, int n, int T, bool shfl = BAND_SHFL) {
  sh.T = T;
  double* p = static_cast<double*>(base);
  sh.part = p; bs.ipart = p; p += band_part_doubles(n, T, shfl);
  sh.red = p; p += 128;
  bs.LDB = band_ldb(n); bs.LD8 = bs.LDB / 8; bs.NGP = band_ngp(n);
  bs.TI = p; p += (size_t)BSLOTS * bs.LDB;
  bs.T1 = p; p += (size_t)BSLOTS * bs.LDB;
  bs.TA = p; p += (size_t)BSLOTS * bs.LDB;
  bs.cI = p; p += (size_t)BR * bs.NGP;
  bs.c1 = p; p += (size_t)BR * bs.NGP;
  bs.cA = p; p += (size_t)BR * bs.NGP;
  bs.G = p; p += GPACK;
  bs.gA = p; p += 32;
  bs.g1 = p; p += 32;
  bs.sIv = p; p += n + 2;
  bs.sm = reinterpret_cast<SmallModel*>(p); p += SM_DOUBLES;
  bs.desc = reinterpret_cast<DiagDesc*>(p); p += DESC_DOUBLES;
  sh.S = reinterpret_cast<uint8_t*>(p);
  sh.grow = nullptr; sh.ghead_b = nullptr; sh.ghead_1 = nullptr;  // the factorised-row tables of the general kernel are not used
}

RP_HD void load_band_weights(const DevModel& M, const BandShared& bs, int tid, int T) {
  for (int x = tid; x < GPACK; x += T) bs.G[x] = M.gpack[x];   // packed on the host (build_dev_model)
  for (int s = tid; s < 32; s += T) { bs.gA[s] = M.gA[s]; bs.g1[s] = M.g1[s]; }
  SmallModel& S = *bs.sm;
  if (tid == 0) {
    S.scale1 = M.scale1; S.mlb1 = M.mlb1; S.expMLclosing = M.expMLclosing; S.expMLintern = M.expMLintern;
    S.expTermAU = M.expTermAU; S.inv_expTermAU = 1.0 / M.expTermAU;
    for (int k = 0; k < 10; k++) S.scale_small[k] = M.scale_small[k];
    S.spw = M.spw;
    S.special_hp = M.special_hp; S.pad = 0;
  }
  for (int x = tid; x < 200; x += T) {
    (&S.mmI[0][0][0])[x] = (&M.mmI[0][0][0])[x];
    (&S.mmH[0][0][0])[x] = (&M.mmH[0][0][0])[x];
    (&S.mmM[0][0][0])[x] = (&M.mmM[0][0][0])[x];
    (&S.mmExt[0][0][0])[x] = (&M.mmExt[0][0][0])[x];
    (&S.mm1n[0][0][0])[x] = (&M.mm1n[0][0][0])[x];
    if (x < 40) {
      (&S.dangle5[0][0])[x] = (&M.dangle5[0][0])[x];
      (&S.dangle3[0][0])[x] = (&M.dangle3[0][0])[x];
    }
  }
}

// position p of a ring row
RP_HD int bidx(const BandShared& bs, int p) { return (p & 7) * bs.LD8 + (p >> 3); }
RP_HD double* brow(double* band, const BandShared& bs, int d) { return band + (size_t)(d & (BSLOTS - 1)) * bs.LDB; }

// Strand segments of the cells (i, i+d), i = 1..n-d, of one diagonal:
//   segment 0: i <  b1   (both ends on strand 1)
//   segment 1: b1 <= i < b2   (the pair crosses the nick)
//   segment 2: i >= b2   (both ends on strand 2)
// Groups of BR cells never straddle a segment boundary.  Single strand: one segment.
struct Segs {
  int b[4];   // first cell of each segment, b[3] = n-d+1
  int G[4];   // first group of each segment, G[3] = number of groups
};
// `cross_only`: only the cells that join the two strands (segment 1) exist -- the outside pass of a two-strand
// problem needs no others (see cross_lo / cross_hi in mcc_core.h): segments 0 and 2 come out empty.
RP_HD Segs make_segs(int n, int cp, int d, bool cross_only = false) {
  Segs s;
  const int C = n - d;
  s.b[0] = 1; s.b[3] = C + 1;
  if (cp <= 0) { s.b[1] = C + 1; s.b[2] = C + 1; }
  else {
    int b1 = cp - d, b2 = cp;
    if (b1 < 1) b1 = 1;
    if (b1 > C + 1) b1 = C + 1;
    if (b2 > C + 1) b2 = C + 1;
    if (b2 < b1) b2 = b1;
    s.b[1] = b1; s.b[2] = b2;
  }
  if (cross_only && cp > 0) { s.b[0] = s.b[1]; s.b[3] = s.b[2]; }
  s.G[0] = 0;
  for (int k = 0; k < 3; k++) s.G[k + 1] = s.G[k] + (s.b[k + 1] - s.b[k] + BR - 1) / BR;
  return s;
}
// element index (r*NGP + g) of cell i in the group-transposed arrays
RP_HD int seg_slot(const Segs& s, const BandShared& bs, int i) {
  const int k = (i >= s.b[1]) + (i >= s.b[2]);
  const int o = i - s.b[k];
  return (o & (BR - 1)) * bs.NGP + s.G[k] + (o >> 3);
}

// Everything the phases of one diagonal need to know about its layout, worked out ONCE (by one thread, a
// phase ahead) and kept in shared memory: the strand segments, the item schedule and the thread roles.
// (Every thread used to redo this arithmetic in every phase: ~6 % of all executed instructions.)
struct DiagDesc {
  Segs sg;
  int gsh, NB, nitems, t0;
};
constexpr int NDESC = 4;   // ring of descriptors (diagonal d at d & 3): a descriptor lives for three phases
static_assert(sizeof(DiagDesc) * NDESC <= DESC_DOUBLES * sizeof(double), "descriptor ring");
RP_HD void band_make_desc(DiagDesc& D, int n, int cp, int d, int T, bool cross_only = false) {
  D.sg = make_segs(n, cp, d, cross_only);
  const int NG = D.sg.G[3], cells = D.sg.b[3] - D.sg.b[0];
  // an item block is GB lanes = GB consecutive groups: a half-warp, or a quarter-warp when the whole
  // diagonal fits in 8 groups (4 slices per warp: half the instructions on the short diagonals)
  D.gsh = NG <= 8 ? 3 : 4;
  const int GB = 1 << D.gsh;
  D.NB = (NG + GB - 1) >> D.gsh;
  D.nitems = NSLICE * D.NB;
  // Thread roles of the long phase: the first `cells` threads complete the previous diagonal, the
  // last `cells` do the small loops; when they fit, the items go to the threads in between, so that
  // no thread has two jobs.
  const int Cw = (cells + 1 + 31) & ~31;   // (the previous diagonal has one more cell)
  D.t0 = (D.nitems * GB + 2 * Cw <= T) ? Cw : 0;
}

// Global load that is issued WHERE IT IS WRITTEN: at the register cap the compiler otherwise sinks
// every load of the finish code next to its first use, which turns one L2 round trip into ten.
#ifdef __CUDA_ARCH__
__device__ __forceinline__ double ldg_now(const double* p) {
  double v;
  asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
#else
inline double ldg_now(const double* p) { return *p; }
#endif
// the same for an optional operand: loads a harmless address when !ok and yields `dflt` (no branch)
RP_HD double ldg_if(bool ok, const double* p, const double* safe, double dflt) {
  const double v = ldg_now(ok ? p : safe);
  return ok ? v : dflt;
}

// Ring element load "valid ? row[ix] : 0" of the item loops.  On the device: one predicated
// ld.shared (no branch, no address clamp); `x <= span` (unsigned) is the validity test.
#ifdef __CUDA_ARCH__
struct RingPtr { unsigned a; };   // shared-window byte address
__device__ __forceinline__ RingPtr ring_ptr(const double* p) { RingPtr r; r.a = (unsigned)__cvta_generic_to_shared(p); return r; }
__device__ __forceinline__ double ring_ld(RingPtr base, int ix, unsigned x, unsigned span) {
  double v;
  asm volatile("{\n\t.reg .pred p;\n\tsetp.le.u32 p, %2, %3;\n\tmov.f64 %0, 0d0000000000000000;\n\t@p ld.shared.f64 %0, [%1];\n\t}"
               : "=d"(v) : "r"(base.a + (unsigned)(ix * 8)), "r"(x), "r"(span));
  return v;
}
__device__ __forceinline__ void ring_adv(RingPtr& p, int elems) { p.a += (unsigned)(elems * 8); }
__device__ __forceinline__ void keep_in_reg(int& v) { asm volatile("" : "+r"(v)); }
#else
struct RingPtr { const double* a; };
inline RingPtr ring_ptr(const double* p) { RingPtr r; r.a = p; return r; }
inline double ring_ld(RingPtr base, int ix, unsigned x, unsigned span) { return x <= span ? base.a[ix] : 0.; }
inline void ring_adv(RingPtr& p, int elems) { p.a += elems; }
inline void keep_in_reg(int&) {}
#endif

// ---------------------------------------------------------------------------
// one work item of the interior sums: slice q (rows q and 30-q) of group g.
// SIGN=+1 inside (rows d-2-s, window starts at i0+1), SIGN=-1 outside (rows
// d+2+s, window starts at k0-1-s).  Result: the group's BR partial sums, already
// multiplied by the cells' closing-pair factors.
// ---------------------------------------------------------------------------
template <int SIGN>
RP_HD void interior_item(const BandShared& bs, int n, int cp, int d, const Segs& sg, int q, int g, double* tot) {
#pragma unroll
  for (int r = 0; r < BR; r++) tot[r] = 0.;
  const int k = (g >= sg.G[1]) + (g >= sg.G[2]);
  const int i0 = sg.b[k] + BR * (g - sg.G[k]);
  const int smax = SIGN > 0 ? (d - 6 < MAXLOOP ? d - 6 : MAXLOOP) : (n - 3 - d < MAXLOOP ? n - 3 - d : MAXLOOP);
  const double* fI = bs.cI + g;   // closing factors of cell r at [r*NGP]: loaded where they are used
  const double* f1 = bs.c1 + g;
  const double* fA = bs.cA + g;
  const int NGP = bs.NGP, LD8 = bs.LD8;
#pragma unroll 1
  for (int h = 0; h < 2; h++) {
    const int s = h == 0 ? q : MAXLOOP - q;
    if (h == 1 && s == q) break;
    if (s > smax || s < 2) continue;
    const int dr = d - SIGN * (2 + s);           // the row's diagonal
    const int P0 = SIGN > 0 ? i0 + 1 : i0 - 1 - s;  // row position of (cell r = 0, tap t = 0)
    // valid positions of the row for this group: inside the row, and on the right side of the nick
    int plo = 1, phi = n - dr;
    if (cp > 0) {
      if (SIGN > 0) {
        if (k == 1) { if (cp - dr > plo) plo = cp - dr; if (cp - 1 < phi) phi = cp - 1; }
      } else {
        if (k == 0) { if (cp - 1 - dr < phi) phi = cp - 1 - dr; }
        else if (k == 2) { if (cp > plo) plo = cp; }
      }
    }
    if (phi < plo) continue;
    // Window element c stands for row position P0 + c; it is valid iff clo <= c <= clo + span, and
    // lives at sub-row (b+c)&7, index q0 + ((b+c)>>3) of the (mod-8 transposed) row.
    const int clo = plo - P0;
    const unsigned span = (unsigned)(phi - plo);
    const int b = P0 & 7;
    const size_t ro = (size_t)(dr & (BSLOTS - 1)) * bs.LDB;
    const RingPtr rI = ring_ptr(bs.TI + ro + (P0 >> 3));   // only dereferenced at valid elements
    const RingPtr r1 = ring_ptr(bs.T1 + ro + (P0 >> 3));
    const RingPtr rA = ring_ptr(bs.TA + ro + (P0 >> 3));
#define RP_IX(e) (((e) & 7) * LD8 + ((e) >> 3))
    // bulge ends (0,s),(s,0): elements r and r+s of the bulge-class row; 1xn ends (1,s-1),(s-1,1): elements r+1
    // and r+s-1 of the 1xn-class row.  ONE rolled loop over the two tables (code size: the per-diagonal loops
    // have to fit the 32 KB instruction cache; the arithmetic is the same either way).
#pragma unroll 1
    for (int tb = 0; tb < (s >= 4 ? 2 : 1); tb++) {
      const RingPtr rp = tb ? r1 : rA;
      const double* f = tb ? f1 : fA;
      const double w = tb ? bs.g1[s] : bs.gA[s];
      const int eL = tb, eR = s - tb;          // first element of the left / right run
      const unsigned xl = (unsigned)(eL - clo), xr = (unsigned)(eR - clo);
#pragma unroll
      for (int r = 0; r < BR; r++) {
        const double x0 = ring_ld(rp, RP_IX(b + eL + r), xl + r, span), x1 = ring_ld(rp, RP_IX(b + eR + r), xr + r, span);
        tot[r] += f[r * NGP] * (w * (x0 + x1));
      }
    }
    if (s >= 6) {  // generic taps t = 2 .. s-2: tap-major walk with a sliding register window
      double acc[BR], win[BR];
#pragma unroll
      for (int r = 0; r < BR; r++) acc[r] = 0.;
#pragma unroll
      for (int r = 0; r < BR - 1; r++) win[r] = ring_ld(rI, RP_IX(b + 2 + r), (unsigned)(2 + r - clo), span);
      win[BR - 1] = 0.;
      // step t loads element t+7; within an unrolled block of 8 steps the 8 element offsets are
      // loop-invariant (the row pointer advances by one per block)
      int off[BR];
#pragma unroll
      for (int u = 0; u < BR; u++) { off[u] = RP_IX(b + 9 + u); keep_in_reg(off[u]); }
      const double* gw = bs.G + s * (s + 1) / 2 + 2;   // weight of tap 2+x at gw[x]
      RingPtr pI = rI;
      unsigned cm = (unsigned)(9 - clo);               // (element of step u) - clo = cm + u
      const int nst = s - 3;                           // number of steps
      int x = 0;
#pragma unroll 1
      for (; x + BR <= nst; x += BR) {
#pragma unroll
        for (int u = 0; u < BR; u++) {
          win[(u + BR - 1) & (BR - 1)] = ring_ld(pI, off[u], cm + u, span);
          const double gv = gw[u];
#pragma unroll
          for (int r = 0; r < BR; r++) acc[r] += gv * win[(u + r) & (BR - 1)];
        }
        ring_adv(pI, 1); cm += BR; gw += BR;
      }
#pragma unroll
      for (int u = 0; u < BR - 1; u++) {
        if (x + u < nst) {
          win[(u + BR - 1) & (BR - 1)] = ring_ld(pI, off[u], cm + u, span);
          const double gv = gw[u];
#pragma unroll
          for (int r = 0; r < BR; r++) acc[r] += gv * win[(u + r) & (BR - 1)];
        }
      }
#pragma unroll
      for (int r = 0; r < BR; r++) tot[r] += fI[r * NGP] * acc[r];
    }
#undef RP_IX
  }
}

// (u1,u2) of the nine table-driven shapes as compile-time functions (special_uv's order)
RP_HD constexpr int sp_u1(int s) { return s == 0 ? 0 : s == 1 ? 1 : s == 2 ? 0 : s == 3 ? 1 : s == 4 ? 1 : s == 5 ? 2 : s == 6 ? 2 : s == 7 ? 2 : 3; }
RP_HD constexpr int sp_u2(int s) { return s == 0 ? 0 : s == 1 ? 0 : s == 2 ? 1 : s == 3 ? 1 : s == 4 ? 2 : s == 5 ? 1 : s == 6 ? 2 : s == 7 ? 3 : 2; }

// value of qb (inside) / out (outside) recovered from the bulge-class row, which holds
// x * expTermAU^[type>2]
RP_HD double band_plain(const BandShared& bs, int d, int p, int type) {
  const double v = bs.TA[(size_t)(d & (BSLOTS - 1)) * bs.LDB + bidx(bs, p)];
  return type > 2 ? v * bs.sm->inv_expTermAU : v;
}

// The table-driven small loops of one cell.  Branch-free: all nine shapes are evaluated with
// clamped indices and masked, so that their (L2-resident) table look-ups overlap instead of
// queueing one after the other.
template <class C>
RP_HD double inside_specials_band(const C& c, const BandShared& bs, int d, int i) {
  const SmallModel& M = *bs.sm;
  const int j = i + d;
  const int type = pair_type(base(c, i), base(c, j));
  const int ddmax = d - (TURN + 1) < MAXLOOP + 2 ? d - (TURN + 1) : MAXLOOP + 2;
  if (!type || ddmax < 2) return 0.;
  const int maxpo = (c.cp > 0 && i < c.cp) ? c.cp - 1 - i : 1000;
  const int maxu2 = (c.cp > 0 && j >= c.cp) ? j - 1 - c.cp : 1000;
  const int si1 = base(c, i + 1), sj1 = base(c, j - 1);
  double v[RP_N_SPECIAL], w[RP_N_SPECIAL];
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) {
    const int u1 = sp_u1(s), u2 = sp_u2(s), dd = u1 + u2 + 2;
    const bool ok = dd <= ddmax && u1 + 1 <= maxpo && u2 <= maxu2;
    const int k = ok ? i + 1 + u1 : i + 1, l = ok ? j - 1 - u2 : j - 1, dr = ok ? d - dd : d - 2;
    const int t2 = pair_type(base(c, k), base(c, l));
    v[s] = (ok && t2) ? band_plain(bs, dr, k, t2) : 0.;
    w[s] = special_loop(M, s, type, rtype(t2), si1, sj1, base(c, k - 1), base(c, l + 1));
  }
  double acc = 0.;
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) acc += v[s] * w[s];
  return acc;
}

template <class C>
RP_HD double outside_specials_band(const C& c, const BandShared& bs, int d, int k) {
  const SmallModel& M = *bs.sm;
  const int n = c.n, l = k + d;
  const int type = pair_type(base(c, k), base(c, l));
  const int ddmax = n - 1 - d < MAXLOOP + 2 ? n - 1 - d : MAXLOOP + 2;
  if (!type || ddmax < 2) return 0.;
  int maxpo = k - 1, maxu2 = n - l - 1;
  if (c.cp > 0) {
    if (k >= c.cp && k - c.cp < maxpo) maxpo = k - c.cp;
    if (l < c.cp && c.cp - 2 - l < maxu2) maxu2 = c.cp - 2 - l;
  }
  if (maxpo < 1 || maxu2 < 0) return 0.;
  const int t2 = rtype(type), sp1 = base(c, k - 1), sq1 = base(c, l + 1);
  double v[RP_N_SPECIAL], w[RP_N_SPECIAL];
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) {
    const int u1 = sp_u1(s), u2 = sp_u2(s), dd = u1 + u2 + 2;
    const bool ok = dd <= ddmax && u1 + 1 <= maxpo && u2 <= maxu2;
    const int i = ok ? k - 1 - u1 : k - 1, j = ok ? l + 1 + u2 : l + 1, dr = ok ? d + dd : d + 2;
    const int t1 = pair_type(base(c, i), base(c, j));
    v[s] = (ok && t1) ? band_plain(bs, dr, i, t1) : 0.;
    w[s] = special_loop(M, s, t1, t2, base(c, i + 1), base(c, j - 1), sp1, sq1);
  }
  double acc = 0.;
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) acc += v[s] * w[s];
  return acc;
}

// phase A of a diagonal: all interior items.  Half-warp hw serves item hw, hw+nhw, ...;
// item -> (slice q = item / NB, block b = item % NB), lane hl of the half-warp owns group 16*b+hl.
// The table-driven small loops (9 per cell) are done one cell per thread by the LAST threads of
// the CTA (idle or lightly loaded in the item schedule) and form slice NSLICE.
template <int SIGN, class C>
RP_HD void band_interior_A(const C& c, const BandShared& bs, int d, int tid, int T) {
  const int n = c.n;
  // layout, item schedule and thread roles of this diagonal: worked out once, a phase ahead (band_make_desc)
  const DiagDesc& D = bs.desc[d & (NDESC - 1)];
  const Segs& sg = D.sg;
  const int NG = sg.G[3], gsh = D.gsh, GB = 1 << gsh, NB = D.NB, nitems = D.nitems, t0 = D.t0;
  const int smax = SIGN > 0 ? d - 6 : n - 3 - d;
  // small loops first: their table look-ups are in flight while the row items run
  for (int x = T - 1 - tid; x < sg.b[3] - sg.b[0]; x += T) {   // (the active cells: all, or the inter-strand ones)
    const int i = sg.b[0] + x;
    double v;
    if (RP_DBG(c) & 8) v = 0.;
    else if (SIGN > 0) v = inside_specials_band(c, bs, d, i);
    else v = outside_specials_band(c, bs, d, i);
    bs.ipart[(size_t)NSLICE * BR * bs.NGP + seg_slot(sg, bs, i)] = v;
  }
  if (smax >= 2 && tid >= t0) {
    const int unit = (tid - t0) >> gsh, hl = (tid - t0) & (GB - 1), nunits = (T - t0) >> gsh;
    for (int item = unit; item < nitems; item += nunits) {
      const int q = NB == 1 ? item : (NB == 2 ? item >> 1 : item / NB), b = item - q * NB;
      const int g = GB * b + hl;
      if (g >= NG) continue;
      double tot[BR];
      if (RP_DBG(c) & 1) {
#pragma unroll
        for (int r = 0; r < BR; r++) tot[r] = 0.;
      } else {
        interior_item<SIGN>(bs, n, c.cp, d, sg, q, g, tot);
      }
      double* out = bs.ipart + (size_t)q * BR * bs.NGP + g;
#pragma unroll
      for (int r = 0; r < BR; r++) out[r * bs.NGP] = tot[r];
    }
  }
}

// sum of the partials of cell i (fixed order: deterministic)
template <int SIGN, class C>
RP_HD double band_interior_sum(const C& c, const BandShared& bs, int d, const Segs& sg, int i) {
  const int slot = seg_slot(sg, bs, i);
  const int smax = SIGN > 0 ? d - 6 : c.n - 3 - d;
  double s = bs.ipart[(size_t)NSLICE * BR * bs.NGP + slot];
  if (smax >= 2) {
    double s0 = 0., s1 = 0.;
#pragma unroll
    for (int q = 0; q < NSLICE; q += 2) {
      s0 += bs.ipart[(size_t)q * BR * bs.NGP + slot];
      s1 += bs.ipart[(size_t)(q + 1) * BR * bs.NGP + slot];
    }
    s += s0 + s1;
  }
  return s;
}

// quick phase between two diagonals: collect the partial interior sums of the diagonal whose
// items have just run (dsum, skipped if < 0) into sIv, and set up the closing factors of the next
// one (dnext, skipped if < 0).  After it the partial-sum buffer is free again.
template <int SIGN, class C>
RP_HD void band_collect(const C& c, const BandShared& bs, int dsum, int dnext, int tid, int T);

// closing-pair factors of the cells of diagonal d (whose interior sums are built next)
template <class C>
RP_HD void band_cfac_inside(const C& c, const BandShared& bs, int d, int tid, int T) {
  const SmallModel& M = *bs.sm;
  const int cells = c.n - d;
  if (cells <= 0) return;
  const Segs& sg = bs.desc[d & (NDESC - 1)].sg;
  for (int x = tid; x < BR * sg.G[3]; x += T) {  // every slot of every group, cells past a segment end get 0
    const int g = x / BR, r = x % BR;
    const int k = (g >= sg.G[1]) + (g >= sg.G[2]);
    const int i = sg.b[k] + BR * (g - sg.G[k]) + r;
    double fI = 0., f1 = 0., fA = 0.;
    if (i < sg.b[k + 1]) {
      const int j = i + d;
      const int type = pair_type(base(c, i), base(c, j));
      if (type) {
        const int si1 = base(c, i + 1), sj1 = base(c, j - 1);
        fI = M.mmI[type][si1][sj1];
        f1 = M.mm1n[type][si1][sj1];
        fA = type > 2 ? M.expTermAU : 1.0;
      }
    }
    bs.cI[r * bs.NGP + g] = fI;
    bs.c1[r * bs.NGP + g] = f1;
    bs.cA[r * bs.NGP + g] = fA;
  }
}
template <class C>
RP_HD void band_cfac_outside(const C& c, const BandShared& bs, int d, int tid, int T) {
  const SmallModel& M = *bs.sm;
  const int n = c.n, cells = n - d;
  if (cells <= 0 || d <= TURN) return;
  const Segs& sg = bs.desc[d & (NDESC - 1)].sg;
  for (int x = tid; x < BR * sg.G[3]; x += T) {
    const int g = x / BR, r = x % BR;
    const int kk = (g >= sg.G[1]) + (g >= sg.G[2]);
    const int k = sg.b[kk] + BR * (g - sg.G[kk]) + r;
    double fI = 0., f1 = 0., fA = 0.;
    if (k < sg.b[kk + 1]) {
      const int l = k + d;
      const int type = pair_type(base(c, k), base(c, l));
      if (type && k > 1 && l < n) {   // (a pair with qb = 0 gets out = 0 when it is finished, whatever its sums)
        const int t2 = rtype(type), sp1 = base(c, k - 1), sq1 = base(c, l + 1);
        fI = M.mmI[t2][sq1][sp1];
        f1 = M.mm1n[t2][sq1][sp1];
        fA = type > 2 ? M.expTermAU : 1.0;
      }
    }
    bs.cI[r * bs.NGP + g] = fI;
    bs.c1[r * bs.NGP + g] = f1;
    bs.cA[r * bs.NGP + g] = fA;
  }
}

// ---------------------------------------------------------------------------
// phase B: finish the cells of diagonal d (one thread per cell), write the ring
// rows, and prepare the closing factors of the next diagonal.  All HBM/L2
// operands of a cell are loaded up front with clamped addresses (one round
// trip), then combined.
// `wide`: also keep the class tables in HBM (the unpaired-window pass of a
// single-strand problem reads their full history).
// ---------------------------------------------------------------------------
// branch-free stem factors (all three candidates are loaded with clamped indices, then selected):
// same values as ext_stem / ml_stem of mcc_core.h
template <class MT>
RP_HD double ext_stem_bf(const MT& M, int type, int s5, int s3) {
  const int a = s5 >= 0 ? s5 : 0, b = s3 >= 0 ? s3 : 0;
  const double both = M.mmExt[type][a][b], d5 = M.dangle5[type][a], d3 = M.dangle3[type][b];
  const double e = (s5 >= 0 && s3 >= 0) ? both : (s5 >= 0 ? d5 : (s3 >= 0 ? d3 : 1.0));
  return type > 2 ? e * M.expTermAU : e;
}
template <class MT>
RP_HD double ml_stem_bf(const MT& M, int type, int s5, int s3) {
  const int a = s5 >= 0 ? s5 : 0, b = s3 >= 0 ? s3 : 0;
  const double both = M.mmM[type][a][b], d5 = M.dangle5[type][a], d3 = M.dangle3[type][b];
  double e = (s5 >= 0 && s3 >= 0) ? both : (s5 >= 0 ? d5 : (s3 >= 0 ? d3 : 1.0));
  if (type > 2) e *= M.expTermAU;
  return e * M.expMLintern;
}

// Finish of a cell, written for latency: (1) every HBM/L2 operand is requested first; (2) while the
// requests are in flight, everything that depends on the sequence alone (pair type, stem and mismatch
// factors: shared-memory look-ups) is evaluated WITHOUT branches; (3) only then the loaded values are
// combined, in half a dozen dependent fp operations, and stored.  (A consumer of a loaded value
// stalls the warp's whole in-order stream, and a branch keeps the compiler from filling the wait.)
template <class C>
RP_HD void band_inside_B(C& c, const Shared& sh, const BandShared& bs, int d, bool wide, int tid) {
  const int T = sh.T, n = c.n, cells = n - d;
  const SmallModel& M = *bs.sm;
  if (RP_DBG(c) & 16) return;
  const int u = d - 1;  // hairpin size
  const int e = d - band_start_inside(d);
  const int vprev = (d & 1) ? V_U0 : V_U1, vcur = (d & 1) ? V_U1 : V_U0;
  for (int x = tid; x < cells; x += T) {
    const int i = 1 + x, j = i + d;
    // ---- (1) loads
#ifdef __CUDA_ARCH__
    long long tp0 = 0;
    if (RP_PROF(c) && tid == 0) tp0 = clock64();
#endif
    const double* safe = c.ptr(T_Q, 0, 1);
    const double sM = ldg_now(c.ptr(T_QM2, d, i));
    double sQ = ldg_now(c.ptr(T_QS, d, i));
    const double qm2c = ldg_now(c.ptr(T_QM2, d - 2, i + 1));
    const double qm1l = ldg_now(c.ptr(T_QM1, d - 1, i)), qm1r = ldg_now(c.ptr(T_QM1, d - 1, i + 1));
    const double qql = ldg_now(c.ptr(T_QQ, d - 1, i));
    const double uprev = ldg_now(&VEC(c, vprev, i + 1));
    const double hpw = ldg_now(&VEC(c, V_HPW, u)), scd = ldg_now(&VEC(c, V_SCALE, d + 1));
    double nq[BAND - 1];
#pragma unroll
    for (int a = 0; a < BAND - 1; a++) {
      const bool ok = a < e && a <= d - TURN - 2;
      nq[a] = ldg_if(ok, c.ptr(T_QQ, ok ? d - 1 - a : 0, ok ? i + 1 + a : 1), safe, 0.);
    }
    const bool sp_case = M.special_hp && (u == 3 || u == 4 || u == 6);
    const double spv = ldg_if(sp_case, &VEC(c, u == 3 ? V_SP3 : (u == 4 ? V_SP4 : V_SP6), i), safe, -1.);
    const bool cross = c.cp > 0 && i < c.cp && j >= c.cp;   // !ss(i,j)
    const bool has1 = cross && i + 1 <= c.cp - 1, has2 = cross && c.cp <= j - 1;
    const double nk1 = ldg_if(has1, c.ptr(T_Q, has1 ? c.cp - 2 - i : 0, has1 ? i + 1 : 1), safe, 1.0);
    const double nk2 = ldg_if(has2, c.ptr(T_Q, has2 ? j - 1 - c.cp : 0, has2 ? c.cp : 1), safe, 1.0);
    // ---- (2) sequence-only factors
    const int type = pair_type(base(c, i), base(c, j));
    const bool tz = type != 0;
    const int rt = rtype(type);
    const int si1 = base(c, i + 1), sj1 = base(c, j - 1);
    const int sim = i > 1 ? base(c, i - 1) : -1, sjp = j < n ? base(c, j + 1) : -1;
    const bool ssl = ss(c, i, i + 1), ssr = ss(c, j - 1, j), ssi = ss(c, i - 1, i), ssj = ss(c, j, j + 1);
    const double au = type > 2 ? M.expTermAU : 1.0;
    const double scale2 = M.scale_small[2];
    const double hfac = (sp_case && u == 3) ? au : M.mmH[type][si1][sj1];                      // hairpin: hpw * hfac
    const double k1 = (tz && ssl && ssr) ? M.expMLclosing * ml_stem_bf(M, rt, sj1, si1) * scale2 : 0.;   // closes a multiloop
    const double k2 = (tz && cross) ? scale2 * ext_stem_bf(M, rt, ssr ? sj1 : -1, ssl ? si1 : -1) : 0.;  // closes the nicked loop
    const double k3 = (tz && ssi && ssj) ? ml_stem_bf(M, type, sim, sjp) : 0.;                 // stem in a multiloop
    const double k4 = tz ? ext_stem_bf(M, type, ssi ? sim : -1, ssj ? sjp : -1) : 0.;          // stem in the exterior loop
    const double gI = tz ? M.mmI[rt][sjp < 0 ? 0 : sjp][sim < 0 ? 0 : sim] : 0.;               // seen as an inner pair
    const double g1 = tz ? M.mm1n[rt][sjp < 0 ? 0 : sjp][sim < 0 ? 0 : sim] : 0.;
    const double gA = tz ? au : 0.;
    const double m1 = ssr ? M.mlb1 : 0., mU = ssl ? M.mlb1 : 0.;
    const double sI = tz ? bs.sIv[i] : 0.;
    const size_t ro = (size_t)(d & (BSLOTS - 1)) * bs.LDB + bidx(bs, i);
#ifdef __CUDA_ARCH__
    long long tp1 = 0;
    if (RP_PROF(c) && tid == 0) tp1 = clock64();
#endif
    if (RP_DBG(c) & 128) { bs.sIv[i] = sM + sQ + qm2c + qm1l + qm1r + qql + uprev + hpw + scd + nq[0] + nq[1] + nq[2] + nq[3] + spv + nk1 + nk2; continue; }
    // ---- (3) combine
#pragma unroll
    for (int a = 0; a < BAND - 1; a++) sQ += M.scale_small[a + 1] * nq[a];   // q(i,i+a) = scale^(a+1), a <= TURN
    const double h = spv >= 0. ? spv : hpw * hfac;
    double qb = (tz && !cross) ? h : 0.;
    qb += sI;
    qb += qm2c * k1;
    qb += k2 * nk1 * nk2;
    if (!(RP_DBG(c) & 256)) RP_ST_STREAM(TB(c, T_QB, d, i), qb);
    const double fI = qb * gI, f1 = qb * g1, fA = qb * gA;
    bs.TI[ro] = fI; bs.T1[ro] = f1; bs.TA[ro] = fA;
    if (wide) { RP_ST_STREAM(TB(c, T_QBI, d, i), fI); RP_ST_STREAM(TB(c, T_QB1N, d, i), f1); RP_ST_STREAM(TB(c, T_QBAU, d, i), fA); }
    const double qm1 = qm1l * m1 + qb * k3;
    const double U = mU * (qm1r + uprev);
    const double qq = qql * M.scale1 + qb * k4;
    if (!(RP_DBG(c) & 256)) {
      TB(c, T_QM1, d, i) = qm1;
      VEC(c, vcur, i) = U;
      TB(c, T_QM, d, i) = qm1 + sM + U;
      TB(c, T_QQ, d, i) = qq;
      TB(c, T_Q, d, i) = scd + qq + sQ;
    } else bs.sIv[i] = qq + qm1 + U;
#ifdef __CUDA_ARCH__
    if (RP_PROF(c) && tid == 0) {
      const long long tp2 = clock64();
      atomicAdd(reinterpret_cast<unsigned long long*>(RP_PROF(c) + 24), (unsigned long long)(tp1 - tp0));
      atomicAdd(reinterpret_cast<unsigned long long*>(RP_PROF(c) + 25), (unsigned long long)(tp2 - tp1));
      atomicAdd(reinterpret_cast<unsigned long long*>(RP_PROF(c) + 32 + 24), 1ull);
      atomicAdd(reinterpret_cast<unsigned long long*>(RP_PROF(c) + 32 + 25), 1ull);
    }
#endif
  }
}

template <class C>
RP_HD void band_outside_B(C& c, const Shared& sh, const BandShared& bs, int d, bool wide, int tid) {
  if (RP_DBG(c) & 16) return;
  const int T = sh.T, n = c.n;
  const SmallModel& M = *bs.sm;
  const int k_lo = cross_lo(c, d), k_hi = cross_hi(c, d);   // two strands: only the inter-strand cells
  for (int x = tid; x <= k_hi - k_lo; x += T) {
    const int k = k_lo + x, l = k + d;
    const bool mlr = l < n && ss(c, l, l + 1);
    const bool mll = k > 1 && ss(c, k - 1, k);
    // ---- (1) loads
    const double* safe = c.ptr(T_Q, 0, 1);
    const double sP = ldg_now(c.ptr(T_PRB, d, k)), sL = ldg_now(c.ptr(T_MLB, d, k));
    const double qbv = ldg_now(c.ptr(T_QB, d, k));
    const double plp = ldg_if(mlr, c.ptr(T_PL, d + 1, k), safe, 0.), mcp = ldg_if(mlr, c.ptr(T_MC, d + 1, k), safe, 0.);
    const double pmp = ldg_if(mll, c.ptr(T_PMLB, d + 1, mll ? k - 1 : 1), safe, 0.);
    const double prp = ldg_if(mll, c.ptr(T_PR, d + 1, mll ? k - 1 : 1), safe, 0.);
    const double q5 = ldg_if(k > 1, c.ptr(T_Q, k > 1 ? k - 2 : 0, 1), safe, 1.0);
    const double q3 = ldg_if(l < n, c.ptr(T_Q, l < n ? n - l - 1 : 0, l < n ? l + 1 : 1), safe, 1.0);
    // (two strands: only inter-strand cells are finished here, and those never sit in the nicked loop)
    // ---- (2) sequence-only factors
    const int type = pair_type(base(c, k), base(c, l));
    const bool tz = type != 0;
    const int rt = rtype(type);
    const int skm = base(c, k - 1), slp = base(c, l + 1), si1 = base(c, k + 1), sj1 = base(c, l - 1);
    const double au = type > 2 ? M.expTermAU : 1.0;
    const double scale2 = M.scale_small[2];
    const double kx = ext_stem_bf(M, type, mll ? skm : -1, mlr ? slp : -1);                     // stem in the exterior loop
    const double km = (mlr && mll) ? ml_stem_bf(M, type, skm, slp) * scale2 : 0.;              // stem in a multiloop
    const double gI = tz ? M.mmI[type][si1][sj1] : 0., g1 = tz ? M.mm1n[type][si1][sj1] : 0., gA = tz ? au : 0.;
    const double gM = (tz && ss(c, k, k + 1) && ss(c, l - 1, l)) ? M.expMLclosing * ml_stem_bf(M, rt, sj1, si1) : 0.;
    const double sIraw = bs.sIv[k];
    const size_t ro = (size_t)(d & (BSLOTS - 1)) * bs.LDB + bidx(bs, k);
    if (RP_DBG(c) & 128) { bs.sIv[k] = sP + sL + qbv + plp + mcp + pmp + prp + q5 + q3; continue; }
    // ---- (3) combine
    const bool live = tz && qbv != 0.;
    const double PL = mlr ? plp * M.mlb1 + mcp : 0.;
    const double PR = mlr ? sP : 0.;
    const double PMLB = mll ? pmp * M.mlb1 + prp : 0.;
    double out = q5 * q3 * c.invZ * kx;
    out += sIraw;
    out += (PMLB + sL) * km;
    out = live ? out : 0.;
    TB(c, T_PL, d, k) = PL;
    TB(c, T_PR, d, k) = PR;
    TB(c, T_PRML, d, k) = PR + PL;
    TB(c, T_PMLB, d, k) = PMLB;
    RP_ST_STREAM(TB(c, T_OUT, d, k), out);
    const double fI = out * gI, f1 = out * g1, fA = out * gA;
    bs.TI[ro] = fI; bs.T1[ro] = f1; bs.TA[ro] = fA;
    if (wide) { RP_ST_STREAM(TB(c, T_OUTI, d, k), fI); RP_ST_STREAM(TB(c, T_OUT1N, d, k), f1); RP_ST_STREAM(TB(c, T_OUTAU, d, k), fA); }
    TB(c, T_MC, d, k) = out * gM;
  }
}

template <int SIGN, class C>
RP_HD void band_collect(const C& c, const BandShared& bs, int dsum, int dnext, int tid, int T) {
  if (RP_DBG(c) & 32) return;
  const int reps = (RP_DBG(c) & 512) ? 2 : 1;   // tuning aid: the same code twice tells cold-code cost from work
#pragma unroll 1
  for (int rep = 0; rep < reps; rep++) {
    if (dsum >= 0) {
      const Segs& sg = bs.desc[dsum & (NDESC - 1)].sg;
      const int first = sg.b[0], cells = sg.b[3] - sg.b[0];
      for (int x = tid; x < cells; x += T) bs.sIv[first + x] = band_interior_sum<SIGN>(c, bs, dsum, sg, first + x);
    }
    if (dnext >= 0) {
      if (SIGN > 0) band_cfac_inside(c, bs, dnext, tid, T);
      else band_cfac_outside(c, bs, dnext, tid, T);
    }
  }
}

}  // namespace rp
#endif
