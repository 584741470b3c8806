// mfe_core.h -- minimum free energy (Zuker) of one problem, written once as per-thread phase functions like mcc_core.h:
// the CUDA kernel (kernels.cu, mfe_kernel) runs them with tid = threadIdx.x and __syncthreads() between phases, the host
// emulation (tests/emul) thread after thread or warp by warp in lockstep.
//
// The minimum is over exactly the structures the general McCaskill kernel sums over (canonical pairs with j-i > TURN,
// interior loops up to MAXLOOP, the problem's constraint keys, dangles = 2, the co-fold's nick guards) of the integer
// energy rp_energy_of_structure gives (eval.cpp; DuplexInit once when a pair joins the strands), plus the stacking
// pseudo-energies es (Es(i)+Es(i+1)+Es(j-1)+Es(j) per stack within one strand) and the unpaired pseudo-energies eu (per
// base left unpaired; a base paired with the partner counts as unpaired).  Unpaired terms enter as pair terms, as in
// the partition function (pair_sc, mcc_core.h): sum_{x unpaired} Eu(x) = sum_x Eu(x) - sum_{(i,j) intramolecular}
// (Eu(i) + Eu(j)), so an intramolecular pair gets -Eu(i)-Eu(j) and the host adds the constant.
//
// Tables (int32, diagonal-major like mcc_core.h: cell (i,j) at d*ld + i, d = j-i):
//   C(i,j)    (i,j) pairs: the energy of everything it encloses, its own loop included
//   FM1(i,j)  multiloop part i..j with exactly one stem, which starts at i; l+1..j unpaired
//   FM2(i,j)  multiloop part i..j with two stems or more, split at k != cp: FML(i,k-1) + FM1(k,j)
//   FML(i,j)  multiloop part i..j with one stem or more
// and two exterior vectors per strand [s0, s1] (strand 1 = 1..cp-1, strand 2 = cp..n; a linear problem is one strand):
//   PRE(y) = the exterior minimum of s0..y,  SUF(x) = the exterior minimum of x..s1.
// A pair that joins the strands closes a nick loop, scored as an exterior loop: ext_stem of the reversed pair plus
// SUF(i+1) over i+1..cp-1 and PRE(j-1) over cp..j-1.  The co-fold's answer is min(PRE(cp-1) + SUF(cp), min over joining
// exterior stems (p,l) of PRE(p-1) + C(p,l) + ext_stem + SUF(l+1) + DuplexInit): at most one exterior stem joins.
//
// Fill: one anti-diagonal per step.  A warp takes a cell: its lanes share the interior-loop candidates (<= 496) and the
// multiloop splits, and a shuffle reduction takes the minimum.  Integer min is order-independent, so the result does not
// depend on the schedule.  PRE and SUF of diagonal d-1 are computed while diagonal d fills (a cell of diagonal d reads
// them up to diagonal d-2 only).
//
// Traceback (one warp): a stack of pending segments, popped depth first; a decision enumerates its candidates in the
// fixed order given at mfe_cand and takes the FIRST whose energy equals the segment's value.
#ifndef RP_MFE_CORE_H
#define RP_MFE_CORE_H

#include "mcc_core.h"

namespace rp {

static_assert(HP_LONG_MAX >= RP_MAX_N, "DevModel::i_hairpin_long must cover every hairpin of a problem");

// Internal sentinel.  Every value of a feasible structure stays below 2^26 in magnitude (the host bounds the
// pseudo-energies, plan.h MFE_MAX_PSEUDO), so a sum of up to three table entries and loop terms neither overflows
// int32 nor falls below MFE_BIG when one operand is MFE_INF; entries at or above MFE_BIG are stored as MFE_INF.
constexpr int MFE_INF = 1 << 29;
constexpr int MFE_BIG = 1 << 28;
RP_HD int mfe_clamp(int v) { return v >= MFE_BIG ? MFE_INF : v; }

enum { MT_C = 0, MT_FML, MT_FM1, MT_FM2, MT_COUNT };
// slot of one problem, in int32: the four tables, PRE, SUF, the traceback's segment stack (n + 8 uint64), 8 scalars
RP_HD size_t mfe_slot_ints(int n) { return MT_COUNT * table_elems(n) + 2 * vector_elems(n) + 2 * vector_elems(n) + 16; }

// One problem of rp_run_mfe (plan_mfe, plan.h): its per-base data at seq_off - 1 + [1..n] of the batch's arrays, laid
// out like the encoded sequences; flags CON_KEYS / CON_STACK / CON_UNPAIRED say which it carries.
struct MfeJob {
  int seq_off, n, cp;
  int flags;
  long long out;    // int16 offset of its pair table in the structure buffer
  int energy_at;    // index of its energy (3 pair + problem)
  int eu_const;     // sum of the unpaired pseudo-energies over its bases, added to the minimum
};

struct MfeCtx {
  const DevModel* M;
  const uint8_t* S;      // S[1..n], as Ctx::S
  int n, cp, ld;
  int* ws;
  unsigned te, ve;
  const uint16_t* key;   // key[1..n] or null (pair allowed iff key[i] == key[j])
  const int* es;         // stacking pseudo-energies es[1..n] (0.01 kcal/mol) or null
  const int* eu;         // unpaired pseudo-energies eu[1..n] or null
  RP_HD int sraw(int i) const { return S[i]; }
  RP_HD int& tb(int t, int d, int i) const { return ws[(unsigned)t * te + (unsigned)d * (unsigned)ld + (unsigned)i]; }
  RP_HD int& pre(int y) const { return ws[(unsigned)MT_COUNT * te + (unsigned)y]; }
  RP_HD int& suf(int x) const { return ws[(unsigned)MT_COUNT * te + ve + (unsigned)x]; }
  RP_HD uint64_t* stack() const { return reinterpret_cast<uint64_t*>(ws + (size_t)MT_COUNT * te + 2 * (size_t)ve); }
  RP_HD int& scalar(int k) const { return ws[(size_t)MT_COUNT * te + 4 * (size_t)ve + k]; }
};

RP_HD void bind_mfe(MfeCtx& c, const DevModel* M, const uint8_t* S, int n, int cp, int* ws) {
  c.M = M; c.S = S; c.n = n; c.cp = cp; c.ld = n + 1; c.ws = ws;
  c.te = (unsigned)table_elems(n); c.ve = (unsigned)vector_elems(n);
  c.key = nullptr; c.es = nullptr; c.eu = nullptr;
}

// ---------------------------------------------------------------------------------------------- energies (eval.cpp)
RP_HD int mfe_type(const MfeCtx& c, int i, int j) {
  const int t = pair_type(c.sraw(i) & 7, c.sraw(j) & 7);
  return (c.key && c.key[i] != c.key[j]) ? 0 : t;
}
// PRE over s0..y and SUF over x..s1, 0 for an empty region
RP_HD int pre0(const MfeCtx& c, int s0, int y) { return y < s0 ? 0 : c.pre(y); }
RP_HD int suf0(const MfeCtx& c, int x, int s1) { return x > s1 ? 0 : c.suf(x); }

RP_HD int e_ext_stem(const DevModel& M, int type, int s5, int s3) {
  int e = 0;
  if (s5 >= 0 && s3 >= 0) e = M.i_mmExt[type][s5][s3];
  else if (s5 >= 0) e = M.i_dangle5[type][s5];
  else if (s3 >= 0) e = M.i_dangle3[type][s3];
  if (type > 2) e += M.i_TermAU;
  return e;
}
RP_HD int e_ml_stem(const DevModel& M, int type, int s5, int s3) {
  int e = 0;
  if (s5 >= 0 && s3 >= 0) e = M.i_mmM[type][s5][s3];
  else if (s5 >= 0) e = M.i_dangle5[type][s5];
  else if (s3 >= 0) e = M.i_dangle3[type][s3];
  if (type > 2) e += M.i_TermAU;
  return e + M.i_MLintern;
}
// exterior stem (p,l) of a PRE / SUF region or the co-fold's exterior loop: dangles on the stem's own strand
RP_HD int e_ext_of(const MfeCtx& c, int type, int p, int l) {
  return e_ext_stem(*c.M, type, (p > 1 && ss(c, p - 1, p)) ? base(c, p - 1) : -1, (l < c.n && ss(c, l, l + 1)) ? base(c, l + 1) : -1);
}
// multiloop stem (k,l)
RP_HD int e_ml_of(const MfeCtx& c, int type, int k, int l) {
  return e_ml_stem(*c.M, type, k > 1 ? base(c, k - 1) : -1, l < c.n ? base(c, l + 1) : -1);
}
RP_HD int e_hairpin(const MfeCtx& c, int i, int j, int type) {
  const DevModel& M = *c.M;
  const int u = j - i - 1;
  const int e = u <= 30 ? M.i_hairpin[u] : M.i_hairpin_long[u];
  if (M.special_hp && (u == 3 || u == 4 || u == 6)) {
    int code = 0;   // window i..j as base-8 digits, 7 for a letter that matches no list entry (prologue2, mcc_core.h)
    for (int p = i; p <= j; p++) code = code * 8 + ((c.sraw(p) & 8) ? 7 : (c.sraw(p) & 7));
    if (u == 4) {
      for (int k = 0; k < M.n_tetra; k++)
        if (M.tetra_code[k] == code) return M.i_tetra[k];
    } else if (u == 6) {
      for (int k = 0; k < M.n_hex; k++)
        if (M.hex_code[k] == code) return M.i_hex[k];
    } else {
      for (int k = 0; k < M.n_tri; k++)
        if (M.tri_code[k] == code) return M.i_tri[k];
    }
  }
  if (u == 3) return e + (type > 2 ? M.i_TermAU : 0);
  return e + M.i_mmH[type][base(c, i + 1)][base(c, j - 1)];
}
// interior loop closed by `type`, inner pair reversed type2, u1 / u2 unpaired (eval.cpp int_loop; u1 + u2 <= MAXLOOP)
RP_HD int e_interior(const DevModel& M, int u1, int u2, int type, int type2, int si1, int sj1, int sp1, int sq1) {
  const int nl = u1 > u2 ? u1 : u2, ns = u1 > u2 ? u2 : u1;
  if (nl == 0) return M.i_stack[type][type2];
  if (ns == 0) {
    int e = M.i_bulge[nl];
    if (nl == 1) return e + M.i_stack[type][type2];
    if (type > 2) e += M.i_TermAU;
    if (type2 > 2) e += M.i_TermAU;
    return e;
  }
  const int ninio = (nl - ns) * M.i_ninio < M.i_MAX_NINIO ? (nl - ns) * M.i_ninio : M.i_MAX_NINIO;
  if (ns == 1) {
    if (nl == 1) return M.i_int11[type][type2][si1][sj1];
    if (nl == 2) return u1 == 1 ? M.i_int21[type][type2][si1][sq1][sj1] : M.i_int21[type2][type][sq1][si1][sp1];
    return M.i_internal[nl + 1] + ninio + M.i_mm1n[type][si1][sj1] + M.i_mm1n[type2][sq1][sp1];
  }
  if (ns == 2) {
    if (nl == 2) return M.i_int22[type][type2][si1][sp1][sq1][sj1];
    if (nl == 3) return M.i_internal[5] + M.i_ninio + M.i_mm23[type][si1][sj1] + M.i_mm23[type2][sq1][sp1];
  }
  return M.i_internal[nl + ns] + ninio + M.i_mmI[type][si1][sj1] + M.i_mmI[type2][sq1][sp1];
}
RP_HD int pair_term(const MfeCtx& c, int i, int j) { return (c.eu && ss(c, i, j)) ? -(c.eu[i] + c.eu[j]) : 0; }

// (u1, u2) of interior candidate x, 0 <= x < 496: rows u1 = 0..30 of lengths 31 - u1, u2 ascending
constexpr int MFE_INT_CANDS = (MAXLOOP + 1) * (MAXLOOP + 2) / 2;
// row r starts at r (2 MAXLOOP + 3 - r) / 2: the root of that quadratic, then exact integer corrections
RP_HD int int_row_start(int r) { return r * (2 * MAXLOOP + 3 - r) / 2; }
RP_HD void int_uv(int x, int& u1, int& u2) {
  const float b = 2.f * MAXLOOP + 3.f;
  int r = (int)((b - sqrtf(b * b - 8.f * (float)x)) * 0.5f);
  r = r < 0 ? 0 : (r > MAXLOOP ? MAXLOOP : r);
  while (r > 0 && int_row_start(r) > x) r--;
  while (r < MAXLOOP && int_row_start(r + 1) <= x) r++;
  u1 = r; u2 = x - int_row_start(r);
}

// Candidate energies.  Orders (the traceback takes the first that reaches the segment's value):
//   C(i,j)   x = 0 hairpin; 1 + t interior loop number t (int_uv); 497 multiloop FM2(i+1,j-1); 498 nick loop
//            (all with the pair term of (i,j))
//   FM1(i,j) x = 0 stem (i,j); 1 j unpaired, FM1(i,j-1)
//   FML(i,j) x = 0 FM1(i,j); 1 i unpaired, FML(i+1,j); 2 FM2(i,j)
//   FM2(i,j) x = k - (i+TURN+2), k ascending, k != cp: FML(i,k-1) + FM1(k,j)
//   PRE s0..y  x = 0 y unpaired; 1 + (k - s0) stem (k,y), k ascending
//   SUF x..s1  x' = 0 x unpaired; 1 + (l - x - TURN - 1) stem (x,l), l ascending
//   TOP (co-fold)  x = 0 no pair joins: PRE(cp-1) + SUF(cp); 1 + (p-1) n2 + (l-cp) the joining exterior stem (p,l)
enum { SG_C = 0, SG_FM1, SG_FML, SG_FM2, SG_PRE, SG_SUF, SG_TOP };
constexpr int MFE_C_CANDS = 1 + MFE_INT_CANDS + 2;

RP_HD int mfe_c_cand(const MfeCtx& c, int i, int j, int type, int x) {
  const DevModel& M = *c.M;
  const int d = j - i;
  if (x == 0) return ss(c, i, j) ? e_hairpin(c, i, j, type) : MFE_INF;
  if (x == MFE_C_CANDS - 2) {
    if (!(ss(c, i, i + 1) && ss(c, j - 1, j)) || d - 2 < 2 * TURN + 2) return MFE_INF;
    return c.tb(MT_FM2, d - 2, i + 1) + M.i_MLclosing + e_ml_stem(M, rtype(type), base(c, j - 1), base(c, i + 1));
  }
  if (x == MFE_C_CANDS - 1) {
    if (ss(c, i, j)) return MFE_INF;
    return e_ext_stem(M, rtype(type), ss(c, j - 1, j) ? base(c, j - 1) : -1, ss(c, i, i + 1) ? base(c, i + 1) : -1) +
           suf0(c, i + 1, c.cp - 1) + pre0(c, c.cp, j - 1);
  }
  int u1, u2;
  int_uv(x - 1, u1, u2);
  const int ddmax = d - (TURN + 1) < MAXLOOP + 2 ? d - (TURN + 1) : MAXLOOP + 2;
  if (u1 + u2 + 2 > ddmax) return MFE_INF;
  // strand guards (inside_interior): the inner pair's 5' end stays on i's strand, its 3' end on j's
  if (c.cp > 0 && i < c.cp && i + 1 + u1 > c.cp - 1) return MFE_INF;
  if (c.cp > 0 && j >= c.cp && j - 1 - u2 < c.cp) return MFE_INF;
  const int k = i + 1 + u1, l = j - 1 - u2;
  const int t2 = mfe_type(c, k, l);
  if (!t2) return MFE_INF;
  int e = c.tb(MT_C, l - k, k) + e_interior(M, u1, u2, type, rtype(t2), base(c, i + 1), base(c, j - 1), base(c, k - 1), base(c, l + 1));
  if (c.es && u1 + u2 == 0 && ss(c, i, j)) e += c.es[i] + c.es[i + 1] + c.es[j - 1] + c.es[j];
  return e;
}
RP_HD int mfe_fm2_cand(const MfeCtx& c, int i, int j, int x) {
  const int k = i + TURN + 2 + x;
  if (c.cp > 0 && k == c.cp) return MFE_INF;
  return c.tb(MT_FML, k - 1 - i, i) + c.tb(MT_FM1, j - k, k);
}
RP_HD int mfe_pre_cand(const MfeCtx& c, int s0, int y, int x) {
  if (x == 0) return pre0(c, s0, y - 1);
  const int k = s0 + x - 1;
  const int t = mfe_type(c, k, y);
  if (!t) return MFE_INF;
  return pre0(c, s0, k - 1) + c.tb(MT_C, y - k, k) + e_ext_of(c, t, k, y);
}
RP_HD int mfe_suf_cand(const MfeCtx& c, int x0, int s1, int x) {
  if (x == 0) return suf0(c, x0 + 1, s1);
  const int l = x0 + TURN + x;
  const int t = mfe_type(c, x0, l);
  if (!t) return MFE_INF;
  return c.tb(MT_C, l - x0, x0) + e_ext_of(c, t, x0, l) + suf0(c, l + 1, s1);
}
RP_HD int mfe_top_cand(const MfeCtx& c, int x) {
  if (x == 0) return c.pre(c.cp - 1) + c.suf(c.cp);
  const int n2 = c.n - c.cp + 1, p = 1 + (x - 1) / n2, l = c.cp + (x - 1) % n2;
  if (l - p <= TURN) return MFE_INF;
  const int t = mfe_type(c, p, l);
  if (!t) return MFE_INF;
  return pre0(c, 1, p - 1) + c.tb(MT_C, l - p, p) + e_ext_of(c, t, p, l) + suf0(c, l + 1, c.n) + c.M->i_DuplexInit;
}

// ------------------------------------------------------------------------------------------- warp reductions
// SHFL: the 32 lanes of a warp share the candidates and meet in shuffles (every lane gets the result); else lane 0 walks
// them alone (the host reference form).
// (the device pass of nvcc and the host emulation, which defines RP_HOST_SHFL and host stand-ins for the intrinsics)
template <bool SHFL>
RP_HD int warp_min(int v) {
#if defined(__CUDA_ARCH__) || defined(RP_HOST_SHFL)
  if constexpr (SHFL) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_down_sync(0xffffffffu, v, o);
      v = y < v ? y : v;
    }
    return __shfl_sync(0xffffffffu, v, 0);
  }
#endif
  return v;
}
// min over candidates x = 0 .. cnt-1 of f(x)
template <bool SHFL, class F>
RP_HD int cand_min(int cnt, int lane, F f) {
  const int step = SHFL ? 32 : 1;
  int best = MFE_INF;
  for (int x = lane; x < cnt; x += step) {
    const int v = f(x);
    best = v < best ? v : best;
  }
  return warp_min<SHFL>(best);
}
// the first x whose f(x) == target, -1 if none: lane L looks at x0 + L of each group of 32
template <bool SHFL, class F>
RP_HD int cand_first(int cnt, int lane, int target, F f) {
  const int step = SHFL ? 32 : 1;
  for (int x0 = 0; x0 < cnt; x0 += step) {
    const int x = x0 + lane;
    int hit = (x < cnt && f(x) == target) ? x : MFE_INF;
    hit = warp_min<SHFL>(hit);
    if (hit < MFE_INF) return hit;
  }
  return -1;
}

// ---------------------------------------------------------------------------------------------------- fill
// diagonals 0..TURN and the exterior vectors: no structure
RP_HD void mfe_prologue(MfeCtx& c, int tid, int T) {
  const int n = c.n, dmax = TURN < n - 1 ? TURN : n - 1;
  for (int x = tid; x < (dmax + 1) * c.ld; x += T)
    for (int t = 0; t < MT_COUNT; t++) c.ws[(unsigned)t * c.te + (unsigned)x] = MFE_INF;
  for (int x = tid; x < (int)c.ve; x += T) { c.pre(x) = 0; c.suf(x) = 0; }
}

// cell (i, i+d), d > TURN, by one warp
template <bool SHFL>
RP_HD void mfe_cell(MfeCtx& c, int d, int i, int lane) {
  const DevModel& M = *c.M;
  const int j = i + d;
  const int type = mfe_type(c, i, j);
  int cv = MFE_INF;
  if (type) {
    cv = cand_min<SHFL>(MFE_C_CANDS, lane, [&](int x) { return mfe_c_cand(c, i, j, type, x); });
    cv = mfe_clamp(cv + pair_term(c, i, j));
  }
  const int cnt2 = d - 2 * TURN - 2;   // k = i+TURN+2 .. j-TURN-1
  const int fm2 = cnt2 > 0 ? mfe_clamp(cand_min<SHFL>(cnt2, lane, [&](int x) { return mfe_fm2_cand(c, i, j, x); })) : MFE_INF;
  int fm1 = ss(c, j - 1, j) ? c.tb(MT_FM1, d - 1, i) + M.i_MLbase : MFE_INF;
  if (type && ss(c, i - 1, i) && ss(c, j, j + 1)) {
    const int s = cv + e_ml_of(c, type, i, j);
    fm1 = s < fm1 ? s : fm1;
  }
  fm1 = mfe_clamp(fm1);
  int fml = fm1 < fm2 ? fm1 : fm2;
  if (ss(c, i, i + 1)) {
    const int s = c.tb(MT_FML, d - 1, i + 1) + M.i_MLbase;
    fml = s < fml ? s : fml;
  }
  if (lane == 0) {
    c.tb(MT_C, d, i) = cv;
    c.tb(MT_FM1, d, i) = fm1;
    c.tb(MT_FM2, d, i) = fm2;
    c.tb(MT_FML, d, i) = mfe_clamp(fml);
  }
}

// exterior vector entry v of diagonal dd by one warp: v = 0 PRE, 1 SUF of strand 1, 2 / 3 of strand 2 (co-fold)
template <bool SHFL>
RP_HD void mfe_vector(MfeCtx& c, int dd, int v, int lane) {
  const int s0 = v < 2 ? 1 : c.cp, s1 = v < 2 ? (c.cp > 0 ? c.cp - 1 : c.n) : c.n;
  if (v & 1) {
    const int x = s1 - dd;
    if (x < s0) return;
    const int cnt = s1 - x - TURN + 1 > 1 ? s1 - x - TURN + 1 : 1;
    const int r = cand_min<SHFL>(cnt, lane, [&](int y) { return mfe_suf_cand(c, x, s1, y); });
    if (lane == 0) c.suf(x) = mfe_clamp(r);
  } else {
    const int y = s0 + dd;
    if (y > s1) return;
    const int cnt = y - TURN - s0 + 1 > 1 ? y - TURN - s0 + 1 : 1;
    const int r = cand_min<SHFL>(cnt, lane, [&](int x) { return mfe_pre_cand(c, s0, y, x); });
    if (lane == 0) c.pre(y) = mfe_clamp(r);
  }
}

// Phase of diagonal d (TURN < d <= n): items 0 .. nv-1 the exterior vectors of diagonal d-1, then the cells of diagonal
// d, dealt out to the warps round robin.
template <bool SHFL>
RP_HD void mfe_diagonal(MfeCtx& c, int d, int tid, int T) {
  const int lane = SHFL ? (tid & 31) : 0, w = tid >> 5, nw = T >> 5;
  if (!SHFL && (tid & 31)) return;
  const int nv = c.cp > 0 ? 4 : 1, cells = d < c.n ? c.n - d : 0;
  for (int it = w; it < nv + cells; it += nw) {
    if (it < nv) mfe_vector<SHFL>(c, d - 1, it, lane);
    else mfe_cell<SHFL>(c, d, 1 + it - nv, lane);
  }
}

// The value of the whole problem (without the unpaired constant) into scalar(0); co-fold: every thread's part of the
// joined minimum in red[tid], then thread 0 takes the minimum.
RP_HD void mfe_top_part(MfeCtx& c, int* red, int tid, int T) {
  if (c.cp <= 0) { red[tid] = MFE_INF; return; }
  const int cnt = 1 + (c.cp - 1) * (c.n - c.cp + 1);
  int best = MFE_INF;
  for (int x = tid; x < cnt; x += T) {
    const int v = mfe_top_cand(c, x);
    best = v < best ? v : best;
  }
  red[tid] = best;
}
RP_HD void mfe_top_finish(MfeCtx& c, const int* red, int tid, int T) {
  if (tid) return;
  int best = MFE_INF;
  if (c.cp <= 0) best = c.pre(c.n);
  else
    for (int t = 0; t < T; t++) best = red[t] < best ? red[t] : best;
  c.scalar(0) = mfe_clamp(best);
}

// ------------------------------------------------------------------------------------------------- traceback
RP_HD uint64_t mseg(int kind, int a, int b) { return (uint64_t)kind | ((uint64_t)(unsigned)a << 8) | ((uint64_t)(unsigned)b << 32); }

// One warp (or lane 0 alone): pair table pt[0..n-1] (pt[k-1] = partner of base k, 0 unpaired) of a structure that reaches
// scalar(0).  Returns 0, or 1 when a decision finds no candidate (cannot happen for a value below MFE_BIG).
template <bool SHFL>
RP_HD int mfe_traceback(MfeCtx& c, int16_t* pt, int lane) {
  const DevModel& M = *c.M;
  const int n = c.n;
  uint64_t* stk = c.stack();
  for (int k = lane; k < n; k += SHFL ? 32 : 1) pt[k] = 0;
  const int top = c.scalar(0);
  if (top >= MFE_BIG) return 0;   // no structure at all cannot happen (the empty one is one); kept for safety
  int sp = 0, bad = 0;
  if (c.cp > 0) stk[sp++] = mseg(SG_TOP, 0, 0);
  else stk[sp++] = mseg(SG_PRE, 1, n);
  while (sp > 0) {
    const uint64_t e = stk[--sp];
    const int kind = (int)(e & 255), a = (int)((e >> 8) & 0xffffff), b = (int)(e >> 32);
    int x;
    switch (kind) {
      case SG_TOP: {
        const int cnt = 1 + (c.cp - 1) * (n - c.cp + 1);
        x = cand_first<SHFL>(cnt, lane, top, [&](int y) { return mfe_top_cand(c, y); });
        if (x < 0) { bad = 1; break; }
        if (x == 0) {
          if (c.cp <= n) stk[sp++] = mseg(SG_SUF, c.cp, n);
          if (c.cp - 1 >= 1) stk[sp++] = mseg(SG_PRE, 1, c.cp - 1);
        } else {
          const int n2 = n - c.cp + 1, p = 1 + (x - 1) / n2, l = c.cp + (x - 1) % n2;
          if (l + 1 <= n) stk[sp++] = mseg(SG_SUF, l + 1, n);
          stk[sp++] = mseg(SG_C, p, l);
          if (p - 1 >= 1) stk[sp++] = mseg(SG_PRE, 1, p - 1);
        }
        break;
      }
      case SG_PRE: {   // region a..b, a = its strand's start
        const int v = c.pre(b);
        if (v == 0 && b - a <= TURN) break;
        x = cand_first<SHFL>(b - TURN - a + 1 > 1 ? b - TURN - a + 1 : 1, lane, v, [&](int y) { return mfe_pre_cand(c, a, b, y); });
        if (x < 0) { bad = 1; break; }
        if (x == 0) {
          if (b - 1 >= a) stk[sp++] = mseg(SG_PRE, a, b - 1);
        } else {
          const int k = a + x - 1;
          stk[sp++] = mseg(SG_C, k, b);
          if (k - 1 >= a) stk[sp++] = mseg(SG_PRE, a, k - 1);
        }
        break;
      }
      case SG_SUF: {   // region a..b, b = its strand's end
        const int v = c.suf(a);
        if (v == 0 && b - a <= TURN) break;
        x = cand_first<SHFL>(b - a - TURN + 1 > 1 ? b - a - TURN + 1 : 1, lane, v, [&](int y) { return mfe_suf_cand(c, a, b, y); });
        if (x < 0) { bad = 1; break; }
        if (x == 0) {
          if (a + 1 <= b) stk[sp++] = mseg(SG_SUF, a + 1, b);
        } else {
          const int l = a + TURN + x;
          if (l + 1 <= b) stk[sp++] = mseg(SG_SUF, l + 1, b);
          stk[sp++] = mseg(SG_C, a, l);
        }
        break;
      }
      case SG_C: {
        const int i = a, j = b, type = mfe_type(c, i, j);
        if (lane == 0) { pt[i - 1] = (int16_t)j; pt[j - 1] = (int16_t)i; }
        const int v = c.tb(MT_C, j - i, i) - pair_term(c, i, j);
        x = cand_first<SHFL>(MFE_C_CANDS, lane, v, [&](int y) { return mfe_c_cand(c, i, j, type, y); });
        if (x < 0) { bad = 1; break; }
        if (x == MFE_C_CANDS - 2) {
          stk[sp++] = mseg(SG_FM2, i + 1, j - 1);
        } else if (x == MFE_C_CANDS - 1) {
          if (j - 1 >= c.cp) stk[sp++] = mseg(SG_PRE, c.cp, j - 1);
          if (i + 1 <= c.cp - 1) stk[sp++] = mseg(SG_SUF, i + 1, c.cp - 1);
        } else if (x > 0) {
          int u1, u2;
          int_uv(x - 1, u1, u2);
          stk[sp++] = mseg(SG_C, i + 1 + u1, j - 1 - u2);
        }
        break;
      }
      case SG_FM1: {
        const int i = a, j = b, d = j - i, v = c.tb(MT_FM1, d, i), type = mfe_type(c, i, j);
        if (type && ss(c, i - 1, i) && ss(c, j, j + 1) && c.tb(MT_C, d, i) + e_ml_of(c, type, i, j) == v) stk[sp++] = mseg(SG_C, i, j);
        else if (ss(c, j - 1, j) && c.tb(MT_FM1, d - 1, i) + M.i_MLbase == v) stk[sp++] = mseg(SG_FM1, i, j - 1);
        else bad = 1;
        break;
      }
      case SG_FML: {
        const int i = a, j = b, d = j - i, v = c.tb(MT_FML, d, i);
        if (c.tb(MT_FM1, d, i) == v) stk[sp++] = mseg(SG_FM1, i, j);
        else if (ss(c, i, i + 1) && c.tb(MT_FML, d - 1, i + 1) + M.i_MLbase == v) stk[sp++] = mseg(SG_FML, i + 1, j);
        else if (c.tb(MT_FM2, d, i) == v) stk[sp++] = mseg(SG_FM2, i, j);
        else bad = 1;
        break;
      }
      default: {   // SG_FM2
        const int i = a, j = b, v = c.tb(MT_FM2, j - i, i);
        x = cand_first<SHFL>(j - i - 2 * TURN - 2, lane, v, [&](int y) { return mfe_fm2_cand(c, i, j, y); });
        if (x < 0) { bad = 1; break; }
        const int k = i + TURN + 2 + x;
        stk[sp++] = mseg(SG_FM1, k, j);
        stk[sp++] = mseg(SG_FML, i, k - 1);
        break;
      }
    }
    if (bad) break;
  }
  return bad;
}

// ------------------------------------------------------------------------------------------------- one problem
// The executor contract of mcc_driver.h (phase(id, f(tid)), nthreads(), kShfl).  red: nthreads() ints of CTA-shared
// scratch.  Writes pt[0..n-1] and returns the minimum (tables only; the host adds the unpaired constant), MFE_INF if the
// traceback failed.
template <class Exec>
RP_HD void solve_mfe(Exec& ex, MfeCtx& c, int* red, int16_t* pt, int* out_e) {
  constexpr bool SHFL = Exec::kShfl;
  const int T = ex.nthreads();
  ex.phase(0, [&](int tid) { mfe_prologue(c, tid, T); });
  for (int d = TURN + 1; d <= c.n; d++) ex.phase(1, [&](int tid) { mfe_diagonal<SHFL>(c, d, tid, T); });
  ex.phase(2, [&](int tid) { mfe_top_part(c, red, tid, T); });
  ex.phase(3, [&](int tid) { mfe_top_finish(c, red, tid, T); });
  ex.phase(4, [&](int tid) {
    if (tid >= 32 || (!SHFL && tid)) return;
    const int bad = mfe_traceback<SHFL>(c, pt, tid);
    if (tid == 0) *out_e = bad ? MFE_INF : c.scalar(0);
  });
}

}  // namespace rp
#endif
