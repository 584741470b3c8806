// mcc_core.h -- the McCaskill wavefront, written once as per-thread phase
// functions.  The CUDA kernels (kernels.cu) run them with tid = threadIdx.x and
// __syncthreads() between phases; tests/emul compiles the SAME functions for
// the host and runs the threads of a CTA one after another, so kernel logic is
// debugged on a CPU-only box.  (The emulator is test infrastructure; the
// product only ever runs the CUDA build.)
//
// What is computed (reference call sites):
//   linear   : Vienna::pf_fold + export_bppm  (src/ractip.cpp:356-367)
//              Vienna::pf_unstru, sum H+I+M+E (src/ractip.cpp:371-375)
//   two-strand: Vienna::co_pf_fold + export_co_bppm (src/ractip.cpp:442-447)
// with dangles=2, TURN=3, MAXLOOP=30, pf_scale from DevModel.
//
// Layout: every O(n^2) table is stored DIAGONAL-MAJOR: cell (i,j), 1<=i<=j<=n,
// lives at element d*ld + i with d=j-i, ld=n+1.  Cells of one anti-diagonal
// wavefront are contiguous, so every operand stream of every recurrence is a
// constant-stride walk:
//   sum_k A(i,k-1)*B(k,j)  ->  sum_a A[a][i] * B[d-1-a][i+1+a]
//   interior rows          ->  sum_u2 g[u1][u2] * B[d-2-u1-u2][i+1+u1]
//
#ifndef RP_MCC_CORE_H
#define RP_MCC_CORE_H

#include <math.h>
#include <stdint.h>

#include "dev_model.h"

#ifdef __CUDACC__
#define RP_HD __host__ __device__ __forceinline__
#else
#define RP_HD inline
#endif

// Tuning hooks (RP_DEBUG_SKIP switches, RP_PROFILE cycle counters) exist only in a -DRP_TUNE build: in the
// product build they cost code size, and the per-diagonal loops have to fit the 32 KB instruction cache.
#ifdef RP_TUNE
#define RP_DBG(c) ((c).dbg)
#define RP_PROF(c) ((c).prof)
#else
#define RP_DBG(c) 0
#define RP_PROF(c) (static_cast<long long*>(nullptr))
#endif

namespace rp {

// ---------------------------------------------------------------------------
// problem descriptor and workspace
// ---------------------------------------------------------------------------
enum { KIND_LINEAR = 0, KIND_COFOLD = 1, KIND_DUPLEX = 2 };

struct Problem {
  int seq_off;        // offset of S[1] in the batch's encoded-sequence buffer
  int n;              // length (n1+n2 for two-strand problems)
  int cp;             // first index of strand 2 (0: single strand)
  int kind;
  int pair;           // index of the rp_pair this problem belongs to
  int which;          // 0: s1, 1: s2, 2: s1&s2
  int max_w;
  int n1, n2;
  long long out_bp;   // float offsets into the dense output, -1 if absent
  long long out_up;
  long long out_hp;
  float th_hy;
  int defer_up;       // 1: the unpaired-window pass runs later in its own kernel (unstru_kernel) on the tables left in ws_off
  long long ws_off;   // >= 0: private workspace (doubles from BatchDev::ws_up) that outlives the wavefront kernel; -1: the CTA's slot
};
// queue entries: problem index, + RP_JOB_UNPAIRED for the unpaired-window pass of a deferred problem as a job of its own
constexpr int RP_JOB_UNPAIRED = 0x40000000;

enum {
  T_Q = 0, T_QQ, T_QM, T_QM1, T_QM2, T_QB, T_QBI, T_QB1N, T_QBAU,
  T_OUT, T_OUTI, T_OUT1N, T_OUTAU, T_MC, T_PR, T_PRML, T_PMLB, T_PL,
  T_DG, T_RR, T_LL, T_XX,
  T_QS, T_PRB, T_MLB,   // band-bulk split sums of the general kernel (see inside_band_A / outside_band_A)
  T_QMR, T_PRMLR,       // wide schedule: ROW-major copies of qm and PRML (element (i,j) at (i-1)*ld + j), see Ctx::rptr
  T_LIST,   // not doubles: per-diagonal lists of pairable cells (uint16), general kernel only
  T_COUNT
};
enum {
  V_SCALE = 0, V_MLB, V_HPW, V_SP3, V_SP4, V_SP6, V_U0, V_U1,
  V_COUNT
};

// longest sequence (n1+n2 for two-strand problems) whose workspace slot stays below 2^32 doubles
constexpr int RP_MAX_N = 12000;
RP_HD size_t table_elems(int n) { return (size_t)n * (size_t)(n + 1) + 8; }
RP_HD size_t vector_elems(int n) { return (size_t)n + 8; }
RP_HD size_t slot_doubles(int n) { return T_COUNT * table_elems(n) + V_COUNT * vector_elems(n); }

// one problem per CTA (or cluster), elements contiguous; the work of a cell is sliced over threads
struct Ctx {
  const DevModel* M;
  const uint8_t* S;   // S[1..n]; low 3 bits base code 0..4, bit 3 = "letter is not A/C/G/U"
  int n, cp, ld, kind, max_w;
  double* ws;         // slot workspace: T_COUNT tables then V_COUNT vectors
  unsigned te, ve;    // elements per table / per vector (a slot is < 2^32 doubles: n <= RP_MAX_N, checked by the host)
  double invZ;        // set after the inside pass
  int dbg;            // tuning aid (RP_DEBUG_SKIP): 1 skip interior rows, 2 skip split sums, 4 skip gap sums
  long long* prof;    // RP_PROFILE counters (slots 40..: fine-grained probes of thread 0) or null
  // Tables whose rows are only read while they are recent are RINGS of a few rows (row d at d & mask):
  // PR/PL/PMLB are read one diagonal after they are written, the band results QS/PRB/MLB within a
  // band.  A full table would leave every written line behind in L2, where it pushes out the history
  // tables the split sums stream (the 126 MB L2 holds the history of all resident problems, not more).
  RP_HD static constexpr unsigned ring_mask(int t) {
    return (t == T_PR || t == T_PL || t == T_PMLB) ? 1u : (t == T_QS || t == T_PRB || t == T_MLB) ? 15u : 0xffffffffu;
  }
  // 32-bit element offsets: one IMAD per term instead of 64-bit multiplies (a third of all instructions otherwise)
  RP_HD unsigned off(int t, int d, int i) const { return (unsigned)t * te + ((unsigned)d & ring_mask(t)) * (unsigned)ld + (unsigned)i; }
  RP_HD double& tb(int t, int d, int i) const { return ws[off(t, d, i)]; }
  RP_HD double* ptr(int t, int d, int i) const { return ws + off(t, d, i); }
  // The ML sum of the outside far pass walks COLUMNS (PRML(i,l), qm(i+1,k-1) over i, lanes = neighbouring l): in the
  // diagonal-major tables neighbouring lanes are a whole row apart (one 32-byte sector per 8-byte operand), in the
  // row-major copies they are neighbours.
  RP_HD double* rptr(int t, int i, int j) const { return ws + ((unsigned)t * te + (unsigned)(i - 1) * (unsigned)ld + (unsigned)j); }
  RP_HD double& v(int vv, int k) const { return ws[(unsigned)T_COUNT * te + (unsigned)vv * ve + (unsigned)k]; }
  RP_HD int dstep() const { return ld; }   // one diagonal up, same position
  RP_HD int pstep() const { return 1; }    // same diagonal, next position
  RP_HD int sraw(int i) const { return S[i]; }
};

RP_HD void bind_ctx(Ctx& c, const DevModel* M, const uint8_t* S, const Problem& p, double* ws) {
  c.M = M; c.S = S; c.n = p.n; c.cp = p.cp; c.ld = p.n + 1; c.kind = p.kind; c.max_w = p.max_w;
  c.ws = ws; c.te = (unsigned)table_elems(p.n); c.ve = (unsigned)vector_elems(p.n);
  c.invZ = 0;
  c.dbg = 0;
  c.prof = nullptr;
}
#define TB(c, t, d, i) ((c).tb(t, d, i))
// store of a value that is not read again soon (qb, out, class tables, outputs): evict-first, so that
// it does not displace the history tables in L2
#ifdef __CUDA_ARCH__
#define RP_ST_STREAM(ref, v) __stcs(&(ref), (v))
#else
#define RP_ST_STREAM(ref, v) ((ref) = (v))
#endif
#define VEC(c, vec_id, k) ((c).v(vec_id, k))

// Per-diagonal compaction of the cells that can pair (static per sequence; general kernel):
//   LIST[d*ld + r] = i of the r-th pairable cell (i,i+d);  POS[d*ld + i] = #pairable cells (i',i'+d), i' < i.
// Interior-loop work is dealt out over these lists, so no thread idles on a cell that cannot pair.
RP_HD uint16_t* listp(const Ctx& c) { return reinterpret_cast<uint16_t*>(c.ptr(T_LIST, 0, 0)); }
RP_HD uint16_t* posp(const Ctx& c) { return reinterpret_cast<uint16_t*>(c.ptr(T_LIST, 0, 0)) + c.te * 2; }

// Width of a band of diagonals whose O(n) split sums depend only on diagonals finished before the
// band starts: qm, qm1 and qq vanish on diagonals <= TURN, so the terms of diagonal d reach back at
// least TURN+2 diagonals.
constexpr int BAND = TURN + 2;
// The general kernel can sum WIDE bands (wide_* functions): a far pass every W <= WIDE_MAX diagonals covers the
// terms whose operands are final by then, the few remaining (near) terms are added when a cell is finished.
constexpr int WIDE_MAX = 15;

// CTA-shared scratch (CUDA shared memory; a heap block in the host emulation)
constexpr int RP_SMEM_SEQ = 4096;  // sequence bytes staged in shared memory (n+2)
struct Shared {
  int T;
  double* part;     // [2*W][T] partial sums of the current phase (general kernel; W = width of its bands)
  double* grow;     // [MAXLOOP+1][GROW_LD] run weights of the factorised interior loops (DevModel::grow)
  double* ghead_b;  // [GROW_LD]
  double* ghead_1;  // [GROW_LD]
  double* red;      // [128] small reductions (nick sums)
  uint8_t* S;       // [RP_SMEM_SEQ + 8] staged sequence(s)
  double* gtile;    // wide builds: staged generic-class rows of a chunk (see "Staged generic interior sums"); aliases part
  double* gpart;    // wide builds: partial generic sums [bin][cell]; aliases part
};
// Staged generic interior sums (wide builds of the general kernel, long problems).  The generic-class taps of the
// interior-loop sum (375 of the 496 terms of a cell) are summed DENSELY out of a shared-memory tile: the rows
// s = 6..30 of the generic class table (diagonals d -/+ (2+s)) over the positions a chunk of cells can reach are
// copied into shared memory once per chunk, zero where a position is invalid, and a thread walks a row for 8
// neighbouring cells with a sliding register window (one shared load per 8 FMAs, no predicates) -- the band
// kernel's scheme, per chunk instead of per problem.  The ends (bulge, 1xn) and the table-driven shapes are five
// batched items per pairable cell (ends_items).
constexpr int GS_ROW0 = 6, GS_NROWS = MAXLOOP - GS_ROW0 + 1;             // rows 6..30
RP_HD int gs_lt(int T) { return (T + MAXLOOP + 8 + 7) / 8 * 8; }          // elements per tile row (multiple of 8)
constexpr int GS_KINDS = 5;   // ends_items: bulge row, 1xn row, bulge heads, 1xn heads, table-driven shapes
RP_HD size_t gs_doubles(int T) { return (size_t)GS_KINDS * T + (size_t)GS_NROWS * gs_lt(T) + 8 * (size_t)T; }   // ends partials + tile + [bin][cell]
RP_HD size_t part_doubles(int T, int W) {
  const size_t far = 2 * (size_t)W * T;
  return (W > BAND && gs_doubles(T) > far) ? gs_doubles(T) : far;
}
RP_HD size_t shared_bytes(int T, int W = BAND) {
  return sizeof(double) * (part_doubles(T, W) + (MAXLOOP + 1) * GROW_LD + 2 * GROW_LD + 128) + RP_SMEM_SEQ + 16;
}
RP_HD void carve_shared(Shared& sh, void* base, int T, int W = BAND) {
  sh.T = T;
  double* p = static_cast<double*>(base);
  sh.part = p; p += part_doubles(T, W);
  sh.gtile = sh.part + (size_t)GS_KINDS * T;
  sh.gpart = sh.gtile + (size_t)GS_NROWS * gs_lt(T);
  sh.grow = p; p += (MAXLOOP + 1) * GROW_LD;
  sh.ghead_b = p; p += GROW_LD;
  sh.ghead_1 = p; p += GROW_LD;
  sh.red = p; p += 128;
  sh.S = reinterpret_cast<uint8_t*>(p);
}

// ---------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------
template <class C>
RP_HD int base(const C& c, int i) { return c.sraw(i) & 7; }

RP_HD int pair_type(int a, int b) {
  // CG=1 GC=2 GU=3 UG=4 AU=5 UA=6 ; a,b in 0..4 (N,A,C,G,U).  One nibble per (a-1,b-1).
  const uint64_t LUT = (5ull << 12) | (1ull << 24) | (2ull << 36) | (3ull << 44) | (6ull << 48) | (4ull << 56);
  const int idx = ((a - 1) & 3) * 4 + ((b - 1) & 3);
  const int t = (int)((LUT >> (4 * idx)) & 15);
  return (a && b) ? t : 0;
}
RP_HD int rtype(int t) { return t == 0 ? 0 : (t == 7 ? 7 : ((t - 1) ^ 1) + 1); }

// ViennaRNA SAME_STRAND(a,b) for a<b
template <class C>
RP_HD bool ss(const C& c, int a, int b) { return c.cp <= 0 || a >= c.cp || b < c.cp; }

// Outside pass of a two-strand problem: RactIP keeps only the probabilities of pairs that JOIN the strands
// (i < cp <= j; reference src/ractip.cpp:451-453), and the outside value of such a pair depends on enclosing
// pairs only, which join the strands as well (exterior, interior and multiloop contexts alike; the
// nicked-loop context exists for same-strand stems only).  So the outside wavefront of a two-strand problem
// runs over the inter-strand cells of a diagonal, k in [cross_lo, cross_hi], and needs no nick sums.
// Single strand: all cells.
template <class C>
RP_HD int cross_lo(const C& c, int d) { return c.cp > 0 ? (c.cp - d > 1 ? c.cp - d : 1) : 1; }
template <class C>
RP_HD int cross_hi(const C& c, int d) { return c.cp > 0 ? (c.cp - 1 < c.n - d ? c.cp - 1 : c.n - d) : c.n - d; }

// (MT: DevModel, or the shared-memory copy of its small tables used by the band kernel)
template <class MT>
RP_HD double ext_stem(const MT& M, int type, int s5, int s3) {
  double e = 1.0;
  if (s5 >= 0 && s3 >= 0) e = M.mmExt[type][s5][s3];
  else if (s5 >= 0) e = M.dangle5[type][s5];
  else if (s3 >= 0) e = M.dangle3[type][s3];
  if (type > 2) e *= M.expTermAU;
  return e;
}
template <class MT>
RP_HD double ml_stem(const MT& M, int type, int s5, int s3) {
  double e = 1.0;
  if (s5 >= 0 && s3 >= 0) e = M.mmM[type][s5][s3];
  else if (s5 >= 0) e = M.dangle5[type][s5];
  else if (s3 >= 0) e = M.dangle3[type][s3];
  if (type > 2) e *= M.expTermAU;
  return e * M.expMLintern;
}

// the nine (u1,u2) combinations that do not factorise
#define RP_N_SPECIAL 9
RP_HD void special_uv(int s, int& u1, int& u2) {
  const int U1[RP_N_SPECIAL] = {0, 1, 0, 1, 1, 2, 2, 2, 3};
  const int U2[RP_N_SPECIAL] = {0, 0, 1, 1, 2, 1, 2, 3, 2};
  u1 = U1[s]; u2 = U2[s];
}
RP_HD int special_index(int u1, int u2) {
  // inverse of special_uv: (0,0)->0 (1,0)->1 (0,1)->2 (1,1)->3 (1,2)->4 (2,1)->5 (2,2)->6 (2,3)->7 (3,2)->8
  if (u1 == 0) return u2 == 0 ? 0 : 2;
  if (u1 == 1) return u2 == 0 ? 1 : (u2 == 1 ? 3 : 4);
  if (u1 == 2) return u2 == 1 ? 5 : (u2 == 2 ? 6 : 7);
  return 8;
}
// weight (incl. scale) of special shape s: closing pair `type` with neighbours
// (si1,sj1), inner pair of reversed type t2r with neighbours (sp1,sq1)
template <class MT>
RP_HD double special_loop(const MT& M, int s, int type, int t2r, int si1, int sj1, int sp1, int sq1) {
  // one look-up in the table of finished weights (DevModel::spw, dev_model.h); with a compile-time s the
  // switch folds away and the index is a handful of integer multiply-adds
  int ix;
  switch (s) {
    case 0: ix = SPW_STACK + type * 8 + t2r; break;
    case 1:
    case 2: ix = SPW_BULGE1 + type * 8 + t2r; break;
    case 3: ix = SPW_INT11 + ((type * 8 + t2r) * 5 + si1) * 5 + sj1; break;
    case 4: ix = SPW_INT21 + (((type * 8 + t2r) * 5 + si1) * 5 + sq1) * 5 + sj1; break;   // u1=1,u2=2
    case 5: ix = SPW_INT21 + (((t2r * 8 + type) * 5 + sq1) * 5 + si1) * 5 + sp1; break;   // u1=2,u2=1
    case 6: ix = SPW_INT22 + ((((type * 8 + t2r) * 5 + si1) * 5 + sp1) * 5 + sq1) * 5 + sj1; break;
    default: ix = SPW_23 + ((((type * 5 + si1) * 5 + sj1) * 8 + t2r) * 5 + sq1) * 5 + sp1; break;
  }
  return M.spw[ix];
}

// hairpin weight of pair (i,j), including scale[u+2]
template <class C>
RP_HD double hairpin(const C& c, int i, int j, int type) {
  const int u = j - i - 1;
  if (c.M->special_hp) {
    if (u == 4 && VEC(c, V_SP4, i) >= 0.) return VEC(c, V_SP4, i);  // type==7 never occurs for ACGU pairs
    if (u == 6 && VEC(c, V_SP6, i) >= 0.) return VEC(c, V_SP6, i);
    if (u == 3) {
      if (VEC(c, V_SP3, i) >= 0.) return VEC(c, V_SP3, i);
      return type > 2 ? VEC(c, V_HPW, 3) * c.M->expTermAU : VEC(c, V_HPW, 3);
    }
  }
  return VEC(c, V_HPW, u) * c.M->mmH[type][base(c, i + 1)][base(c, j - 1)];
}

// weighted sum along one row of the factorised interior loops:
//   sum_{u2=lo..hi} g[u2] * p[u2*step]
RP_HD double row_sum(const double* g, const double* p, int step, int lo, int hi) {
  double a0 = 0., a1 = 0., a2 = 0., a3 = 0.;
  const double* q = p + (long)lo * step;
  g += lo;
  int cnt = hi - lo + 1;
  for (; cnt >= 4; cnt -= 4) {
    a0 += g[0] * q[0];
    a1 += g[1] * q[step];
    a2 += g[2] * q[2 * step];
    a3 += g[3] * q[3 * step];
    g += 4;
    q += 4 * step;
  }
  for (; cnt > 0; cnt--) {
    a0 += g[0] * q[0];
    g++;
    q += step;
  }
  return (a0 + a1) + (a2 + a3);
}

// The factorised part of the interior-loop sum of one cell, restricted to the
// row pairs (q, 30-q), q = sl, sl+SI, ... (each pair holds 32 terms, so slices
// are balanced).  SIGN=+1: inside, inner pair (i+1+u1, j-1-u2) lies u1+u2+2
// diagonals below the cell; SIGN=-1: outside, enclosing pair (k-1-u1, l+1+u2)
// lies above.  TI/T1/TA point at the cell's own entry of the three class
// tables; ds/ps are the diagonal and position strides.  Bounds: u1 <= u1max,
// u2 <= u2cap, u1+u2+2 <= ddmax; every element touched is a valid cell.
template <int SIGN>
RP_HD void interior_rows(const Shared& sh, const double* TI, const double* T1, const double* TA, int ds, int ps,
                         int u1max, int u2cap, int ddmax, int sl, int SI, double& sI, double& s1, double& sA) {
  const int step = -SIGN * ds;
  for (int q = sl; q <= MAXLOOP / 2; q += SI) {
    for (int h = 0; h < 2; h++) {
      const int u1 = h == 0 ? q : MAXLOOP - q;
      if (h == 1 && u1 == q) break;
      if (u1 > u1max) continue;
      int u2hi = MAXLOOP - u1;
      if (u2cap < u2hi) u2hi = u2cap;
      if (ddmax - 2 - u1 < u2hi) u2hi = ddmax - 2 - u1;
      if (u2hi < 0) continue;
      const long o0 = -(long)SIGN * ((long)(u1 + 2) * ds - (long)(1 + u1) * ps);  // element (u1, u2=0)
      const double* g = sh.grow + u1 * GROW_LD;
      if (u1 == 0) {
        if (u2hi >= 2) sA += row_sum(g, TA + o0, step, 2, u2hi);
      } else if (u1 == 1) {
        if (u2hi >= 3) s1 += row_sum(g, T1 + o0, step, 3, u2hi);
      } else {
        sA += sh.ghead_b[u1] * TA[o0];
        if (u2hi >= 1) s1 += sh.ghead_1[u1] * T1[o0 + step];
        if (u2hi >= 2) sI += row_sum(g, TI + o0, step, 2, u2hi);
      }
    }
  }
}

// sum of A[x*sa] * B[x*sb] over x in [x0,x1) with x = s (mod S)
RP_HD double dot_range(const double* A, int sa, const double* B, int sb, int x0, int x1, int s, int S) {
  int x = x0 + ((s - x0) % S + S) % S;
  if (x >= x1) return 0.;
  int cnt = (x1 - 1 - x) / S + 1;
  const double* a = A + (long)x * sa;
  const double* b = B + (long)x * sb;
  const int da = S * sa, db = S * sb;
  double a0 = 0., a1 = 0., a2 = 0., a3 = 0.;
  for (; cnt >= 4; cnt -= 4) {
    a0 += a[0] * b[0];
    a1 += a[da] * b[db];
    a2 += a[2 * da] * b[2 * db];
    a3 += a[3 * da] * b[3 * db];
    a += 4 * da;
    b += 4 * db;
  }
  for (; cnt > 0; cnt--) {
    a0 += a[0] * b[0];
    a += da;
    b += db;
  }
  return (a0 + a1) + (a2 + a3);
}
// same over x in [0,cnt) skipping x == skip (the split that would fall on the nick)
RP_HD double strided_dot(const double* A, int sa, const double* B, int sb, int cnt, int s, int S, int skip) {
  if (skip < 0 || skip >= cnt) return dot_range(A, sa, B, sb, 0, cnt, s, S);
  return dot_range(A, sa, B, sb, 0, skip, s, S) + dot_range(A, sa, B, sb, skip + 1, cnt, s, S);
}
// Up to 8 dot products that share the streamed operand A:
//   acc[t] += sum_{x<cnt} A[x*sa] * B[t*tb + x*sb],  t < nu
RP_HD void multi_dot(const double* A, int sa, const double* B, int sb, int tb, int cnt, int nu, double* acc) {
  for (int x = 0; x < cnt; x++, A += sa, B += sb) {
    const double a = *A;
#pragma unroll
    for (int t = 0; t < 8; t++)
      if (t < nu) acc[t] += a * B[t * tb];
  }
}

// The same when the shifts advance along the stream itself (tb == sb):
//   acc[t] += sum_{x<cnt} A[x*sa] * B[(x+t)*sb],  t = 0..7
// B is walked ONCE with an 8-deep register window (2 loads per 8 FMAs instead of 9), and the 16
// loads of a block of 8 steps are issued together (one memory round trip per block).
// Window element z = x+t is read only if zlo <= z <= zhi (else it counts as 0); the caller
// ignores the acc[t] it did not ask for.  Negative strides walk a stream backwards.
RP_HD void multi_dot_slide(const double* A, long sa, const double* B, long sb, int cnt, int zlo, int zhi, double* acc) {
  if (cnt <= 0) return;
  double win[8];
#pragma unroll
  for (int t = 0; t < 7; t++) win[t] = (t >= zlo && t <= zhi) ? B[t * sb] : 0.;
  win[7] = 0.;
  const double* bp = B + 7 * sb;  // next element to enter the window
  int z = 7;
  int x = 0;
#pragma unroll 1
  for (; x + 8 <= cnt; x += 8) {
    double nb[8], na[8];
    if (z >= zlo && z + 7 <= zhi) {
#pragma unroll
      for (int u = 0; u < 8; u++) nb[u] = bp[u * sb];
    } else {
#pragma unroll
      for (int u = 0; u < 8; u++) nb[u] = (z + u >= zlo && z + u <= zhi) ? bp[u * sb] : 0.;
    }
#pragma unroll
    for (int u = 0; u < 8; u++) na[u] = A[u * sa];
    bp += 8 * sb; A += 8 * sa; z += 8;
#pragma unroll
    for (int u = 0; u < 8; u++) {
      win[(u + 7) & 7] = nb[u];
#pragma unroll
      for (int t = 0; t < 8; t++) acc[t] += na[u] * win[(u + t) & 7];
    }
  }
#pragma unroll
  for (int u = 0; u < 7; u++) {
    if (x + u < cnt) {
      win[(u + 7) & 7] = (z >= zlo && z <= zhi) ? *bp : 0.;
      bp += sb; z++;
      const double a = *A;
      A += sa;
#pragma unroll
      for (int t = 0; t < 8; t++) acc[t] += a * win[(u + t) & 7];
    }
  }
}

// partition of a chunk of `C` cells over T threads: Cp cells x S slices (general kernel)
struct Split {
  int Cp, S;
};
RP_HD Split make_split(int C, int T) {
  Split s;
  int Cp = (C + 31) & ~31;
  if (Cp > T) Cp = T;
  s.Cp = Cp;
  s.S = T / Cp;
  if (s.S < 1) s.S = 1;
  return s;
}
// work split of the interior-loop items of a chunk: cnt pairable cells x SI slices
struct ISplit {
  int lo, cnt, cntp, SI;
};
RP_HD ISplit make_isplit(const Ctx& c, int d, int i0, int C, int T) {
  const uint16_t* P = posp(c) + (size_t)d * c.ld;
  ISplit s;
  s.lo = P[i0];
  s.cnt = (int)P[i0 + C] - s.lo;
  int cp = (s.cnt + 31) & ~31;
  if (cp > T) cp = T;
  if (cp < 32) cp = 32;
  s.cntp = cp;
  int si = T / cp;  // slices per cell: a power of two <= 16 (there are 16 row pairs)
  s.SI = si >= 16 ? 16 : si >= 8 ? 8 : si >= 4 ? 4 : si >= 2 ? 2 : 1;
  return s;
}

// ---------------------------------------------------------------------------
// prologue.  (ct, nct) = index and number of the threads that share one problem.
// ---------------------------------------------------------------------------
RP_HD void load_shared_model(const DevModel& M, const Shared& sh, int tid) {
  for (int x = tid; x < (MAXLOOP + 1) * GROW_LD; x += sh.T) sh.grow[x] = M.grow[x / GROW_LD][x % GROW_LD];
  for (int x = tid; x < GROW_LD; x += sh.T) {
    sh.ghead_b[x] = M.ghead_b[x];
    sh.ghead_1[x] = M.ghead_1[x];
  }
}

template <class C>
RP_HD void prologue_vectors(C& c, int ct, int nct) {
  const DevModel& M = *c.M;
  const int n = c.n;
  // scale[k] = pf_scale^-k, mlb[k] = (expMLbase/pf_scale)^k: built by repeated
  // multiplication by one thread so that every consumer sees the same values
  if (ct == 0) {
    double s = 1.0, b = 1.0;
    for (int k = 0; k <= n + 2; k++) {
      VEC(c, V_SCALE, k) = s;
      VEC(c, V_MLB, k) = b;
      s *= M.scale1;
      b *= M.mlb1;
    }
  }
  (void)nct;
}

// pair lists of the general kernel: one thread per diagonal
RP_HD void prologue_lists(Ctx& c, int tid, int T) {
  const int n = c.n;
  uint16_t* LIST = listp(c);
  uint16_t* POS = posp(c);
  for (int d = tid; d < n; d += T) {
    uint16_t* L = LIST + (size_t)d * c.ld;
    uint16_t* P = POS + (size_t)d * c.ld;
    int cnt = 0;
    for (int i = 1; i <= n - d; i++) {
      P[i] = (uint16_t)cnt;
      if (d > TURN && pair_type(base(c, i), base(c, i + d))) L[cnt++] = (uint16_t)i;
    }
    P[n - d + 1 <= n ? n - d + 1 : n] = (uint16_t)cnt;  // d = 0: i = n+1 does not exist and is never asked for
    if (d == 0) P[n] = 0;
  }
}

template <class C>
RP_HD void prologue2(C& c, int ct, int nct) {
  const DevModel& M = *c.M;
  const int n = c.n;
  for (int u = ct; u <= n; u += nct) {
    double q;
    if (u <= 30) q = M.exphairpin[u];
    else q = M.exphairpin[30] * exp(-(M.lxc * log(u / 30.)) * 10. / M.kT);
    VEC(c, V_HPW, u) = q * VEC(c, V_SCALE, u + 2);
  }
  for (int i = ct; i <= n + 1; i += nct) {
    double s3 = -1., s4 = -1., s6 = -1.;
    if (i >= 1) {
      // window codes: base-8 digits, 7 for letters that cannot match a list entry
      int code = 0;
      bool in = true;
      for (int k = 0; k < 8; k++) {
        int p = i + k;
        int dgt = 0;
        if (p <= n) dgt = (c.sraw(p) & 8) ? 7 : (c.sraw(p) & 7);
        else in = false;
        code = code * 8 + dgt;
        // a hairpin window never spans the nick (hairpins need ss(i,j))
        if (k == 4 && in) {
          for (int e = 0; e < M.n_tri; e++)
            if (M.tri_code[e] == code) { s3 = M.exptri[e] * VEC(c, V_SCALE, 5); break; }
        } else if (k == 5 && in) {
          for (int e = 0; e < M.n_tetra; e++)
            if (M.tetra_code[e] == code) { s4 = M.exptetra[e] * VEC(c, V_SCALE, 6); break; }
        } else if (k == 7 && in) {
          for (int e = 0; e < M.n_hex; e++)
            if (M.hex_code[e] == code) { s6 = M.exphex[e] * VEC(c, V_SCALE, 8); break; }
        }
      }
    }
    VEC(c, V_SP3, i) = s3; VEC(c, V_SP4, i) = s4; VEC(c, V_SP6, i) = s6;
    VEC(c, V_U0, i) = 0.; VEC(c, V_U1, i) = 0.;
  }
  // diagonals 0..TURN: q = scale[d+1], everything else 0
  const int dmax = TURN < n - 1 ? TURN : n - 1;
  const int cells = (dmax + 1) * c.ld;
  for (int x = ct; x < cells; x += nct) {
    int d = x / c.ld, i = x % c.ld;
    bool valid = i >= 1 && i + d <= n;
    TB(c, T_Q, d, i) = valid ? VEC(c, V_SCALE, d + 1) : 0.;
    TB(c, T_QQ, d, i) = 0.; TB(c, T_QM, d, i) = 0.; TB(c, T_QM1, d, i) = 0.; TB(c, T_QM2, d, i) = 0.;
    TB(c, T_QB, d, i) = 0.; TB(c, T_QBI, d, i) = 0.; TB(c, T_QB1N, d, i) = 0.; TB(c, T_QBAU, d, i) = 0.;
    TB(c, T_OUT, d, i) = 0.; TB(c, T_OUTI, d, i) = 0.; TB(c, T_OUT1N, d, i) = 0.; TB(c, T_OUTAU, d, i) = 0.;
    TB(c, T_MC, d, i) = 0.; TB(c, T_PR, d, i) = 0.; TB(c, T_PRML, d, i) = 0.; TB(c, T_PMLB, d, i) = 0.;
    TB(c, T_PL, d, i) = 0.; TB(c, T_DG, d, i) = 0.;
  }
}

// ---------------------------------------------------------------------------
// inside pass, cell (i, j=i+d), d >= TURN+1
// ---------------------------------------------------------------------------
// slice sl of SI of the interior-loop sum of a cell that can pair
template <class C>
RP_HD double inside_interior(const C& c, const Shared& sh, int d, int i, int type, int sl, int SI) {
  const DevModel& M = *c.M;
  const int ddmax = d - (TURN + 1) < MAXLOOP + 2 ? d - (TURN + 1) : MAXLOOP + 2;
  if (ddmax < 2) return 0.;
  const int j = i + d;
  // strand guards: inner 5' end must stay on i's strand, inner 3' end on j's
  const int maxpo = (c.cp > 0 && i < c.cp) ? c.cp - 1 - i : 1000;
  const int maxu2 = (c.cp > 0 && j >= c.cp) ? j - 1 - c.cp : 1000;
  const int si1 = base(c, i + 1), sj1 = base(c, j - 1);
  int u1max = ddmax - 2 < MAXLOOP ? ddmax - 2 : MAXLOOP;
  if (maxpo - 1 < u1max) u1max = maxpo - 1;
  double sI = 0., s1 = 0., sA = 0.;
  if (!(RP_DBG(c) & 1))
    interior_rows<1>(sh, c.ptr(T_QBI, d, i), c.ptr(T_QB1N, d, i), c.ptr(T_QBAU, d, i), c.dstep(), c.pstep(), u1max, maxu2,
                     ddmax, sl, SI, sI, s1, sA);
  double accI = M.mmI[type][si1][sj1] * sI + M.mm1n[type][si1][sj1] * s1 + (type > 2 ? M.expTermAU : 1.0) * sA;
  // table-driven small loops
  for (int s = sl; s < RP_N_SPECIAL; s += SI) {
    int u1, u2;
    special_uv(s, u1, u2);
    const int dd = u1 + u2 + 2;
    if (dd > ddmax || u1 + 1 > maxpo || u2 > maxu2) continue;
    const int k = i + 1 + u1, l = j - 1 - u2;
    const int t2 = pair_type(base(c, k), base(c, l));
    if (!t2) continue;
    accI += TB(c, T_QB, d - dd, k) * special_loop(M, s, type, rtype(t2), si1, sj1, base(c, k - 1), base(c, l + 1));
  }
  return accI;
}

// slice `slice` of S of the two split sums of cell (i,j)
template <class C>
RP_HD void inside_splits(const C& c, int d, int i, int slice, int S, double& accM, double& accQ) {
  const int ds = c.dstep(), ps = c.pstep();
  accM = 0.; accQ = 0.;
  if (RP_DBG(c) & 2) return;
  // QM2(i,j) = sum_a qm[a][i] * qm1[d-1-a][i+1+a], a = TURN+1 .. d-2-TURN; the split k=i+1+a may not be the nick
  const int cntM = d - 2 * TURN - 2;
  if (cntM > 0) {
    const int skip = c.cp > 0 ? c.cp - 1 - i - (TURN + 1) : -1;  // a = cp-1-i  <=> k = cp
    accM = strided_dot(c.ptr(T_QM, TURN + 1, i), ds, c.ptr(T_QM1, d - 2 - TURN, i + TURN + 2), ps - ds, cntM, slice, S, skip);
  }
  // sum_a q[a][i] * qq[d-1-a][i+1+a], a = 0 .. d-2-TURN
  const int cntQ = d - 1 - TURN;
  if (cntQ > 0) accQ = strided_dot(c.ptr(T_Q, 0, i), ds, c.ptr(T_QQ, d - 1, i + 1), ps - ds, cntQ, slice, S, -1);
}

// combine: everything of cell (i,j) that is O(1) once the three sums are known
template <class C>
RP_HD void inside_finish(C& c, int d, int i, int type, double sI, double sM, double sQ) {
  const DevModel& M = *c.M;
  const int j = i + d, n = c.n;
  const double scale2 = VEC(c, V_SCALE, 2);
  double qb = 0.;
  if (type) {
    if (ss(c, i, j)) qb += hairpin(c, i, j, type);
    qb += sI;
    if (ss(c, i, i + 1) && ss(c, j - 1, j))
      qb += TB(c, T_QM2, d - 2, i + 1) * M.expMLclosing * ml_stem(M, rtype(type), base(c, j - 1), base(c, i + 1)) * scale2;
    if (!ss(c, i, j)) {
      // the loop that contains the nick is an exterior loop
      double t = scale2;
      if (i + 1 <= c.cp - 1) t *= TB(c, T_Q, c.cp - 2 - i, i + 1);
      if (c.cp <= j - 1) t *= TB(c, T_Q, j - 1 - c.cp, c.cp);
      t *= ext_stem(M, rtype(type), ss(c, j - 1, j) ? base(c, j - 1) : -1, ss(c, i, i + 1) ? base(c, i + 1) : -1);
      qb += t;
    }
  }
  TB(c, T_QB, d, i) = qb;
  TB(c, T_QM2, d, i) = sM;
  double fI = 0., f1 = 0., fA = 0.;
  if (type && qb != 0.) {
    const int t2 = rtype(type), sq1 = j < n ? base(c, j + 1) : 0, sp1 = i > 1 ? base(c, i - 1) : 0;
    fI = qb * M.mmI[t2][sq1][sp1];
    f1 = qb * M.mm1n[t2][sq1][sp1];
    fA = type > 2 ? qb * M.expTermAU : qb;
  }
  TB(c, T_QBI, d, i) = fI;
  TB(c, T_QB1N, d, i) = f1;
  TB(c, T_QBAU, d, i) = fA;
  // qm1: one stem starting at i, unpaired to its right
  double qm1 = ss(c, j - 1, j) ? TB(c, T_QM1, d - 1, i) * M.mlb1 : 0.;
  if (type && ss(c, i - 1, i) && ss(c, j, j + 1))
    qm1 += qb * ml_stem(M, type, i > 1 ? base(c, i - 1) : -1, j < n ? base(c, j + 1) : -1);
  TB(c, T_QM1, d, i) = qm1;
  // U(i,j) = sum_k mlb[k-i] qm1(k,j) = mlb1*(qm1(i+1,j) + U(i+1,j)), cut at the nick
  const int vprev = (d & 1) ? V_U0 : V_U1, vcur = (d & 1) ? V_U1 : V_U0;
  const double U = ss(c, i, i + 1) ? M.mlb1 * (TB(c, T_QM1, d - 1, i + 1) + VEC(c, vprev, i + 1)) : 0.;
  VEC(c, vcur, i) = U;
  TB(c, T_QM, d, i) = qm1 + sM + U;
  // exterior
  double qq = TB(c, T_QQ, d - 1, i) * M.scale1;
  if (type)
    qq += qb * ext_stem(M, type, (i > 1 && ss(c, i - 1, i)) ? base(c, i - 1) : -1,
                        (j < n && ss(c, j, j + 1)) ? base(c, j + 1) : -1);
  TB(c, T_QQ, d, i) = qq;
  TB(c, T_Q, d, i) = VEC(c, V_SCALE, d + 1) + qq + sQ;
}

template <class C>
RP_HD void inside_end(C& c) { c.invZ = 1.0 / TB(c, T_Q, c.n - 1, 1); }

// General kernel.  The two O(n) split sums of the inside pass are computed a BAND of diagonals at
// a time (inside_band_A/B): for row i the cells (i, i+d0+e), e < BAND, share the operand qm[a][i]
// (resp. q[a][i]), so one thread keeps BAND accumulators and loads 1+BAND values per BAND FMAs
// instead of 2 per FMA, and every operand lies on a diagonal < d0, already final.
//   M[e] = QM2(i,i+d0+e) = sum_{a=TURN+1}^{d0+e-TURN-2} qm[a][i] * qm1[d0+e-1-a][i+1+a]   (complete)
//   Q[e] = sum_{a=e}^{d0+e-TURN-2} q[a][i] * qq[d0+e-1-a][i+1+a]   (the e terms a<e touch qq on
//          diagonals >= d0 and are added when the cell is finished)
// partials: sh.part[(w*BAND+e)*T + tid], w = 0 (M), 1 (Q)
RP_HD int band_start_inside(int d) { return TURN + 1 + (d - TURN - 1) / BAND * BAND; }
RP_HD void inside_band_A(const Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const Split sp = make_split(C, T);
  const int cell = tid % sp.Cp, slice = tid / sp.Cp, S = sp.S;
  if (slice >= S || cell >= C) return;
  const int i = i0 + cell, ds = c.dstep();
  double m[BAND], q[BAND];
#pragma unroll
  for (int e = 0; e < BAND; e++) m[e] = q[e] = 0.;
  if (!(RP_DBG(c) & 2)) {
    const int amax = d0 - 1;                    // largest a any diagonal of the band needs
    const int lim = d0 - TURN - 2;              // term a belongs to diagonal d0+e iff a <= lim + e
    const int askip = c.cp > 0 ? c.cp - 1 - i : -1;  // split k = i+1+a on the nick (M only)
    const long es = ds;                         // per e: one diagonal up, same position
    // head of the q-split, a <= TURN: only e <= a is not "recent"
    for (int a = slice; a <= TURN && a <= amax; a += S) {
      const double A = TB(c, T_Q, a, i);
      const double* B = c.ptr(T_QQ, d0 - 1 - a, i + 1 + a);
      const int emin = a - lim;
#pragma unroll
      for (int e = 0; e < BAND; e++)
        if (e >= emin && e <= a) q[e] += A * B[e * es];
    }
    // main part, TURN < a <= lim: every diagonal of the band takes the term; both sums share the walk
    int a = TURN + 1 + slice;
    for (; a <= lim; a += S) {
      const double Am = (a == askip) ? 0. : TB(c, T_QM, a, i);
      const double Aq = TB(c, T_Q, a, i);
      const double* Bm = c.ptr(T_QM1, d0 - 1 - a, i + 1 + a);
      const double* Bq = c.ptr(T_QQ, d0 - 1 - a, i + 1 + a);
      double bm[BAND], bq[BAND];
#pragma unroll
      for (int e = 0; e < BAND; e++) { bm[e] = Bm[e * es]; bq[e] = Bq[e * es]; }
#pragma unroll
      for (int e = 0; e < BAND; e++) { m[e] += Am * bm[e]; q[e] += Aq * bq[e]; }
    }
    // tail, lim < a <= amax: the term only reaches the later diagonals of the band
    for (; a <= amax; a += S) {
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
#pragma unroll
  for (int e = 0; e < BAND; e++) {
    sh.part[(size_t)e * T + tid] = m[e];
    sh.part[(size_t)(BAND + e) * T + tid] = q[e];
  }
}
RP_HD void inside_band_B(Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const Split sp = make_split(C, T);
  for (int x = tid; x < BAND * C; x += T) {
    const int e = x / C, cell = x % C, i = i0 + cell;
    if (i + d0 + e > c.n) continue;
    double m = 0., q = 0.;
    for (int s = 0; s < sp.S; s++) {
      m += sh.part[(size_t)e * T + s * sp.Cp + cell];
      q += sh.part[(size_t)(BAND + e) * T + s * sp.Cp + cell];
    }
    TB(c, T_QM2, d0 + e, i) = m;
    TB(c, T_QS, d0 + e, i) = q;
  }
}
// per diagonal, phase A: interior-loop work items (pairable cell, slice), partials to sh.part[tid]
RP_HD void inside_A(const Ctx& c, const Shared& sh, int d, int i0, int C, int tid) {
  const int T = sh.T;
  if (d - (TURN + 1) < 2) return;
  const ISplit is = make_isplit(c, d, i0, C, T);
  const int r = tid % is.cntp, sl = tid / is.cntp;
  if (sl < is.SI && r < is.cnt) {
    const int i = listp(c)[(size_t)d * c.ld + is.lo + r];
    sh.part[tid] = inside_interior(c, sh, d, i, pair_type(base(c, i), base(c, i + d)), sl, is.SI);
  }
}
// per diagonal, phase B: one thread per cell
RP_HD void inside_B(Ctx& c, const Shared& sh, int d, int i0, int C, int tid) {
  const int T = sh.T;
  if (tid >= C) return;
  const int i = i0 + tid;
  double sI = 0.;
  const double sM = TB(c, T_QM2, d, i);
  double sQ = TB(c, T_QS, d, i);
  // the terms of the q-split that the band pass could not see yet: a < e, qq on diagonals >= d0
  const int e = d - band_start_inside(d);
  for (int a = 0; a < e && a <= d - TURN - 2; a++) sQ += TB(c, T_Q, a, i) * TB(c, T_QQ, d - 1 - a, i + 1 + a);
  const int type = pair_type(base(c, i), base(c, i + d));
  if (type && d - (TURN + 1) >= 2) {
    const ISplit is = make_isplit(c, d, i0, C, T);
    const int r = (int)posp(c)[(size_t)d * c.ld + i] - is.lo;
    for (int s = 0; s < is.SI; s++) sI += sh.part[s * is.cntp + r];
  }
  inside_finish(c, d, i, type, sI, sM, sQ);
}
// ---------------------------------------------------------------------------
// outside pass, diagonal d from n-1 down to TURN+1.
// out(k,l) = Z_outside(k,l)/Z  (ViennaRNA's probs[] before the final *qb).
// ---------------------------------------------------------------------------
// (Two strands: only the inter-strand cells are finished -- cross_lo / cross_hi -- and a cell that joins the strands
// never sits in the loop that holds the nick, so the outside pass needs no nick sums.)

// slice sl of SI of the interior-loop sum seen from the inner pair (k,l) (which can pair)
template <class C>
RP_HD double outside_interior(const C& c, const Shared& sh, int d, int k, int sl, int SI) {
  const DevModel& M = *c.M;
  const int n = c.n, l = k + d;
  const int ddmax = n - 1 - d < MAXLOOP + 2 ? n - 1 - d : MAXLOOP + 2;
  if (ddmax < 2) return 0.;
  // enclosing pair (i,j) = (k-1-u1, l+1+u2)
  int maxpo = k - 1, maxu2 = n - l - 1;
  if (c.cp > 0) {
    if (k >= c.cp && k - c.cp < maxpo) maxpo = k - c.cp;        // i must stay on k's strand
    if (l < c.cp && c.cp - 2 - l < maxu2) maxu2 = c.cp - 2 - l;  // j must stay on l's strand
  }
  if (maxpo < 1 || maxu2 < 0 || TB(c, T_QB, d, k) == 0.) return 0.;
  const int type = pair_type(base(c, k), base(c, l));
  const int t2 = rtype(type), sp1 = base(c, k - 1), sq1 = base(c, l + 1);
  int u1max = ddmax - 2 < MAXLOOP ? ddmax - 2 : MAXLOOP;
  if (maxpo - 1 < u1max) u1max = maxpo - 1;
  double sI = 0., s1 = 0., sA = 0.;
  if (!(RP_DBG(c) & 1))
    interior_rows<-1>(sh, c.ptr(T_OUTI, d, k), c.ptr(T_OUT1N, d, k), c.ptr(T_OUTAU, d, k), c.dstep(), c.pstep(), u1max,
                      maxu2, ddmax, sl, SI, sI, s1, sA);
  double accI = M.mmI[t2][sq1][sp1] * sI + M.mm1n[t2][sq1][sp1] * s1 + (type > 2 ? M.expTermAU : 1.0) * sA;
  for (int s = sl; s < RP_N_SPECIAL; s += SI) {
    int u1, u2;
    special_uv(s, u1, u2);
    const int dd = u1 + u2 + 2;
    if (dd > ddmax || u1 + 1 > maxpo || u2 > maxu2) continue;
    const int i = k - 1 - u1, j = l + 1 + u2;
    const int t1 = pair_type(base(c, i), base(c, j));
    if (!t1) continue;
    const double o = TB(c, T_OUT, d + dd, i);
    if (o == 0.) continue;
    accI += o * special_loop(M, s, t1, t2, base(c, i + 1), base(c, j - 1), sp1, sq1);
  }
  return accI;
}

// slice of the two multiloop sums of cell (k,l); `pairs` = the cell can pair
template <class C>
RP_HD void outside_splits(const C& c, int d, int k, bool pairs, int slice, int S, double& accP, double& accL) {
  const int ds = c.dstep(), ps = c.pstep(), n = c.n, l = k + d;
  accP = 0.; accL = 0.;
  if (RP_DBG(c) & 2) return;
  // PR(k,l) = sum_b Mc[d+2+b][k] * qm[b][l+1], b = TURN+1 .. n-l-2   [k is the closing 5' end]
  if (l + 2 <= n && ss(c, l, l + 1)) {
    const int cnt = n - l - 2 - TURN;
    if (cnt > 0) accP = strided_dot(c.ptr(T_MC, d + 3 + TURN, k), ds, c.ptr(T_QM, TURN + 1, l + 1), ds, cnt, slice, S, -1);
  }
  // ML-left(k,l) = sum_cc PRML[d+2+cc][k-2-cc] * qm[cc][k-1-cc], cc = TURN+1 .. k-3
  if (pairs && l < n && k > 2 && ss(c, k - 1, k) && ss(c, l, l + 1)) {
    const int cnt = k - 3 - TURN;
    if (cnt > 0 && TB(c, T_QB, d, k) != 0.)
      accL = strided_dot(c.ptr(T_PRML, d + 3 + TURN, k - 3 - TURN), ds - ps, c.ptr(T_QM, TURN + 1, k - 2 - TURN), ds - ps, cnt,
                         slice, S, -1);
  }
}

template <class C>
RP_HD void outside_finish(C& c, int d, int k, int type, double sI, double sP, double sL) {
  const DevModel& M = *c.M;
  const int l = k + d, n = c.n;
  const double scale2 = VEC(c, V_SCALE, 2);
  const bool mlr = l < n && ss(c, l, l + 1);  // something may follow l inside a multiloop
  // right side all unpaired: PL(k,l) = sum_{j>l} Mc(k,j) mlb^(j-l-1)
  const double PL = mlr ? TB(c, T_PL, d + 1, k) * M.mlb1 + TB(c, T_MC, d + 1, k) : 0.;
  const double PR = mlr ? sP : 0.;
  TB(c, T_PL, d, k) = PL;
  TB(c, T_PR, d, k) = PR;
  TB(c, T_PRML, d, k) = PR + PL;
  // left side all unpaired: PMLB(k,l) = sum_{i<k} PR(i,l) mlb^(k-1-i)
  double PMLB = 0.;
  if (k > 1 && ss(c, k - 1, k)) PMLB = TB(c, T_PMLB, d + 1, k - 1) * M.mlb1 + TB(c, T_PR, d + 1, k - 1);
  TB(c, T_PMLB, d, k) = PMLB;

  double out = 0.;
  if (type && TB(c, T_QB, d, k) != 0.) {
    const double q5 = k > 1 ? TB(c, T_Q, k - 2, 1) : 1.0;
    const double q3 = l < n ? TB(c, T_Q, n - l - 1, l + 1) : 1.0;
    out = q5 * q3 * c.invZ *
          ext_stem(M, type, (k > 1 && ss(c, k - 1, k)) ? base(c, k - 1) : -1, (l < n && ss(c, l, l + 1)) ? base(c, l + 1) : -1);
    out += sI;
    if (mlr && k > 1 && ss(c, k - 1, k)) out += (PMLB + sL) * ml_stem(M, type, base(c, k - 1), base(c, l + 1)) * scale2;
  }
  TB(c, T_OUT, d, k) = out;
  double fI = 0., f1 = 0., fA = 0., mc = 0.;
  if (out != 0.) {
    const int si1 = base(c, k + 1), sj1 = base(c, l - 1);
    fI = out * M.mmI[type][si1][sj1];
    f1 = out * M.mm1n[type][si1][sj1];
    fA = type > 2 ? out * M.expTermAU : out;
    if (ss(c, k, k + 1) && ss(c, l - 1, l)) mc = out * M.expMLclosing * ml_stem(M, rtype(type), sj1, si1);
  }
  TB(c, T_OUTI, d, k) = fI;
  TB(c, T_OUT1N, d, k) = f1;
  TB(c, T_OUTAU, d, k) = fA;
  TB(c, T_MC, d, k) = mc;
}

// General kernel, outside pass: the two multiloop sums are computed for a band of diagonals
// d0, d0-1, ..., d0-BAND+1 at once (all of their operands lie on diagonals > d0+1 or in the inside
// tables).  Item r serves row k = 1+r for PR and column l = d0-BAND+2+r for ML-left:
//   PR(k, k+d0-e)   = sum_{j} Mc(k,j) * qm(l+1, j-1),  j = l+2+TURN+1 .. n      share Mc(k,j)   over e
//   MLL(l-d0+e, l)  = sum_{i} PRML(i,l) * qm(i+1, k-1), i = 1 .. k-3-TURN        share PRML(i,l) over e
// partials: sh.part[(w*BAND+e)*T + tid], w = 0 (PR), 1 (MLL)
RP_HD void outside_band_A(const Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T;
  const Split sp = make_split(C, T);
  const int cell = tid % sp.Cp, slice = tid / sp.Cp, S = sp.S;
  if (slice >= S || cell >= C) return;
  const int r = r0 + cell, n = c.n, ds = c.dstep(), ps = c.pstep();
  double pr[BAND], ml[BAND];
#pragma unroll
  for (int e = 0; e < BAND; e++) pr[e] = ml[e] = 0.;
  if (!(RP_DBG(c) & 2)) {
    {  // PR, row k; t = j - (k+d0+TURN+3), valid for diagonal d0-e iff t >= -e
      const int k = 1 + r;
      const int tmax = n - k - d0 - (TURN + 3);
      int ecell = k + d0 - n;  // the cell (k, k+d0-e) exists iff e >= ecell
      if (ecell < 0) ecell = 0;
      const long es = ds - ps;  // per e one diagonal up, one cell left
      int t = -(BAND - 1) + slice;
      for (; t < 0 && t <= tmax; t += S) {  // head: the term only reaches the lower diagonals of the band
        const double A = TB(c, T_MC, d0 + TURN + 3 + t, k);
        const double* B = c.ptr(T_QM, TURN + 1 + t, k + d0 + 1);
        const int emin = -t > ecell ? -t : ecell;
#pragma unroll
        for (int e = 0; e < BAND; e++)
          if (e >= emin) pr[e] += A * B[e * es];
      }
      for (; t <= tmax; t += S) {           // main: every existing cell of the row takes the term
        const double A = TB(c, T_MC, d0 + TURN + 3 + t, k);
        const double* B = c.ptr(T_QM, TURN + 1 + t, k + d0 + 1);
        double bv[BAND];
#pragma unroll
        for (int e = 0; e < BAND; e++) bv[e] = B[e * es];
#pragma unroll
        for (int e = 0; e < BAND; e++)
          if (e >= ecell) pr[e] += A * bv[e];
      }
    }
    {  // ML-left, column l; cells (k0+e, l), k0 = l-d0; i <= k0+e-TURN-3
      const int l = d0 - BAND + 2 + r, k0 = l - d0;
      if (l <= n) {
        unsigned need = 0;
        for (int e = 0; e < BAND; e++) {
          const int k = k0 + e, d = d0 - e;
          if (k > 2 && d > TURN && pair_type(base(c, k), base(c, l)) && TB(c, T_QB, d, k) != 0.) need |= 1u << e;
        }
        if (need) {
          const int imax = k0 + (BAND - 1) - TURN - 3, imain = k0 - TURN - 3;
          int i = 1 + slice;
          for (; i <= imain; i += S) {       // main: every needed cell of the column takes the term
            const double A = TB(c, T_PRML, l - i, i);
            const double* B = c.ptr(T_QM, 0, i + 1) + (long)(k0 - 2 - i) * ds;
            double bv[BAND];
#pragma unroll
            for (int e = 0; e < BAND; e++) bv[e] = ((need >> e) & 1) ? B[(long)e * ds] : 0.;
#pragma unroll
            for (int e = 0; e < BAND; e++) ml[e] += A * bv[e];
          }
          for (; i <= imax; i += S) {        // tail: only the cells further right (larger k)
            const double A = TB(c, T_PRML, l - i, i);
            const double* B = c.ptr(T_QM, 0, i + 1) + (long)(k0 - 2 - i) * ds;  // e = 0 may lie below diagonal 0: not read then
            const int emin = i - k0 + TURN + 3;
#pragma unroll
            for (int e = 0; e < BAND; e++)
              if (e >= emin && ((need >> e) & 1)) ml[e] += A * B[(long)e * ds];
          }
        }
      }
    }
  }
#pragma unroll
  for (int e = 0; e < BAND; e++) {
    sh.part[(size_t)e * T + tid] = pr[e];
    sh.part[(size_t)(BAND + e) * T + tid] = ml[e];
  }
}
RP_HD void outside_band_B(Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T, n = c.n;
  const bool keep = c.kind == KIND_LINEAR && c.max_w > 0;
  const Split sp = make_split(C, T);
  for (int x = tid; x < BAND * C; x += T) {
    const int e = x / C, cell = x % C, r = r0 + cell, d = d0 - e;
    if (d < 1) continue;
    double a = 0., b = 0.;
    for (int s = 0; s < sp.S; s++) {
      a += sh.part[(size_t)e * T + s * sp.Cp + cell];
      b += sh.part[(size_t)(BAND + e) * T + s * sp.Cp + cell];
    }
    const int k = 1 + r;                       // PR cell (k, k+d)
    if (k + d <= n) {
      TB(c, T_PRB, d, k) = a;
      if (keep) RP_ST_STREAM(TB(c, T_XX, d, k), a);   // the unpaired-window pass reads PR again (unstru_windows)
    }
    const int l = d0 - BAND + 2 + r, k2 = l - d;  // MLL cell (l-d, l)
    if (l <= n && k2 >= 1) TB(c, T_MLB, d, k2) = b;
  }
}
// per diagonal, phase A: interior-loop items, partials to sh.part[tid]
RP_HD void outside_A(const Ctx& c, const Shared& sh, int d, int i0, int C, int tid) {
  const int T = sh.T;
  if (c.n - 1 - d < 2) return;
  const ISplit is = make_isplit(c, d, i0, C, T);
  const int r = tid % is.cntp, sl = tid / is.cntp;
  if (sl < is.SI && r < is.cnt) {
    const int k = listp(c)[(size_t)d * c.ld + is.lo + r];
    sh.part[tid] = outside_interior(c, sh, d, k, sl, is.SI);
  }
}
RP_HD void outside_B(Ctx& c, const Shared& sh, int d, int i0, int C, int tid) {
  const int T = sh.T;
  if (tid >= C) return;
  const int k = i0 + tid;
  double sI = 0.;
  const double sP = TB(c, T_PRB, d, k), sL = TB(c, T_MLB, d, k);
  const int type = pair_type(base(c, k), base(c, k + d));
  if (type && c.n - 1 - d >= 2 && TB(c, T_QB, d, k) != 0.) {
    const ISplit is = make_isplit(c, d, i0, C, T);
    const int r = (int)posp(c)[(size_t)d * c.ld + k] - is.lo;
    for (int s = 0; s < is.SI; s++) sI += sh.part[s * is.cntp + r];
  }
  outside_finish(c, d, k, type, sI, sP, sL);
}
// ---------------------------------------------------------------------------
// Wide bands (general kernel, long problems).  With BAND = TURN+2 diagonals per pass every operand of
// the split sums is final when the pass runs, but each pass streams the whole history of the tables
// for 5 FMAs per loaded element -- for long problems that stream comes from HBM.  A band of W > BAND
// diagonals reuses every loaded element W times.  The price: for the later diagonals of the band some
// operands lie on diagonals of the band itself.  The far pass (wide_*_A/B, below) leaves those terms
// out; inside_near / outside_near add them when the cell is finished (at most 2(W-BAND) per sum).
//   inside, band D0 .. D0+W-1, cell (i, i+D0+e):  term a (operands qm[a][i], qm1[D0+e-1-a][i+1+a]) is
//     far iff a <= D0-1 (first operand final) and a >= e (second operand final)
//   outside, band d0 .. d0-W+1, cell of diagonal d0-e: term b (operand Mc or PRML on diagonal d+2+b)
//     is far iff b >= e (diagonals >= d0+2 are final when the pass runs)
// ---------------------------------------------------------------------------
// prologue of the wide schedule: the row-major copy of qm vanishes on diagonals <= TURN like the table itself
RP_HD void prologue_rowmajor(const Ctx& c, int ct, int nct) {
  for (int x = ct; x < (TURN + 1) * c.n; x += nct) {
    const int d = x / c.n, i = 1 + x % c.n;
    if (i + d <= c.n) *c.rptr(T_QMR, i, i + d) = 0.;
  }
}
template <int W>
RP_HD int wide_start_inside(int d) { return TURN + 1 + (d - TURN - 1) / W * W; }
template <int W>
RP_HD int wide_start_outside(int n, int d) { return n - 1 - (n - 1 - d) / W * W; }
// rows one far-pass call takes with T threads: a warp of the shuffle variants owns 32-(W-1) rows
// (W = BAND: mcc_band_shfl.cuh, W > BAND: mcc_wide_shfl.cuh)
template <int W>
RP_HD int wide_chunk(int T) { return (32 - (W - 1)) * (T / 32); }

// host / reference form of the far pass (the CUDA build runs the shuffle variants of mcc_band_shfl.cuh)
template <int W>
RP_HD void wide_inside_A(const Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const Split sp = make_split(C, T);
  const int cell = tid % sp.Cp, slice = tid / sp.Cp, S = sp.S;
  if (slice >= S || cell >= C) return;
  const int i = i0 + cell;
  const long es = c.dstep();
  double m[W], q[W];
  for (int e = 0; e < W; e++) m[e] = q[e] = 0.;
  if (!(RP_DBG(c) & 2)) {
    const int amax = d0 - 1, lim = d0 - TURN - 2;
    const int askip = c.cp > 0 ? c.cp - 1 - i : -1;
    for (int a = slice; a <= amax; a += S) {
      const double Aq = TB(c, T_Q, a, i);
      const double Am = (a > TURN && a != askip) ? TB(c, T_QM, a, i) : 0.;
      const double* Bm = c.ptr(T_QM1, d0 - 1 - a, i + 1 + a);
      const double* Bq = c.ptr(T_QQ, d0 - 1 - a, i + 1 + a);
      for (int e = 0; e < W; e++)
        if (e >= a - lim && e <= a && i + d0 + e <= c.n) { m[e] += Am * Bm[e * es]; q[e] += Aq * Bq[e * es]; }
    }
  }
  for (int e = 0; e < W; e++) {
    sh.part[(size_t)e * T + tid] = m[e];
    sh.part[(size_t)(W + e) * T + tid] = q[e];
  }
}
template <int W>
RP_HD void wide_inside_B(Ctx& c, const Shared& sh, int d0, int i0, int C, int tid) {
  const int T = sh.T;
  const Split sp = make_split(C, T);
  for (int x = tid; x < W * C; x += T) {
    const int e = x / C, cell = x % C, i = i0 + cell;
    if (i + d0 + e > c.n) continue;
    double m = 0., q = 0.;
    for (int s = 0; s < sp.S; s++) {
      m += sh.part[(size_t)e * T + s * sp.Cp + cell];
      q += sh.part[(size_t)(W + e) * T + s * sp.Cp + cell];
    }
    TB(c, T_QM2, d0 + e, i) = m;
    TB(c, T_QS, d0 + e, i) = q;
  }
}
// the terms of cell (i, i+d) the far pass of its band could not see: a < e (second operand on a
// diagonal of the band) and a >= max(d0, e) (first operand on one).  All operands are loaded before
// the first product is formed: the loop is short (<= 2(W-BAND)+BAND terms) but every load is an L2 or
// HBM round trip, and this runs in the one-thread-per-cell finishing phase.
template <int W>
RP_HD void inside_near(const Ctx& c, int d, int i, double& sM, double& sQ) {
  const int d0 = wide_start_inside<W>(d), e = d - d0, hi = d - TURN - 2;
  const int askip = c.cp > 0 ? c.cp - 1 - i : -1;
  int n1 = (e - 1 < hi ? e - 1 : hi) + 1;                  // terms a = 0 .. n1-1
  if (n1 < 0) n1 = 0;
  const int a2 = d0 > e ? d0 : e;                          // terms a = a2 .. hi
  const int total = n1 + (hi >= a2 ? hi - a2 + 1 : 0);
  constexpr int CH = 5;   // operands of CH terms per round trip (4*CH doubles in registers)
#pragma unroll 1
  for (int x0 = 0; x0 < total; x0 += CH) {
    double aq[CH], bq[CH], am[CH], bm[CH];
#pragma unroll
    for (int u = 0; u < CH; u++) {
      const int x = x0 + u;
      const bool on = x < total;
      const int a = x < n1 ? x : a2 + (x - n1);
      const bool onm = on && a > TURN && a != askip;
      aq[u] = on ? TB(c, T_Q, a, i) : 0.;
      bq[u] = on ? TB(c, T_QQ, d - 1 - a, i + 1 + a) : 0.;
      am[u] = onm ? TB(c, T_QM, a, i) : 0.;
      bm[u] = onm ? TB(c, T_QM1, d - 1 - a, i + 1 + a) : 0.;
    }
#pragma unroll
    for (int u = 0; u < CH; u++) { sQ += aq[u] * bq[u]; sM += am[u] * bm[u]; }
  }
}

template <int W>
RP_HD void wide_outside_A(const Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T;
  const Split sp = make_split(C, T);
  const int cell = tid % sp.Cp, slice = tid / sp.Cp, S = sp.S;
  if (slice >= S || cell >= C) return;
  const int r = r0 + cell, n = c.n, ds = c.dstep(), ps = c.pstep();
  double pr[W], ml[W];
  for (int e = 0; e < W; e++) pr[e] = ml[e] = 0.;
  if (!(RP_DBG(c) & 2)) {
    {  // PR, row k; t = b - (TURN+1) - e: Mc on diagonal d0+TURN+3+t (final iff t >= -(TURN+1)), qm on diagonal TURN+1+t+e
      const int k = 1 + r;
      const int tmax = n - k - d0 - (TURN + 3);
      const long es = ds - ps;
      for (int t = -(TURN + 1) + slice; t <= tmax; t += S) {
        const double A = TB(c, T_MC, d0 + TURN + 3 + t, k);
        const double* B = c.ptr(T_QM, TURN + 1 + t, k + d0 + 1);
        for (int e = 0; e < W; e++)
          if (e >= -t && k + d0 - e <= n && d0 - e >= 1) pr[e] += A * B[e * es];
      }
    }
    {  // ML-left, column l; cells (k0+e, l), k0 = l-d0; term i: PRML(i,l) on diagonal l-i (final iff i <= k0-2)
      const int l = d0 - W + 2 + r, k0 = l - d0;
      if (l <= n) {
        unsigned need = 0;
        for (int e = 0; e < W; e++) {
          const int k = k0 + e, d = d0 - e;
          if (k > 2 && d > TURN && pair_type(base(c, k), base(c, l)) && TB(c, T_QB, d, k) != 0.) need |= 1u << e;
        }
        if (need) {
          const int ifar = k0 - 2;
          for (int i = 1 + slice; i <= ifar; i += S) {
            const double A = *c.rptr(T_PRMLR, i, l);
            const double* B = c.rptr(T_QMR, i + 1, k0 - 1);   // qm(i+1, k0-1+e)
            const int emin = i - k0 + TURN + 3;
            for (int e = 0; e < W; e++)
              if (e >= emin && ((need >> e) & 1)) ml[e] += A * B[e];
          }
        }
      }
    }
  }
  for (int e = 0; e < W; e++) {
    sh.part[(size_t)e * T + tid] = pr[e];
    sh.part[(size_t)(W + e) * T + tid] = ml[e];
  }
}
template <int W>
RP_HD void wide_outside_B(Ctx& c, const Shared& sh, int d0, int r0, int C, int tid) {
  const int T = sh.T, n = c.n;
  const Split sp = make_split(C, T);
  for (int x = tid; x < W * C; x += T) {
    const int e = x / C, cell = x % C, r = r0 + cell, d = d0 - e;
    if (d < 1) continue;
    double a = 0., b = 0.;
    for (int s = 0; s < sp.S; s++) {
      a += sh.part[(size_t)e * T + s * sp.Cp + cell];
      b += sh.part[(size_t)(W + e) * T + s * sp.Cp + cell];
    }
    const int k = 1 + r;                        // PR cell (k, k+d)
    if (k + d <= n) TB(c, T_PRB, d, k) = a;
    const int l = d0 - W + 2 + r, k2 = l - d;   // MLL cell (l-d, l)
    if (l <= n && k2 >= 1) TB(c, T_MLB, d, k2) = b;
  }
}
// per diagonal, phase B of the wide schedule: as inside_B, plus the near terms
// how generic_items deals a chunk of C cells out over the warps (the finishes read the partials back the same way)
struct GSplit {
  int NG, nb, wpb, cap;   // groups of 8 cells, blocks of 32 groups, warps (= bins) per block, cells per bin row
};
RP_HD GSplit make_gsplit(int C, int T) {
  GSplit g;
  g.NG = (C + 7) / 8;
  g.nb = (g.NG + 31) / 32;
  g.wpb = (T / 32) / g.nb;
  if (g.wpb < 1) g.wpb = 1;
  g.cap = g.nb * 256;
  return g;
}
RP_HD double generic_partials(const Shared& sh, int C, int cell) {
  const GSplit gs = make_gsplit(C, sh.T);
  double t = 0.;
  for (int b = 0; b < gs.wpb; b++) t += sh.gpart[(size_t)b * gs.cap + cell];
  return t;
}

// ---------------------------------------------------------------------------
// The rest of a staged chunk's interior sums: per pairable cell five items, each one batched strided walk
// (kind-major, so the lanes of a warp run the same walk for neighbouring cells):
//   0  bulges on the 5' side of the inner pair   u1 = 0, u2 = 2..      2  bulges on the 3' side      u2 = 0, u1 = 2..
//   1  1xn loops, single base 5'                 u1 = 1, u2 = 3..      3  1xn loops, single base 3'  u2 = 1, u1 = 2..
//   4  the table-driven small shapes
// Partial (kind, cell r) goes to sh.part[kind * cntp + r], closing factor included.
// ---------------------------------------------------------------------------
RP_HD double row_sum8(const double* g, const double* p, long step, int lo, int hi) {
  double a[8];
#pragma unroll
  for (int u = 0; u < 8; u++) a[u] = 0.;
  const double* q = p + (long)lo * step;
  g += lo;
  int cnt = hi - lo + 1;
#pragma unroll 1
  for (; cnt >= 8; cnt -= 8) {
    double v[8];
#pragma unroll
    for (int u = 0; u < 8; u++) v[u] = q[u * step];
#pragma unroll
    for (int u = 0; u < 8; u++) a[u] += g[u] * v[u];
    g += 8;
    q += 8 * step;
  }
  {
    double v[8];
#pragma unroll
    for (int u = 0; u < 7; u++) v[u] = u < cnt ? q[u * step] : 0.;
#pragma unroll
    for (int u = 0; u < 7; u++) a[u] += (u < cnt ? g[u] : 0.) * v[u];
  }
  return ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
}
// the four walks.  TA / T1 point at the cell's own entry of the bulge / 1xn class tables (see interior_rows for
// SIGN, the strides and the bounds).
template <int SIGN>
RP_HD double ends_walk(const Shared& sh, int kind, const double* TA, const double* T1, int ds, int ps, int u1max, int u2cap,
                       int ddmax) {
  const long step = -(long)SIGN * ds, across = -(long)SIGN * (ds - ps);
  const long o0 = -(long)SIGN * (2L * ds - ps);   // element (u1 = 0, u2 = 0); (u1, u2) at o0 + u1*across + u2*step
  if (u1max < 0 || u2cap < 0) return 0.;
  if (kind == 0) {
    int hi = MAXLOOP;
    if (u2cap < hi) hi = u2cap;
    if (ddmax - 2 < hi) hi = ddmax - 2;
    return hi >= 2 ? row_sum8(sh.grow, TA + o0, step, 2, hi) : 0.;
  }
  if (kind == 1) {
    if (u1max < 1) return 0.;
    int hi = MAXLOOP - 1;
    if (u2cap < hi) hi = u2cap;
    if (ddmax - 3 < hi) hi = ddmax - 3;
    return hi >= 3 ? row_sum8(sh.grow + GROW_LD, T1 + o0 + across, step, 3, hi) : 0.;
  }
  if (kind == 2) return u1max >= 2 ? row_sum8(sh.ghead_b, TA + o0, across, 2, u1max) : 0.;
  int hi = u1max;
  if (MAXLOOP - 1 < hi) hi = MAXLOOP - 1;
  if (ddmax - 3 < hi) hi = ddmax - 3;
  return (u2cap >= 1 && hi >= 2) ? row_sum8(sh.ghead_1, T1 + o0 + step, across, 2, hi) : 0.;
}
RP_HD double inside_ends_item(const Ctx& c, const Shared& sh, int d, int i, int kind) {
  const DevModel& M = *c.M;
  const int ddmax = d - (TURN + 1) < MAXLOOP + 2 ? d - (TURN + 1) : MAXLOOP + 2;
  if (ddmax < 2) return 0.;
  const int j = i + d, type = pair_type(base(c, i), base(c, j));
  const int maxpo = (c.cp > 0 && i < c.cp) ? c.cp - 1 - i : 1000;
  const int maxu2 = (c.cp > 0 && j >= c.cp) ? j - 1 - c.cp : 1000;
  const int si1 = base(c, i + 1), sj1 = base(c, j - 1);
  if (kind < 4) {
    int u1max = ddmax - 2 < MAXLOOP ? ddmax - 2 : MAXLOOP;
    if (maxpo - 1 < u1max) u1max = maxpo - 1;
    const double w = ends_walk<1>(sh, kind, c.ptr(T_QBAU, d, i), c.ptr(T_QB1N, d, i), c.dstep(), c.pstep(), u1max, maxu2, ddmax);
    return w * ((kind & 1) ? M.mm1n[type][si1][sj1] : (type > 2 ? M.expTermAU : 1.0));
  }
  // all nine inner pairs fetched before any is used
  double qv[RP_N_SPECIAL];
  int t2v[RP_N_SPECIAL];
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) {
    int u1, u2;
    special_uv(s, u1, u2);
    const int dd = u1 + u2 + 2;
    const bool ok = dd <= ddmax && u1 + 1 <= maxpo && u2 <= maxu2;
    const int k = i + 1 + u1, l = j - 1 - u2;
    t2v[s] = ok ? pair_type(base(c, k), base(c, l)) : 0;
    qv[s] = t2v[s] ? TB(c, T_QB, d - dd, k) : 0.;
  }
  double acc = 0.;
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) {
    if (!t2v[s]) continue;
    int u1, u2;
    special_uv(s, u1, u2);
    const int k = i + 1 + u1, l = j - 1 - u2;
    acc += qv[s] * special_loop(M, s, type, rtype(t2v[s]), si1, sj1, base(c, k - 1), base(c, l + 1));
  }
  return acc;
}
RP_HD double outside_ends_item(const Ctx& c, const Shared& sh, int d, int k, int kind) {
  const DevModel& M = *c.M;
  const int n = c.n, l = k + d;
  const int ddmax = n - 1 - d < MAXLOOP + 2 ? n - 1 - d : MAXLOOP + 2;
  if (ddmax < 2) return 0.;
  int maxpo = k - 1, maxu2 = n - l - 1;
  if (c.cp > 0) {
    if (k >= c.cp && k - c.cp < maxpo) maxpo = k - c.cp;
    if (l < c.cp && c.cp - 2 - l < maxu2) maxu2 = c.cp - 2 - l;
  }
  if (maxpo < 1 || maxu2 < 0 || TB(c, T_QB, d, k) == 0.) return 0.;
  const int type = pair_type(base(c, k), base(c, l));
  const int t2 = rtype(type), sp1 = base(c, k - 1), sq1 = base(c, l + 1);
  if (kind < 4) {
    int u1max = ddmax - 2 < MAXLOOP ? ddmax - 2 : MAXLOOP;
    if (maxpo - 1 < u1max) u1max = maxpo - 1;
    const double w = ends_walk<-1>(sh, kind, c.ptr(T_OUTAU, d, k), c.ptr(T_OUT1N, d, k), c.dstep(), c.pstep(), u1max, maxu2, ddmax);
    return w * ((kind & 1) ? M.mm1n[t2][sq1][sp1] : (type > 2 ? M.expTermAU : 1.0));
  }
  double ov[RP_N_SPECIAL];
  int t1v[RP_N_SPECIAL];
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) {
    int u1, u2;
    special_uv(s, u1, u2);
    const int dd = u1 + u2 + 2;
    const bool ok = dd <= ddmax && u1 + 1 <= maxpo && u2 <= maxu2;
    const int i = k - 1 - u1, j = l + 1 + u2;
    t1v[s] = ok ? pair_type(base(c, i), base(c, j)) : 0;
    ov[s] = t1v[s] ? TB(c, T_OUT, d + dd, i) : 0.;
  }
  double acc = 0.;
#pragma unroll
  for (int s = 0; s < RP_N_SPECIAL; s++) {
    if (!t1v[s] || ov[s] == 0.) continue;
    int u1, u2;
    special_uv(s, u1, u2);
    const int i = k - 1 - u1, j = l + 1 + u2;
    acc += ov[s] * special_loop(M, s, t1v[s], t2, base(c, i + 1), base(c, j - 1), sp1, sq1);
  }
  return acc;
}
template <int SIGN>
RP_HD void ends_items(const Ctx& c, const Shared& sh, int d, int i0, int C, int tid) {
  const int T = sh.T;
  if ((SIGN > 0 ? d - (TURN + 1) : c.n - 1 - d) < 2) return;
  const ISplit is = make_isplit(c, d, i0, C, T);
  const uint16_t* L = listp(c) + (size_t)d * c.ld + is.lo;
  for (int x = tid; x < GS_KINDS * is.cntp; x += T) {
    const int kind = x / is.cntp, r = x - kind * is.cntp;
    if (r >= is.cnt) continue;
    sh.part[x] = SIGN > 0 ? inside_ends_item(c, sh, d, L[r], kind) : outside_ends_item(c, sh, d, L[r], kind);
  }
}

template <int W>
RP_HD void wide_inside_finish(Ctx& c, const Shared& sh, int d, int i0, int C, int tid, bool staged = false) {
  const int T = sh.T;
  if (tid >= C) return;
  const int i = i0 + tid;
  double sI = 0.;
  double sM = TB(c, T_QM2, d, i), sQ = TB(c, T_QS, d, i);
  inside_near<W>(c, d, i, sM, sQ);
  const int type = pair_type(base(c, i), base(c, i + d));
  if (type && d - (TURN + 1) >= 2) {
    const ISplit is = make_isplit(c, d, i0, C, T);
    const int r = (int)posp(c)[(size_t)d * c.ld + i] - is.lo;
    const int NS = staged ? GS_KINDS : is.SI;
    for (int s = 0; s < NS; s++) sI += sh.part[s * is.cntp + r];
    if (staged)   // the generic-class taps, summed densely out of the staged tile (generic_items)
      sI += c.M->mmI[type][base(c, i + 1)][base(c, i + d - 1)] * generic_partials(sh, C, i - i0);
  }
  TB(c, T_QM2, d, i) = sM;   // complete now: the closing sum of (i-1,i+d+1) and the unpaired-window pass read it
  inside_finish(c, d, i, type, sI, sM, sQ);
  *c.rptr(T_QMR, i, i + d) = TB(c, T_QM, d, i);
}
// near terms of cell (k, k+d): Mc / PRML on diagonals d+2+b < d0+2, i.e. b < e = d0-d
template <int W>
RP_HD void outside_near(const Ctx& c, int d, int k, bool pairs, double& sP, double& sL) {
  const int n = c.n, l = k + d, d0 = wide_start_outside<W>(n, d), e = d0 - d;
  for (int b = TURN + 1; b < e && b <= n - l - 2; b++) sP += TB(c, T_MC, d + 2 + b, k) * TB(c, T_QM, b, l + 1);
  if (pairs)
    for (int cc = TURN + 1; cc < e && cc <= k - 3; cc++) sL += TB(c, T_PRML, d + 2 + cc, k - 2 - cc) * TB(c, T_QM, cc, k - 1 - cc);
}
template <int W>
RP_HD void wide_outside_finish(Ctx& c, const Shared& sh, int d, int i0, int C, int tid, bool staged = false) {
  const int T = sh.T;
  if (tid >= C) return;
  const int k = i0 + tid, l = k + d;
  double sI = 0.;
  double sP = TB(c, T_PRB, d, k), sL = TB(c, T_MLB, d, k);
  const int type = pair_type(base(c, k), base(c, l));
  const bool pairs = type && TB(c, T_QB, d, k) != 0.;
  outside_near<W>(c, d, k, pairs && k > 2 && l < c.n, sP, sL);
  if (pairs && c.n - 1 - d >= 2) {
    const ISplit is = make_isplit(c, d, i0, C, T);
    const int r = (int)posp(c)[(size_t)d * c.ld + k] - is.lo;
    const int NS = staged ? GS_KINDS : is.SI;
    for (int s = 0; s < NS; s++) sI += sh.part[s * is.cntp + r];
    if (staged && k > 1 && l < c.n)
      sI += c.M->mmI[rtype(type)][base(c, l + 1)][base(c, k - 1)] * generic_partials(sh, C, k - i0);
  }
  if (c.kind == KIND_LINEAR && c.max_w > 0) RP_ST_STREAM(TB(c, T_XX, d, k), sP);   // PR for the unpaired-window pass
  outside_finish(c, d, k, type, sI, sP, sL);
  *c.rptr(T_PRMLR, k, l) = TB(c, T_PRML, d, k);
}

// ---------------------------------------------------------------------------
// Staged generic interior sums (see the note at struct Shared).  Chunk = cells i0 .. i0+C-1 of diagonal d (one strand
// segment: `crossing` says the cells join the strands, which confines their inner pairs to inter-strand cells too).
// Tile row s (6 <= s <= smax) holds the class row of diagonal d -/+ (2+s) from position P(s) on, P(s) = i0+1 inside,
// i0-1-s outside; element e of a row at ((e & 7) * LT/8 + (e >> 3)), so that the 32 lanes of a warp, which own 32
// consecutive groups of 8 cells, read 32 consecutive doubles.  Cell r of group g, tap t reads element 8g + r + t.
// ---------------------------------------------------------------------------
RP_HD int gs_smax(int n, int d, int SIGN) {
  const int m = SIGN > 0 ? d - 6 : n - 3 - d;
  return m < MAXLOOP ? m : MAXLOOP;
}
template <int SIGN>
RP_HD void stage_generic_tile(const Ctx& c, const Shared& sh, int d, int i0, int C, bool crossing, int tid) {
  const int T = sh.T, n = c.n, LT = gs_lt(T), L8 = LT / 8;
  const int smax = gs_smax(n, d, SIGN);
  const int nrows = smax - GS_ROW0 + 1;
  if (nrows <= 0) return;
  const int len = ((C + 7) & ~7) + MAXLOOP + 8;   // elements any group of the chunk can reach (<= LT)
  // a warp takes (row, NL interleaved segments of 32 elements) items: consecutive lanes load consecutive positions
  constexpr int NL = 8;                            // loads in flight per thread
  const int nblk = (len + 32 * NL - 1) / (32 * NL);
  const int warp = tid >> 5, lane = tid & 31, nwarp = T >> 5;
  for (int it = warp; it < nrows * nblk; it += nwarp) {
    const int row = it / nblk, blk = it - row * nblk, sdiag = GS_ROW0 + row;
    const int dr = d - SIGN * (2 + sdiag);
    const int pos0 = (SIGN > 0 ? i0 + 1 : i0 - 1 - sdiag);
    int plo = 1, phi = n - dr;
    if (crossing) { if (c.cp - dr > plo) plo = c.cp - dr; if (c.cp - 1 < phi) phi = c.cp - 1; }
    const double* src = c.ptr(SIGN > 0 ? T_QBI : T_OUTI, dr, 0);
    double* dstrow = sh.gtile + (size_t)row * LT;
    double v[NL];
#pragma unroll
    for (int u = 0; u < NL; u++) {
      const int e = (u * nblk + blk) * 32 + lane, pos = pos0 + e;
      v[u] = (e < len && pos >= plo && pos <= phi) ? src[pos] : 0.;
    }
#pragma unroll
    for (int u = 0; u < NL; u++) {
      const int e = (u * nblk + blk) * 32 + lane;
      if (e < len) dstrow[(e & 7) * L8 + (e >> 3)] = v[u];
    }
  }
}
// one warp: the rows of its bin for the 32 groups of its block; lane = group; partial sums to gpart[bin][cell]
template <int SIGN>
RP_HD void generic_items(const Ctx& c, const Shared& sh, int d, int i0, int C, int tid) {
  const int T = sh.T, LT = gs_lt(T), L8 = LT / 8;
  const GSplit gs = make_gsplit(C, T);
  const int warp = tid >> 5, lane = tid & 31;
  const int blk = warp / gs.wpb, bin = warp - blk * gs.wpb;
  if (blk >= gs.nb) return;
  const int g = blk * 32 + lane;
  const int smax = gs_smax(c.n, d, SIGN), nrows = smax - GS_ROW0 + 1;
  double tot[8];
#pragma unroll
  for (int r = 0; r < 8; r++) tot[r] = 0.;
  if (g < gs.NG) {
    // rows dealt out long / short alternately, so that every bin gets about the same number of taps
    for (int idx = bin; idx < nrows; idx += gs.wpb) {
      const int s = (idx & 1) ? GS_ROW0 + (idx >> 1) : smax - (idx >> 1);
      const double* row = sh.gtile + (size_t)(s - GS_ROW0) * LT + g;   // element 8g + c at row[(c & 7) * L8 + (c >> 3)]
#define RP_GX(cc) (((cc) & 7) * L8 + ((cc) >> 3))
      double win[8];
#pragma unroll
      for (int r = 0; r < 7; r++) win[r] = row[RP_GX(2 + r)];
      win[7] = 0.;
      const int nst = s - 3;   // taps t = 2 .. s-2; step x loads element 9 + x, weight g(2+x, s-2-x)
      int x = 0;
#pragma unroll 1
      for (; x + 8 <= nst; x += 8) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
          win[(u + 7) & 7] = row[RP_GX(9 + u) + (x >> 3)];
          const double gv = sh.grow[(2 + x + u) * GROW_LD + (s - 2 - x - u)];
#pragma unroll
          for (int r = 0; r < 8; r++) tot[r] += gv * win[(u + r) & 7];
        }
      }
#pragma unroll
      for (int u = 0; u < 7; u++) {
        if (x + u < nst) {
          win[(u + 7) & 7] = row[RP_GX(9 + u) + (x >> 3)];
          const double gv = sh.grow[(2 + x + u) * GROW_LD + (s - 2 - x - u)];
#pragma unroll
          for (int r = 0; r < 8; r++) tot[r] += gv * win[(u + r) & 7];
        }
      }
#undef RP_GX
    }
  }
#pragma unroll
  for (int r = 0; r < 8; r++)
    if (8 * g + r < gs.cap) sh.gpart[(size_t)bin * gs.cap + 8 * g + r] = tot[r];
}

// ---------------------------------------------------------------------------
// unpaired windows (single strand): up(i,d) = P(i..i+d unpaired), d < max_w
// ---------------------------------------------------------------------------
// U1: DG(p,o) = out(p,o)*hairpin(p,o)   (loop whose unpaired run is (p,o))
template <class C>
RP_HD void unstru_hairpin(C& c, int tid, int T) {
  const int n = c.n;
  const unsigned total = (unsigned)n * (unsigned)c.ld, ld = (unsigned)c.ld;   // n <= RP_MAX_N: 32-bit index arithmetic
  for (unsigned x = tid; x < total; x += T) {
    const int d = (int)(x / ld), i = (int)(x - (unsigned)d * ld);
    if (i < 1 || i + d > n) continue;
    double v = 0.;
    if (d > TURN) {
      const double o = TB(c, T_OUT, d, i);
      if (o != 0.) v = o * hairpin(c, i, i + d, pair_type(base(c, i), base(c, i + d)));
    }
    TB(c, T_DG, d, i) = v;
  }
}
// class of the loop shape (u1,u2), u1+u2 <= MAXLOOP: the rule of build_dev_model (dev_model.cpp), in registers
RP_HD int loop_class(int u1, int u2) {
  const int ul = u1 > u2 ? u1 : u2, us = u1 > u2 ? u2 : u1;
  if (us == 0) return ul >= 2 ? CLS_BULGE : CLS_SPECIAL;
  if (us == 1) return ul >= 3 ? CLS_1N : CLS_SPECIAL;
  return (us == 2 && (ul == 2 || ul == 3)) ? CLS_SPECIAL : CLS_GENERIC;
}

// The table-driven shapes (9 small loops, dev_model.h) of the gap sums: item (side, gap size
// ug <= 3, gap start a, slice) sums the loops of all special shapes with that gap size over
// every `nsl`-th position of the free pair end and leaves the partial in a scratch row of T_RR
// (free until unstru_ml_tables): row (side*3+ug-1)*nsl+slice, position a.  unstru_gaps adds the
// slices up in fixed order.  Branch-free body: cells that cannot pair carry qb = out = 0.
RP_HD int gap_special_slices(int n) { return n >= 48 ? 4 : 1; }
template <class C, class MT>
RP_HD void unstru_gap_specials(C& c, const MT& M, int tid, int T) {
  const int n = c.n;
  if (n < 7) return;   // rows 0..5 of the scratch must exist; shorter sequences have no such loops to speak of (handled below)
  const int nsl = gap_special_slices(n);
  const int items = (RP_DBG(c) & 4) ? 0 : 2 * 3 * nsl * n;
  for (int x = tid; x < items; x += T) {
    const int a = x % n + 1;
    int y = x / n;
    const int sl = y % nsl; y /= nsl;
    const int ug = y % 3 + 1, side = y / 3;
    const int b = a + ug + 1;
    double acc = 0.;
    if (b <= n) {
      if (side == 0) {
        const int p = a, k = b, u1 = ug, lmin = k + TURN + 1;
        const int sp1 = base(c, k - 1), si1 = base(c, p + 1);
        for (int u2 = 0; u2 <= 3; u2++) {
          if (loop_class(u1, u2) != CLS_SPECIAL) continue;
          const int lmax = n - 1 - u2, sidx = special_index(u1, u2);
          // four positions per round trip: the eight table loads go out before the first weight is looked up
          for (int l0 = lmin + sl; l0 <= lmax; l0 += 4 * nsl) {
            double qb[4], ou[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int l = l0 + u * nsl;
              const bool on = l <= lmax;
              qb[u] = on ? TB(c, T_QB, l - k, k) : 0.;
              ou[u] = on ? TB(c, T_OUT, l + 1 + u2 - p, p) : 0.;
            }
            double w[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {   // branch-free: the four weight look-ups (L2) are in flight together
              const int l = l0 + u * nsl <= lmax ? l0 + u * nsl : lmax, o = l + 1 + u2;
              w[u] = special_loop(M, sidx, pair_type(base(c, p), base(c, o)), rtype(pair_type(base(c, k), base(c, l))),
                                  si1, base(c, o - 1), sp1, base(c, l + 1));
            }
#pragma unroll
            for (int u = 0; u < 4; u++) acc += ou[u] * qb[u] * w[u];
          }
        }
      } else {
        const int l = a, o = b, u2 = ug;
        const int sq1 = base(c, l + 1), sj1 = base(c, o - 1);
        for (int u1 = 0; u1 <= 3; u1++) {
          if (loop_class(u1, u2) != CLS_SPECIAL) continue;
          const int pmax = l - TURN - 2 - u1, sidx = special_index(u1, u2);
          for (int p0 = 1 + sl; p0 <= pmax; p0 += 4 * nsl) {
            double qb[4], ou[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int p = p0 + u * nsl;
              const bool on = p <= pmax;
              ou[u] = on ? TB(c, T_OUT, o - p, p) : 0.;
              qb[u] = on ? TB(c, T_QB, l - (p + 1 + u1), p + 1 + u1) : 0.;
            }
            double w[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const int p = p0 + u * nsl <= pmax ? p0 + u * nsl : pmax, k = p + 1 + u1;
              w[u] = special_loop(M, sidx, pair_type(base(c, p), base(c, o)), rtype(pair_type(base(c, k), base(c, l))),
                                  base(c, p + 1), sj1, base(c, k - 1), sq1);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) acc += ou[u] * qb[u] * w[u];
          }
        }
      }
    }
    TB(c, T_RR, ((side * 3 + ug - 1) * nsl + sl), a) = acc;
  }
}

// U2 (side=0): DG(p,k) += weight of all interior loops closed by some (p,o) with inner pair (k,l): 5' gap (p,k)
// U3 (side=1): DG(l,o) += the same loops seen from their 3' gap (l,o)
// One item per gap.  For the factorised classes the sum over the free pair end is a dot
// product of two table rows that already carry the pair factors:
//   side 0:  sum_l  outX(p, l+1+u2) * qbX(k, l)          (both advance one diagonal per l)
//   side 1:  sum_p  outX(p, o)      * qbX(p+1+u1, l)     (both step one diagonal down, one cell right)
// Runs of up to 8 shifts of one class share the streamed operand (multi_dot).
// gfull: the weights g(u1,u2) incl. scale, row stride GROW_LD (DevModel::gfull, or a shared-memory copy)
template <class C>
RP_HD void unstru_gaps(C& c, const double* gfull, int side, int tid, int T) {
  const int n = c.n, ds = c.dstep(), ps = c.pstep();
  const int items = (RP_DBG(c) & 4) ? 0 : n * (MAXLOOP + 1);
  const int tabO[3] = {T_OUTI, T_OUT1N, T_OUTAU};
  const int tabQ[3] = {T_QBI, T_QB1N, T_QBAU};
  for (int x = tid; x < items; x += T) {
    const int ug = x / n;      // size of the gap this item owns
    const int a = x % n + 1;   // gap is the open interval (a, a+ug+1)
    const int b = a + ug + 1;
    if (b > n || ug < 1) continue;  // an empty gap cannot contain a window
    double acc = 0.;
    if (side == 0) {
      const int p = a, k = b, u1 = ug;
      const int lmin = k + TURN + 1;
      for (int u2 = 0; u1 + u2 <= MAXLOOP;) {
        if (n - 1 - u2 < lmin) break;
        const int cls = loop_class(u1, u2);
        if (cls != CLS_SPECIAL) {
          // run of up to 8 consecutive u2 of the same class
          int nu = 1;
          while (nu < 8 && u1 + u2 + nu <= MAXLOOP && loop_class(u1, u2 + nu) == cls && n - 1 - (u2 + nu) >= lmin) nu++;
          double av[8] = {0., 0., 0., 0., 0., 0., 0., 0.};
          const double* Q = c.ptr(tabQ[cls], lmin - k, k);           // qbX(k,l), one diagonal per l
          const double* O = c.ptr(tabO[cls], lmin + 1 + u2 - p, p);  // outX(p,l+1+u2), one diagonal per u2
          const int cmain = n - 1 - (u2 + nu - 1) - lmin + 1;        // l range valid for every u2 of the run
          // the shorter shifts reach further (l up to n-1-(u2+t)): walk to the end of the longest one;
          // window elements past the last diagonal count as 0
          const int X = cmain + nu - 1;
          if (nu == 1) av[0] = dot_range(Q, ds, O, ds, 0, X, 0, 1);   // a lone shift (the bulge / 1xn heads): plain dot product
          else multi_dot_slide(Q, ds, O, ds, X, 0, X - 1, av);
          for (int t = 0; t < nu; t++) acc += gfull[u1 * GROW_LD + u2 + t] * av[t];
          u2 += nu;
        } else {
          u2++;  // table-driven shapes: summed by unstru_gap_specials into the scratch rows
        }
      }
    } else {
      const int l = a, o = b, u2 = ug;
      for (int u1 = 0; u1 + u2 <= MAXLOOP;) {
        if (l - TURN - 2 - u1 < 1) break;  // k = p+1+u1 <= l-TURN-1 needs p >= 1
        const int cls = loop_class(u1, u2);
        if (cls != CLS_SPECIAL) {
          int nu = 1;
          while (nu < 8 && u1 + nu + u2 <= MAXLOOP && loop_class(u1 + nu, u2) == cls && l - TURN - 2 - (u1 + nu) >= 1) nu++;
          double av[8] = {0., 0., 0., 0., 0., 0., 0., 0.};
          const double* O = c.ptr(tabO[cls], o - 1, 1);               // outX(p,o): one diagonal down, one cell right per p
          const double* Q = c.ptr(tabQ[cls], l - 2 - u1, 2 + u1);     // qbX(p+1+u1,l); per u1 likewise
          const int cmain = l - TURN - 2 - (u1 + nu - 1);             // p = 1..cmain valid for every u1 of the run
          // walked from the largest p downwards: then the lanes of a warp (consecutive gaps) read
          // consecutive addresses.  Reversed window: element z holds Q[X+6-z], shift t' = 7-t.
          if (cmain > 0) {
            const long st = ps - ds;
            const int X = cmain + nu - 1;   // steps of the longest shift (t = 0)
            if (nu == 1) {
              av[0] = dot_range(O + (long)(X - 1) * st, (int)-st, Q + (long)(X - 1) * st, (int)-st, 0, X, 0, 1);
            } else {
              double rv[8] = {0., 0., 0., 0., 0., 0., 0., 0.};
              multi_dot_slide(O + (long)(X - 1) * st, -st, Q + (long)(X + 6) * st, -st, X, 7, X + 6, rv);
#pragma unroll
              for (int t = 0; t < 8; t++) av[t] = rv[7 - t];
            }
          }
          for (int t = 0; t < nu; t++) acc += gfull[(u1 + t) * GROW_LD + u2] * av[t];
          u1 += nu;
        } else {
          u1++;
        }
      }
    }
    if (ug <= 3 && n >= 7) {
      const int nsl = gap_special_slices(n);
      for (int sl = 0; sl < nsl; sl++) acc += TB(c, T_RR, ((side * 3 + ug - 1) * nsl + sl), a);
    }
    TB(c, T_DG, b - a, a) += acc;
  }
}
// U4a: suffix sums over b for each a ; U4b: prefix sums over a for each b
template <class C>
RP_HD void unstru_dom_rows(C& c, int tid, int T) {
  const int n = c.n;
  for (int a = 1 + tid; a <= n; a += T) {
    double s = 0.;
    for (int b = n; b > a; b--) {
      s += TB(c, T_DG, b - a, a);
      TB(c, T_DG, b - a, a) = s;
    }
  }
}
template <class C>
RP_HD void unstru_dom_cols(C& c, int tid, int T) {
  const int n = c.n;
  for (int b = 2 + tid; b <= n; b += T) {
    double s = 0.;
    for (int a = 1; a < b; a++) {
      s += TB(c, T_DG, b - a, a);
      TB(c, T_DG, b - a, a) = s;
    }
  }
}
// U5/U6: the multiloop part of the unpaired-window probabilities.  The window [i..j] (dd = j-i) lies in
// the loop closed by (p,o), p < i, j < o, next to the closing pair's unpaired run or between stems:
//   m1 = sum_{p<i} mlb^(j-p)  sum_{o>=j+2} Mc(p,o) QM2(j+1,o-1)           window in the 5' run, >= 2 stems follow
//   m2 = sum_{o>j} mlb^(o-i)  sum_{p<=i-2} Mc(p,o) QM2(p+1,i-1)           window in the 3' run, >= 2 stems before
//   m3 = mlb^(dd+1) sum_{p,o} qm(p+1,i-1) Mc(p,o) qm(j+1,o-1)             stems on both sides
// Summed in this order the inner sums are O(n) per CELL (O(n^3) in all, as in ViennaRNA's pf_unstru).
// Exchanging the sums leaves O(n) per WINDOW (n*max_w windows):
//   m1 = mlb^dd     sum_o QM2(j+1,o-1) K(i,o),     K(i,o)  = sum_{p<i} Mc(p,o) mlb^(i-p)     column scan of Mc
//   m2 = mlb^(dd+1) sum_p QM2(p+1,i-1) PLf(p,j),   PLf(p,j) = sum_{o>j} Mc(p,o) mlb^(o-j-1)  row scan of Mc
//   m3 = mlb^(dd+1) sum_p qm(p+1,i-1)  PR(p,j),    PR(p,j)  = sum_o Mc(p,o) qm(j+1,o-1)
// and PR is the outside pass's own right-hand multiloop sum, which the band phases leave in T_XX for
// single-strand problems with windows.  Tables: K -> T_RR, PLf -> T_LL.
template <class C>
RP_HD void unstru_ml_tables(C& c, int tid, int T) {
  const int n = c.n;
  const double mlb1 = c.M->mlb1;
  // both scans walk the diagonals downwards, every thread on the same diagonal at the same step, so
  // that the threads of a warp touch consecutive elements
  for (int p0 = 1; p0 < n; p0 += T) {          // row p: PLf(p,j), j = n .. p+1
    const int p = p0 + tid;
    double s = 0.;
#pragma unroll 8
    for (int d = n - p0; d >= 1; d--) {
      if (d > n - p) continue;
      const double mc = TB(c, T_MC, d, p);
      TB(c, T_LL, d, p) = s;
      s = s * mlb1 + mc;
    }
  }
  for (int o0 = 2; o0 <= n; o0 += T) {         // column o: K(i,o), i = 1 .. o-1
    const int o = o0 + tid, top = (o0 + T - 1 < n ? o0 + T - 1 : n) - 1;
    double s = 0.;
#pragma unroll 8
    for (int d = top; d >= 1; d--) {
      if (o > n || d > o - 1) continue;
      const double mc = TB(c, T_MC, d, o - d);
      TB(c, T_RR, d, o - d) = s;
      s = mlb1 * (s + mc);
    }
  }
}
// U6: assemble; writes fp32 in the reference layout up[(i-1)*max_w + d].  Consecutive threads take
// consecutive i of the same window length: every operand stream is unit-stride across the warp.
template <class C>
RP_HD void unstru_windows(C& c, float* up, int tid, int T) {
  const int n = c.n, w = c.max_w;
  for (int x = tid; x < n * w; x += T) {
    const int dd = x / n, i = x % n + 1, j = i + dd;
    double v = 0.;
    if (j <= n) {
      const double q5 = i > 1 ? TB(c, T_Q, i - 2, 1) : 1.0;
      const double q3 = j < n ? TB(c, T_Q, n - j - 1, j + 1) : 1.0;
      v = q5 * VEC(c, V_SCALE, dd + 1) * q3 * c.invZ;
      if (i > 1 && j < n) {
        v += TB(c, T_DG, j - i + 2, i - 1);
        double m1 = 0., m2 = 0., m3 = 0.;
        {
          const double* A = c.ptr(T_QM2, 2 * TURN + 3, j + 1);
          const double* B = c.ptr(T_RR, dd + 2 * TURN + 5, i);
          const int cnt = n - j - 2 - (2 * TURN + 3) + 1, ds = c.dstep();
#pragma unroll 4
          for (int t = 0; t < cnt; t++) m1 += A[(long)t * ds] * B[(long)t * ds];
        }
        {
          const int cnt = i - 3 - TURN, st = c.dstep() - c.pstep();   // cc = TURN+1+t: one diagonal up, one cell left
          const double* A2 = c.ptr(T_QM2, TURN + 1, i - 2 - TURN);
          const double* A1 = c.ptr(T_QM, TURN + 1, i - 2 - TURN);
          const double* BL = c.ptr(T_LL, dd + TURN + 3, i - 3 - TURN);
          const double* BR = c.ptr(T_XX, dd + TURN + 3, i - 3 - TURN);
#pragma unroll 4
          for (int t = 0; t < cnt; t++) {
            m2 += A2[(long)t * st] * BL[(long)t * st];
            m3 += A1[(long)t * st] * BR[(long)t * st];
          }
        }
        // Mc carries no scale factor for the closing pair's two bases: apply it here
        v += (m1 * VEC(c, V_MLB, dd) + (m2 + m3) * VEC(c, V_MLB, dd + 1)) * VEC(c, V_SCALE, 2);
      }
    }
    RP_ST_STREAM(up[(size_t)(i - 1) * w + dd], (float)v);
  }
}

// ---------------------------------------------------------------------------
// outputs in the reference's layouts
// ---------------------------------------------------------------------------
// bp[offset[i]+j] = (float) pr(i,j), offset[i] = i*(2L+1-i)/2   (src/ractip.cpp:314-317,365-367)
template <class C>
RP_HD void write_bp(const C& c, float* bp, int tid, int T) {
  const int L = c.n;
  const size_t total = (size_t)(L + 1) * (L + 2) / 2;
  for (size_t x = tid; x < total; x += T) RP_ST_STREAM(bp[x], 0.f);
}
template <class C>
RP_HD void write_bp2(const C& c, float* bp, int tid, int T) {
  const int L = c.n;
  const unsigned total = (unsigned)L * (unsigned)c.ld, ld = (unsigned)c.ld;
  for (unsigned x = tid; x < total; x += T) {
    const int d = (int)(x / ld), i = (int)(x - (unsigned)d * ld);
    if (i < 1 || i + d > L || d < 1) continue;
    const double p = d > TURN ? TB(c, T_OUT, d, i) * TB(c, T_QB, d, i) : 0.;
    RP_ST_STREAM(bp[(size_t)i * (2 * L + 1 - i) / 2 + (i + d)], (float)p);
  }
}
// hp[i][j-cp+1] = p if i<cp<=j and p>th_hy (float compare)   (src/ractip.cpp:404-405,447-453)
template <class C>
RP_HD void write_hp(const C& c, float* hp, int n1, int n2, float th_hy, int tid, int T) {
  const int cp = c.cp;
  const int total = (n1 + 1) * (n2 + 1);
  for (int x = tid; x < total; x += T) {
    const int i = x / (n2 + 1), jj = x % (n2 + 1);
    float v = 0.f;
    if (i >= 1 && jj >= 1) {
      const int j = jj + cp - 1, d = j - i;
      if (d > TURN) {
        const double p = TB(c, T_OUT, d, i) * TB(c, T_QB, d, i);
        const float pf = (float)p;
        if (p >= (double)th_hy && pf > th_hy) v = pf;
      }
    }
    RP_ST_STREAM(hp[x], v);
  }
}

}  // namespace rp
#endif
