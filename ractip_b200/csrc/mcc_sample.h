// mcc_sample.h -- stochastic sampling of secondary structures (RNAfold -p --stochBT) from the inside tables the general
// kernel leaves in a problem's workspace slot: structures drawn with probability exp(-E/kT) / Z of exactly the ensemble
// whose log Z the kernel reports (constraint keys, stacking factors and unpaired pseudo-energies included).  A phase of its own between the
// inside and the outside pass (mcc_driver.h, emit_samples).
//
// Traceback.  A sample is a stack of pending SEGMENTS, each one term of the inside recursion:
//   SG_Q   (i,j)  q(i,j):   the exterior-like region i..j (d = j-i > TURN; shorter ones are all unpaired)
//   SG_QQ  (k,j)  qq(k,j):  k pairs with some l <= j, l+1..j unpaired
//   SG_QB  (i,j)  qb(i,j):  (i,j) pairs
//   SG_QM  (p,r)  qm(p,r):  at least one multiloop stem in p..r
//   SG_QM1 (k,r)  qm1(k,r): k pairs with some l <= r, l+1..r unpaired (multiloop)
//   SG_QM2 (p,r)  QM2(p,r): the inside of a multiloop, two or more stems
// The top segment is popped and decided: its candidates are enumerated in a fixed order (sample_count / sample_weight,
// below), each with the weight the inside recursion gives that term -- the kernel's own factors, so that sampling from
// the kernel's tables is exact by construction -- and the first candidate whose running sum exceeds u * total is taken,
// total being the sum of the same candidate weights (not the stored table entry, so the choice never falls off the
// end; should rounding leave u * total above every running sum, the last candidate of positive weight is taken).  Its
// sub-segments are pushed 3' first, so the traceback runs depth first, 5' first, and uses one uniform number per
// decision, in that order (philox.h: rp_sample_block, t = 0, 1, ...; one block serves four decisions).
//
// On the device a warp takes one sample at a time and its 32 lanes evaluate the candidates of a decision 32 at a
// time (sample_pick_shfl); the host reference form (sample_pick_direct) walks them one by one.  The pending segments of
// a warp live in the problem's T_RR table, which only the unpaired-window pass uses, and which it writes before it
// reads: n + 2 entries per warp, so at most te / (n + 2) warps sample one problem.
#ifndef RP_MCC_SAMPLE_H
#define RP_MCC_SAMPLE_H

#include "mcc_core.h"
#include "philox.h"

namespace rp {

enum { SG_Q = 0, SG_QQ, SG_QB, SG_QM, SG_QM1, SG_QM2 };
constexpr int SAMPLE_QB_CANDS = 2 + (MAXLOOP + 1) * (MAXLOOP + 1) + 1;   // hairpin, interior (u1,u2) grid, multiloop, nick

RP_HD uint64_t seg_pack(int kind, int i, int j) { return (uint64_t)kind | ((uint64_t)i << 8) | ((uint64_t)j << 32); }

// q(i, i+d) with q(i, i-1) = 1
RP_HD double q_or_one(const Ctx& c, int i, int j) { return j < i ? 1. : TB(c, T_Q, j - i, i); }

// number of candidates of a decision
RP_HD int sample_count(int kind, int i, int j) {
  switch (kind) {
    case SG_Q: return j - i - TURN + 1;             // all unpaired; then k = i .. j-TURN-1 (5' end of the last stem)
    case SG_QQ: return j - i - TURN;                // l = i+TURN+1 .. j
    case SG_QB: return SAMPLE_QB_CANDS;
    case SG_QM: return 2 * (j - i - TURN);          // k = p .. r-TURN-1, two each
    case SG_QM1: return j - i - TURN;               // l = k+TURN+1 .. r
    default: return j - i - 2 * TURN - 2 > 0 ? j - i - 2 * TURN - 2 : 0;   // SG_QM2: k = p+TURN+2 .. r-TURN-1
  }
}

// Weight of candidate x of segment (kind, i, j).  Orders:
//   SG_Q   x = 0: i..j unpaired, scale^(d+1);  x = 1 + (k-i): q(i,k-1) qq(k,j)
//   SG_QQ  x = l - (i+TURN+1): qb(i,l) extstem scale^(j-l)
//   SG_QB  x = 0: hairpin;  x = 1 + u1 (MAXLOOP+1) + u2: interior loop with inner pair (i+1+u1, j-1-u2), by its class
//          (dev_model.h: bulge, 1xn and generic from the class tables QBAU / QB1N / QBI times g, the nine small shapes
//          table-driven, with the stacking factor);  x = last-1: multiloop;  x = last: the exterior loop over the nick
//          (without the pair factor of (i,j), pair_sc: it is common to every candidate, and the decision compares the
//          candidates with their own sum, so it does not change which one is taken)
//   SG_QM  x = 2(k-p): p..k-1 unpaired, mlb^(k-p) qm1(k,r);  x = 2(k-p)+1: qm(p,k-1) qm1(k,r)
//   SG_QM1 x = l - (k+TURN+1): qb(k,l) mlstem mlb^(r-l)
//   SG_QM2 x = k - (p+TURN+2): qm(p,k-1) qm1(k,r), not at the nick
RP_HD double sample_weight(const Ctx& c, int kind, int i, int j, int x) {
  const DevModel& M = *c.M;
  const int n = c.n;
  switch (kind) {
    case SG_Q: {
      if (x == 0) return VEC(c, V_SCALE, j - i + 1);
      const int k = i + x - 1;
      return q_or_one(c, i, k - 1) * TB(c, T_QQ, j - k, k);
    }
    case SG_QQ: {
      const int l = i + TURN + 1 + x;
      const int type = cell_type(c, i, l);
      if (!type) return 0.;
      return TB(c, T_QB, l - i, i) *
             ext_stem(M, type, (i > 1 && ss(c, i - 1, i)) ? base(c, i - 1) : -1, (l < n && ss(c, l, l + 1)) ? base(c, l + 1) : -1) *
             VEC(c, V_SCALE, j - l);
    }
    case SG_QB: {
      const int d = j - i, type = cell_type(c, i, j);
      if (x == 0) return ss(c, i, j) ? hairpin(c, i, j, type) : 0.;
      if (x == SAMPLE_QB_CANDS - 2) {
        if (!(ss(c, i, i + 1) && ss(c, j - 1, j))) return 0.;
        return TB(c, T_QM2, d - 2, i + 1) * M.expMLclosing * ml_stem(M, rtype(type), base(c, j - 1), base(c, i + 1)) *
               VEC(c, V_SCALE, 2);
      }
      if (x == SAMPLE_QB_CANDS - 1) {
        if (ss(c, i, j)) return 0.;
        double t = VEC(c, V_SCALE, 2) * q_or_one(c, i + 1, c.cp - 1) * q_or_one(c, c.cp, j - 1);
        return t * ext_stem(M, rtype(type), ss(c, j - 1, j) ? base(c, j - 1) : -1, ss(c, i, i + 1) ? base(c, i + 1) : -1);
      }
      const int u1 = (x - 1) / (MAXLOOP + 1), u2 = (x - 1) % (MAXLOOP + 1);
      const int dd = u1 + u2 + 2;
      const int ddmax = d - (TURN + 1) < MAXLOOP + 2 ? d - (TURN + 1) : MAXLOOP + 2;
      if (u1 + u2 > MAXLOOP || dd > ddmax) return 0.;
      // strand guards of inside_interior: the inner pair's 5' end stays on i's strand, its 3' end on j's
      const int maxpo = (c.cp > 0 && i < c.cp) ? c.cp - 1 - i : 1000;
      const int maxu2 = (c.cp > 0 && j >= c.cp) ? j - 1 - c.cp : 1000;
      if (u1 + 1 > maxpo || u2 > maxu2) return 0.;
      const int k = i + 1 + u1, l = j - 1 - u2;
      const int si1 = base(c, i + 1), sj1 = base(c, j - 1);
      switch (M.gcls[u1][u2]) {
        case CLS_SPECIAL: {
          const int t2 = cell_type(c, k, l);
          if (!t2) return 0.;
          const int s = special_index(u1, u2);
          return TB(c, T_QB, d - dd, k) * stack_sc(c, s, i, j, special_loop(M, s, type, rtype(t2), si1, sj1, base(c, k - 1), base(c, l + 1)));
        }
        case CLS_BULGE: return (type > 2 ? M.expTermAU : 1.0) * M.gfull[u1][u2] * TB(c, T_QBAU, d - dd, k);
        case CLS_1N: return M.mm1n[type][si1][sj1] * M.gfull[u1][u2] * TB(c, T_QB1N, d - dd, k);
        case CLS_GENERIC: return M.mmI[type][si1][sj1] * M.gfull[u1][u2] * TB(c, T_QBI, d - dd, k);
        default: return 0.;
      }
    }
    case SG_QM: {
      const int k = i + (x >> 1);
      const double m1 = TB(c, T_QM1, j - k, k);
      if (!(x & 1)) return ss(c, i, k) ? VEC(c, V_MLB, k - i) * m1 : 0.;
      return (k - 1 - i >= TURN + 1 && ss(c, k - 1, k)) ? TB(c, T_QM, k - 1 - i, i) * m1 : 0.;
    }
    case SG_QM1: {
      const int l = i + TURN + 1 + x;
      const int type = cell_type(c, i, l);
      if (!type || !ss(c, i - 1, i) || !ss(c, l, l + 1) || !ss(c, l, j)) return 0.;
      return TB(c, T_QB, l - i, i) * ml_stem(M, type, i > 1 ? base(c, i - 1) : -1, l < n ? base(c, l + 1) : -1) *
             VEC(c, V_MLB, j - l);
    }
    default: {
      const int k = i + TURN + 2 + x;
      if (!ss(c, k - 1, k)) return 0.;
      return TB(c, T_QM, k - 1 - i, i) * TB(c, T_QM1, j - k, k);
    }
  }
}

// Host reference form of a decision: the candidates one by one.  Returns the candidate taken, -1 if none has weight.
RP_HD int sample_pick_direct(const Ctx& c, int kind, int i, int j, double u) {
  const int cnt = sample_count(kind, i, j);
  double total = 0.;
  int last = -1;
  for (int x = 0; x < cnt; x++) {
    const double w = sample_weight(c, kind, i, j, x);
    total += w;
    if (w > 0.) last = x;
  }
  const double target = u * total;
  double run = 0.;
  for (int x = 0; x < cnt; x++) {
    const double w = sample_weight(c, kind, i, j, x);
    run += w;
    if (w > 0. && run > target) return x;
  }
  return last;
}

#ifdef RP_SHFL_FORMS
// The warp form: lane L takes candidate x0 + 31 - L of each group of 32, so that a running sum in candidate order is a
// suffix sum over the lanes (shuffles down only, each from one source offset, as mcc_band_shfl.cuh uses them).  All 32
// lanes call it and get the same result.
RP_HD int sample_pick_shfl(const Ctx& c, int kind, int i, int j, double u, int lane) {
  const unsigned FULL = 0xffffffffu;
  const int cnt = sample_count(kind, i, j);
  double total = 0.;
  int last = -1;
  for (int x0 = 0; x0 < cnt; x0 += 32) {
    const int x = x0 + 31 - lane;
    double w = x < cnt ? sample_weight(c, kind, i, j, x) : 0.;
    if (w > 0. && x > last) last = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double y = __shfl_down_sync(FULL, w, o);
      if (lane + o < 32) w += y;
    }
    total += __shfl_sync(FULL, w, 0);
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_down_sync(FULL, last, o);
    last = y > last ? y : last;
  }
  last = __shfl_sync(FULL, last, 0);
  const double target = u * total;
  double run = 0.;
  for (int x0 = 0; x0 < cnt; x0 += 32) {
    const int x = x0 + 31 - lane;
    const double w = x < cnt ? sample_weight(c, kind, i, j, x) : 0.;
    double s = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double y = __shfl_down_sync(FULL, s, o);
      if (lane + o < 32) s += y;
    }
    int hit = (w > 0. && run + s > target) ? lane : -1;   // the first candidate that crosses is the highest lane
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_down_sync(FULL, hit, o);
      hit = y > hit ? y : hit;
    }
    hit = __shfl_sync(FULL, hit, 0);
    if (hit >= 0) return x0 + 31 - hit;
    run += __shfl_sync(FULL, s, 0);
  }
  return last;
}
#endif

// one sample of the problem into pt[0..n-1] (zero on entry): pt[k-1] = partner of base k, 1-based.  `stk`: the warp's
// pending segments.  Every lane of a warp runs it (the shuffle form) or lane 0 alone (the direct form); lanes store
// the same values to the same addresses.
template <bool SHFL>
RP_HD void sample_one(const Ctx& c, uint64_t seed, int pair, int kind, int sample, int16_t* pt, uint64_t* stk, int lane) {
  const int n = c.n;
  int sp = 0, t = 0;
  uint64_t blk[4] = {0, 0, 0, 0};
  if (n - 1 >= TURN + 1) stk[sp++] = seg_pack(SG_Q, 1, n);
  while (sp > 0) {
    const uint64_t e = stk[--sp];
    const int sk = (int)(e & 255), i = (int)((e >> 8) & 0xffffff), j = (int)(e >> 32);
    if ((t & 3) == 0) rp_sample_block(seed, pair, kind, sample, t >> 2, blk);
    const double u = rp_uniform53(blk[t & 3]);
    t++;
    int x;
#ifdef RP_SHFL_FORMS
    if constexpr (SHFL) x = sample_pick_shfl(c, sk, i, j, u, lane);
    else
#endif
      x = sample_pick_direct(c, sk, i, j, u);
    (void)lane;
    if (x < 0) continue;   // (a segment of weight 0 is never pushed; kept for safety against underflow)
    switch (sk) {
      case SG_Q:
        if (x > 0) {
          const int k = i + x - 1;
          stk[sp++] = seg_pack(SG_QQ, k, j);
          if (k - 1 - i >= TURN + 1) stk[sp++] = seg_pack(SG_Q, i, k - 1);
        }
        break;
      case SG_QQ: stk[sp++] = seg_pack(SG_QB, i, i + TURN + 1 + x); break;
      case SG_QB:
        pt[i - 1] = (int16_t)j;
        pt[j - 1] = (int16_t)i;
        if (x == SAMPLE_QB_CANDS - 2) {
          stk[sp++] = seg_pack(SG_QM2, i + 1, j - 1);
        } else if (x == SAMPLE_QB_CANDS - 1) {
          if (j - 1 - c.cp >= TURN + 1) stk[sp++] = seg_pack(SG_Q, c.cp, j - 1);
          if (c.cp - 1 - (i + 1) >= TURN + 1) stk[sp++] = seg_pack(SG_Q, i + 1, c.cp - 1);
        } else if (x > 0) {
          const int u1 = (x - 1) / (MAXLOOP + 1), u2 = (x - 1) % (MAXLOOP + 1);
          stk[sp++] = seg_pack(SG_QB, i + 1 + u1, j - 1 - u2);
        }
        break;
      case SG_QM: {
        const int k = i + (x >> 1);
        stk[sp++] = seg_pack(SG_QM1, k, j);
        if (x & 1) stk[sp++] = seg_pack(SG_QM, i, k - 1);
        break;
      }
      case SG_QM1: stk[sp++] = seg_pack(SG_QB, i, i + TURN + 1 + x); break;
      default: {
        const int k = i + TURN + 2 + x;
        stk[sp++] = seg_pack(SG_QM1, k, j);
        stk[sp++] = seg_pack(SG_QM, i, k - 1);
        break;
      }
    }
  }
}

}  // namespace rp
#endif
