/* oracle_sample.c -- TEST INFRASTRUCTURE.  A CPU sampler of secondary structures on the soft oracle's tables
 * (oracle_soft.c: the allowed-pair matrix and the stacking factors, over oracle/rp_oracle.c), the reference of the
 * general kernel's sampling phase (ractip_b200/csrc/mcc_sample.h).  It draws the same Philox numbers (philox.h), makes
 * the same decisions in the same order -- depth first, 5' first, one uniform number per decision -- over the same
 * candidates in the same order, and takes the first candidate whose running sum exceeds u * total.  Its weights come
 * from the oracle's own loop functions (exp_intloop, exp_hairpin, ...), not from the kernel's class tables, so that the
 * two agree sample by sample only up to rounding far below the spacing of the uniform numbers.  Built by
 * tests/test_sampling.py. */
#include "oracle_soft.c"
#include "philox.h"

enum { SG_Q = 0, SG_QQ, SG_QB, SG_QM, SG_QM1, SG_QM2 };
#define QB_CANDS (2 + (MAXLOOP + 1) * (MAXLOOP + 1) + 1)

typedef struct {
  const orc_params* P;
  const seq_t* sq;
  const tables_t* t;
  const double* qq;   /* qq(i,j) as inside_soft builds it (it keeps no copy) */
  const unsigned char* allow;
  const double* f;    /* stacking factors */
} smp_t;

static int count_of(int kind, int i, int j) {
  switch (kind) {
    case SG_Q: return j - i - TURN + 1;
    case SG_QQ: return j - i - TURN;
    case SG_QB: return QB_CANDS;
    case SG_QM: return 2 * (j - i - TURN);
    case SG_QM1: return j - i - TURN;
    default: return MAX2(j - i - 2 * TURN - 2, 0);
  }
}

static double weight_of(const smp_t* X, int kind, int i, int j, int x) {
  const orc_params* P = X->P;
  const tables_t* t = X->t;
  const int n = t->n, cp = t->cp, ld = t->ld;
  const int* S = X->sq->S;
  const double *q = t->q, *qb = t->qb, *qm = t->qm, *qm1 = t->qm1, *qm2 = t->qm2, *qq = X->qq;
#define SS(a, b) same_strand(cp, a, b)
#define TYPE(a, b) (ALLOWED(X->allow, a, b, n) ? PAIR[S[a]][S[b]] : 0)
  switch (kind) {
    case SG_Q: {
      if (x == 0) return t->scale[j - i + 1];
      const int k = i + x - 1;
      return T(q, i, k - 1) * T(qq, k, j);
    }
    case SG_QQ: {
      const int l = i + TURN + 1 + x, type = TYPE(i, l);
      if (!type) return 0.;
      return T(qb, i, l) * exp_extstem(P, type, (i > 1 && SS(i - 1, i)) ? S[i - 1] : -1, (l < n && SS(l, l + 1)) ? S[l + 1] : -1) *
             t->scale[j - l];
    }
    case SG_QB: {
      const int type = TYPE(i, j);
      if (x == 0) return SS(i, j) ? exp_hairpin(P, j - i - 1, type, S[i + 1], S[j - 1], X->sq->str + i - 1) * t->scale[j - i + 1] : 0.;
      if (x == QB_CANDS - 2) {
        if (!(SS(i, i + 1) && SS(j - 1, j))) return 0.;
        return T(qm2, i + 1, j - 1) * P->expMLclosing * exp_mlstem(P, RTYPE[type], S[j - 1], S[i + 1]) * t->scale[2];
      }
      if (x == QB_CANDS - 1) {
        if (SS(i, j)) return 0.;
        return T(q, i + 1, cp - 1) * T(q, cp, j - 1) * t->scale[2] *
               exp_extstem(P, RTYPE[type], SS(j - 1, j) ? S[j - 1] : -1, SS(i, i + 1) ? S[i + 1] : -1);
      }
      const int u1 = (x - 1) / (MAXLOOP + 1), u2 = (x - 1) % (MAXLOOP + 1);
      const int k = i + 1 + u1, l = j - 1 - u2;
      if (u1 + u2 > P->maxloop || l - k < TURN + 1 || !SS(i, k) || !SS(l, j)) return 0.;
      const int t2 = PAIR[S[k]][S[l]];
      if (!t2) return 0.;
      double w = T(qb, k, l) * exp_intloop(P, u1, u2, type, RTYPE[t2], S[i + 1], S[j - 1], S[k - 1], S[l + 1]) *
                 t->scale[u1 + u2 + 2];
      if (u1 == 0 && u2 == 0) w *= STACK_SC(X->f, cp, i, j);
      return w;
    }
    case SG_QM: {
      const int k = i + (x >> 1);
      if (!(x & 1)) return SS(i, k) ? t->mlb[k - i] * T(qm1, k, j) : 0.;
      return (k - 1 - i >= TURN + 1 && SS(k - 1, k)) ? T(qm, i, k - 1) * T(qm1, k, j) : 0.;
    }
    case SG_QM1: {
      const int l = i + TURN + 1 + x, type = TYPE(i, l);
      if (!type || !SS(i - 1, i) || !SS(l, l + 1) || !SS(l, j)) return 0.;
      return T(qb, i, l) * exp_mlstem(P, type, i > 1 ? S[i - 1] : -1, l < n ? S[l + 1] : -1) * t->mlb[j - l];
    }
    default: {
      const int k = i + TURN + 2 + x;
      return SS(k - 1, k) ? T(qm, i, k - 1) * T(qm1, k, j) : 0.;
    }
  }
#undef TYPE
#undef SS
}

static int pick(const smp_t* X, int kind, int i, int j, double u) {
  const int cnt = count_of(kind, i, j);
  double total = 0.;
  int last = -1;
  for (int x = 0; x < cnt; x++) {
    const double w = weight_of(X, kind, i, j, x);
    total += w;
    if (w > 0.) last = x;
  }
  const double target = u * total;
  double run = 0.;
  for (int x = 0; x < cnt; x++) {
    const double w = weight_of(X, kind, i, j, x);
    run += w;
    if (w > 0. && run > target) return x;
  }
  return last;
}

/* Samples first .. first+num-1 of the problem (kind 0 s1, 1 s2, 2 s1&s2 of pair `pair`, for the Philox key) into
 * out[s*n .. s*n+n-1]: pair tables, out[k-1] = 1-based partner of base k, 0 if unpaired.  allow, E as orc_fold_soft.
 * Returns 0, or 1 for bad arguments. */
int orc_sample_soft(const orc_params* P, const char* seq, int n, int cp, const unsigned char* allow, const int* E,
                    uint64_t seed, int pair, int kind, int first, int num, int16_t* out) {
  if (!P || n < 1 || num < 0) return 1;
  seq_t sq; tables_t t;
  seq_init(&sq, seq, n, cp);
  tables_alloc(&t, n, cp, P->pf_scale, P->expMLbase);
  double* f = stack_factors(P, E, n);
  inside_soft(P, &sq, &t, allow, f);
  const int ld = t.ld;
  double* qq = (double*)calloc((size_t)ld * ld, sizeof(double));
  for (int j = TURN + 2; j <= n; j++)
    for (int i = j - TURN - 1; i >= 1; i--) {   /* inside_soft's qq, term for term */
      const int type = ALLOWED(allow, i, j, n) ? PAIR[sq.S[i]][sq.S[j]] : 0;
      double e = T(qq, i, j - 1) * t.scale[1];
      if (type)
        e += T(t.qb, i, j) * exp_extstem(P, type, (i > 1 && same_strand(cp, i - 1, i)) ? sq.S[i - 1] : -1,
                                         (j < n && same_strand(cp, j, j + 1)) ? sq.S[j + 1] : -1);
      T(qq, i, j) = e;
    }
  smp_t X = {P, &sq, &t, qq, allow, f};
  uint64_t* stk = (uint64_t*)malloc(sizeof(uint64_t) * (size_t)(n + 2));
  for (int s = 0; s < num; s++) {
    int16_t* pt = out + (size_t)s * n;
    memset(pt, 0, sizeof(int16_t) * (size_t)n);
    int sp = 0, dec = 0;
    uint64_t blk[4] = {0, 0, 0, 0};
#define PUSH(k, a, b) (stk[sp++] = (uint64_t)(k) | ((uint64_t)(a) << 8) | ((uint64_t)(b) << 32))
    if (n - 1 >= TURN + 1) PUSH(SG_Q, 1, n);
    while (sp > 0) {
      const uint64_t e = stk[--sp];
      const int sk = (int)(e & 255), i = (int)((e >> 8) & 0xffffff), j = (int)(e >> 32);
      if ((dec & 3) == 0) rp_sample_block(seed, pair, kind, first + s, dec >> 2, blk);
      const int x = pick(&X, sk, i, j, rp_uniform53(blk[dec & 3]));
      dec++;
      if (x < 0) continue;
      switch (sk) {
        case SG_Q:
          if (x > 0) {
            const int k = i + x - 1;
            PUSH(SG_QQ, k, j);
            if (k - 1 - i >= TURN + 1) PUSH(SG_Q, i, k - 1);
          }
          break;
        case SG_QQ: PUSH(SG_QB, i, i + TURN + 1 + x); break;
        case SG_QB:
          pt[i - 1] = (int16_t)j;
          pt[j - 1] = (int16_t)i;
          if (x == QB_CANDS - 2) {
            PUSH(SG_QM2, i + 1, j - 1);
          } else if (x == QB_CANDS - 1) {
            if (j - 1 - cp >= TURN + 1) PUSH(SG_Q, cp, j - 1);
            if (cp - 1 - (i + 1) >= TURN + 1) PUSH(SG_Q, i + 1, cp - 1);
          } else if (x > 0) {
            PUSH(SG_QB, i + 1 + (x - 1) / (MAXLOOP + 1), j - 1 - (x - 1) % (MAXLOOP + 1));
          }
          break;
        case SG_QM: {
          const int k = i + (x >> 1);
          PUSH(SG_QM1, k, j);
          if (x & 1) PUSH(SG_QM, i, k - 1);
          break;
        }
        case SG_QM1: PUSH(SG_QB, i, i + TURN + 1 + x); break;
        default: {
          const int k = i + TURN + 2 + x;
          PUSH(SG_QM1, k, j);
          PUSH(SG_QM, i, k - 1);
          break;
        }
      }
    }
#undef PUSH
  }
  free(stk);
  free(qq);
  free(f);
  tables_free(&t);
  seq_free(&sq);
  return 0;
}

/* the Philox block of (counter, key), for the test of philox.h against numpy */
void orc_philox(const uint64_t* ctr, const uint64_t* key, uint64_t* out) { rp_philox4x64(ctr, key, out); }
