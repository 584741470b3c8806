/* oracle_masked.c -- TEST INFRASTRUCTURE.  The CPU oracle (oracle/rp_oracle.c, compiled into the same library) on an
 * ensemble restricted by an allowed-pair matrix: allow[i*(n+1)+j] != 0 lets (i,j), 1 <= i < j <= n, pair (allow ==
 * NULL: every pair).  This is what a structure constraint does to each McCaskill problem (rp_batch_create_constrained):
 * it removes pairs and changes no loop energy.
 *   orc_fold_masked       McCaskill with qb(i,j) = 0 for every removed pair.  The outside pass and the unpaired
 *                         windows then leave such a pair out by themselves: they only ever give an outside value to a
 *                         pair with qb > 0, and only use a pair as an enclosing loop through that value.
 *   orc_enumerate_masked  exhaustive enumeration of the structures whose pairs are all allowed.
 * Built by tests/test_constraints.py. */
#include "../../oracle/rp_oracle.c"

#define ALLOWED(a, i, j, n) (!(a) || (a)[(size_t)(i) * ((n) + 1) + (j)])

/* inside() of rp_oracle.c with the one restriction: qb of a removed pair is 0 */
static void inside_masked(const orc_params* P, const seq_t* sq, tables_t* t, const unsigned char* allow) {
  const int n = t->n, cp = t->cp, ld = t->ld;
  const int* S = sq->S;
  double *q = t->q, *qb = t->qb, *qm = t->qm, *qm1 = t->qm1, *qm2 = t->qm2;
  const double* scale = t->scale;
  double* qq = (double*)calloc((size_t)(n + 2) * (n + 2), sizeof(double));
#define SS(a, b) same_strand(cp, a, b)
  for (int i = 1; i <= n + 1; i++) T(q, i, i - 1) = 1.0;
  for (int d = 0; d <= TURN && d < n; d++)
    for (int i = 1; i + d <= n; i++) T(q, i, i + d) = scale[d + 1];
  for (int j = TURN + 2; j <= n; j++) {
    for (int i = j - TURN - 1; i >= 1; i--) {
      int type = ALLOWED(allow, i, j, n) ? PAIR[S[i]][S[j]] : 0;
      int u = j - i - 1;
      double qbt = 0.;
      double m2 = 0.;
      for (int k = i + 2; k <= j - 1; k++)
        if (SS(k - 1, k)) m2 += T(qm, i + 1, k - 1) * T(qm1, k, j - 1);
      T(qm2, i + 1, j - 1) = m2;
      if (type) {
        if (SS(i, j)) qbt += exp_hairpin(P, u, type, S[i + 1], S[j - 1], sq->str + i - 1) * scale[u + 2];
        for (int k = i + 1; k <= MIN2(i + P->maxloop + 1, j - TURN - 2); k++) {
          int u1 = k - i - 1;
          if (!SS(i, k)) break;
          for (int l = MAX2(k + TURN + 1, j - 1 - P->maxloop + u1); l < j; l++) {
            if (!SS(l, j)) continue;
            int t2 = PAIR[S[k]][S[l]];
            if (!t2) continue;
            qbt += T(qb, k, l) * exp_intloop(P, u1, j - l - 1, type, RTYPE[t2], S[i + 1], S[j - 1], S[k - 1], S[l + 1]) * scale[u1 + j - l + 1];
          }
        }
        if (SS(i, i + 1) && SS(j - 1, j))
          qbt += m2 * P->expMLclosing * exp_mlstem(P, RTYPE[type], S[j - 1], S[i + 1]) * scale[2];
        if (!SS(i, j)) {
          double tmp = T(q, i + 1, cp - 1) * T(q, cp, j - 1) * scale[2];
          tmp *= exp_extstem(P, RTYPE[type], SS(j - 1, j) ? S[j - 1] : -1, SS(i, i + 1) ? S[i + 1] : -1);
          qbt += tmp;
        }
      }
      T(qb, i, j) = qbt;
      double v = SS(j - 1, j) ? T(qm1, i, j - 1) * t->mlb[1] : 0.;
      if (type && SS(i - 1, i) && SS(j, j + 1))
        v += qbt * exp_mlstem(P, type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
      T(qm1, i, j) = v;
      double tm = 0.;
      for (int k = i + 1; k <= j; k++) {
        double a = 0.;
        if (SS(k - 1, k)) a += T(qm, i, k - 1);
        if (SS(i, k)) a += t->mlb[k - i];
        tm += a * T(qm1, k, j);
      }
      T(qm, i, j) = tm + v;
      double e = T(qq, i, j - 1) * scale[1];
      if (type) e += qbt * exp_extstem(P, type, (i > 1 && SS(i - 1, i)) ? S[i - 1] : -1, (j < n && SS(j, j + 1)) ? S[j + 1] : -1);
      T(qq, i, j) = e;
      double tq = scale[j - i + 1] + e;
      for (int k = i + 1; k <= j; k++) tq += T(q, i, k - 1) * T(qq, k, j);
      T(q, i, j) = tq;
    }
  }
  t->Z = T(q, 1, n);
  free(qq);
#undef SS
}

int orc_fold_masked(const orc_params* P, const char* seq, int n, int cp, const unsigned char* allow, double* pr, double* up,
                    int max_w, double* logZ) {
  if (!P || n < 1) return 1;
  seq_t sq; tables_t t;
  seq_init(&sq, seq, n, cp);
  tables_alloc(&t, n, cp, P->pf_scale, P->expMLbase);
  inside_masked(P, &sq, &t, allow);
  if (logZ) *logZ = log(t.Z) + n * log(P->pf_scale);
  if (pr || up) outside(P, &sq, &t);
  if (pr) {
    memset(pr, 0, sizeof(double) * (size_t)(n + 1) * (n + 1));
    const int ld = t.ld;
    for (int i = 1; i <= n; i++)
      for (int j = i + TURN + 1; j <= n; j++) pr[(size_t)i * (n + 1) + j] = T(t.out, i, j) * T(t.qb, i, j);
  }
  if (up && max_w > 0) unpaired_windows(P, &sq, &t, max_w, up);
  tables_free(&t);
  seq_free(&sq);
  return 0;
}

/* enum_rec() of rp_oracle.c, opening only allowed pairs */
static const unsigned char* g_allow;
static void enum_rec_masked(enum_t* E, int pos, int* stack, int sp) {
  const int n = E->n;
  if (pos > n) { enum_eval(E); return; }
  if (E->pt[pos]) {
    enum_rec_masked(E, pos + 1, stack, sp - 1);
    return;
  }
  enum_rec_masked(E, pos + 1, stack, sp);
  int limit = sp > 0 ? stack[sp - 1] - 1 : n;
  for (int j = pos + TURN + 1; j <= limit; j++) {
    if (E->pt[j] || !PAIR[E->sq->S[pos]][E->sq->S[j]] || !ALLOWED(g_allow, pos, j, n)) continue;
    E->pt[pos] = j; E->pt[j] = pos;
    int saved = stack[sp];
    stack[sp] = j;
    enum_rec_masked(E, pos + 1, stack, sp + 1);
    stack[sp] = saved;
    E->pt[pos] = 0; E->pt[j] = 0;
  }
}

int orc_enumerate_masked(const orc_params* P, const char* seq, int n, int cp, const unsigned char* allow, double* pr,
                         double* up, int max_w, double* logZ) {
  if (!P || n < 1 || n > 24) return 1;
  seq_t sq;
  seq_init(&sq, seq, n, cp);
  enum_t E;
  E.P = P; E.sq = &sq; E.n = n; E.cp = cp; E.w = max_w;
  E.pt = (int*)calloc(n + 2, sizeof(int));
  E.Z = 0.;
  E.pr = pr; E.up = (max_w > 0) ? up : NULL;
  memset(pr, 0, sizeof(double) * (size_t)(n + 1) * (n + 1));
  if (E.up) memset(up, 0, sizeof(double) * (size_t)n * max_w);
  int* stack = (int*)calloc(n + 2, sizeof(int));
  g_allow = allow;
  enum_rec_masked(&E, 1, stack, 0);
  g_allow = NULL;
  for (size_t x = 0; x < (size_t)(n + 1) * (n + 1); x++) pr[x] /= E.Z;
  if (E.up) for (size_t x = 0; x < (size_t)n * max_w; x++) up[x] /= E.Z;
  if (logZ) *logZ = log(E.Z);
  free(stack); free(E.pt);
  seq_free(&sq);
  return 0;
}
