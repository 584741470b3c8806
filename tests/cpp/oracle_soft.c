/* oracle_soft.c -- TEST INFRASTRUCTURE.  The CPU oracle (oracle/rp_oracle.c) on an ensemble with stacking
 * pseudo-energies, the soft constraint of rp_batch_create_soft, optionally restricted by an allowed-pair matrix as in
 * oracle_masked.c (allow == NULL: every pair).  E[0..n-1] holds one integer pseudo-energy per base of the problem's
 * sequence in 0.01 kcal/mol (E == NULL: none).  Every stack -- an interior loop closed by (i,j) around (i+1,j-1) with
 * i and j on one strand -- has its weight multiplied by exp(-(E_i + E_{i+1} + E_{j-1} + E_j) * 10 / kT).
 *   orc_fold_soft       McCaskill with that factor on the stack term of the inside and of the outside recursion.  The
 *                       unpaired windows (unpaired_windows of rp_oracle.c, unchanged) need nothing more: a stack leaves
 *                       no base unpaired, so it adds to no gap weight a window can see.
 *   orc_enumerate_soft  exhaustive enumeration that finds every stack of a structure itself and adds its four
 *                       pseudo-energies to the structure's energy.
 * It lives apart from oracle_masked.c, which stays the exact reference of the constraint tests; with E == NULL
 * orc_fold_soft equals orc_fold_masked (and with allow == NULL too, orc_fold) bit for bit, which tests/test_shape.py
 * checks.  Built by tests/test_shape.py. */
#include "oracle_masked.c"

/* per-base factors f[1..n] = exp(-E * 10 / kT), 1 without data */
static double* stack_factors(const orc_params* P, const int* E, int n) {
  double* f = (double*)malloc(sizeof(double) * (size_t)(n + 2));
  for (int i = 0; i <= n + 1; i++) f[i] = 1.;
  if (E)
    for (int i = 1; i <= n; i++) f[i] = exp(-(double)E[i - 1] * 10. / P->kT);
  return f;
}

/* the factor of the stack closed by (i,j); intermolecular stacks carry none */
#define STACK_SC(f, cp, i, j) (same_strand(cp, i, j) ? (f)[i] * (f)[(i) + 1] * (f)[(j) - 1] * (f)[j] : 1.)

/* inside_masked() of oracle_masked.c with the stack factor */
static void inside_soft(const orc_params* P, const seq_t* sq, tables_t* t, const unsigned char* allow, const double* f) {
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
            double w = T(qb, k, l) * exp_intloop(P, u1, j - l - 1, type, RTYPE[t2], S[i + 1], S[j - 1], S[k - 1], S[l + 1]) * scale[u1 + j - l + 1];
            if (u1 == 0 && l == j - 1) w *= STACK_SC(f, cp, i, j);
            qbt += w;
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

/* outside() of rp_oracle.c with the stack factor in the interior-loop context (step 2) */
static void outside_soft(const orc_params* P, const seq_t* sq, tables_t* t, const double* f) {
  const int n = t->n, cp = t->cp, ld = t->ld;
  const int* S = sq->S;
  double *q = t->q, *qb = t->qb, *qm = t->qm, *out = t->out;
  const double* scale = t->scale;
  const double Z = t->Z;
#define SS(a, b) same_strand(cp, a, b)
  double* prml = (double*)calloc(n + 2, sizeof(double));
  double* prm_l = (double*)calloc(n + 2, sizeof(double));
  double* prm_l1 = (double*)calloc(n + 2, sizeof(double));
  double* Ql = (double*)calloc(n + 2, sizeof(double));
  double* Qr = (double*)calloc(n + 2, sizeof(double));
  double* Qlout = (double*)calloc(n + 2, sizeof(double));
  int ql_ready = 0;

  for (int i = 1; i <= n; i++)
    for (int j = i + TURN + 1; j <= n; j++) {
      int type = PAIR[S[i]][S[j]];
      if (type && T(qb, i, j) > 0.)
        T(out, i, j) = T(q, 1, i - 1) * T(q, j + 1, n) / Z *
                       exp_extstem(P, type, (i > 1 && SS(i - 1, i)) ? S[i - 1] : -1, (j < n && SS(j, j + 1)) ? S[j + 1] : -1);
    }

  for (int l = n; l > TURN + 1; l--) {
    for (int k = 1; k < l - TURN; k++) {
      int t2 = PAIR[S[k]][S[l]];
      if (!t2 || T(qb, k, l) == 0.) continue;
      t2 = RTYPE[t2];
      double acc = 0.;
      for (int i = MAX2(1, k - P->maxloop - 1); i <= k - 1; i++) {
        if (!SS(i, k)) continue;
        int u1 = k - i - 1;
        for (int j = l + 1; j <= MIN2(l + P->maxloop - u1 + 1, n); j++) {
          if (!SS(l, j)) break;
          int type = PAIR[S[i]][S[j]];
          if (!type || T(out, i, j) == 0.) continue;
          double w = T(out, i, j) * scale[u1 + j - l + 1] *
                     exp_intloop(P, u1, j - l - 1, type, t2, S[i + 1], S[j - 1], S[k - 1], S[l + 1]);
          if (u1 == 0 && j == l + 1) w *= STACK_SC(f, cp, i, j);
          acc += w;
        }
      }
      T(out, k, l) += acc;
    }
    if (l < n && SS(l, l + 1)) {
      double prm_MLb = 0.;
      for (int k = 2; k < l - TURN; k++) {
        int i = k - 1;
        double prmt = 0., prmt1 = 0.;
        if (SS(i, i + 1)) {
          int tt = PAIR[S[i]][S[l + 1]];
          if (tt && l + 1 - i > TURN)
            prmt1 = T(out, i, l + 1) * P->expMLclosing * exp_mlstem(P, RTYPE[tt], S[l], S[i + 1]);
          for (int j = l + 2; j <= n; j++) {
            if (!SS(j - 1, j)) continue;
            tt = PAIR[S[i]][S[j]];
            if (!tt || T(out, i, j) == 0.) continue;
            prmt += T(out, i, j) * exp_mlstem(P, RTYPE[tt], S[j - 1], S[i + 1]) * T(qm, l + 1, j - 1);
          }
          prmt *= P->expMLclosing;
        }
        prm_l[i] = prm_l1[i] * t->mlb[1] + prmt1;
        if (SS(k - 1, k)) prm_MLb = prm_MLb * t->mlb[1] + prmt;
        else prm_MLb = 0.;
        prml[i] = prmt + prm_l[i];
        int tk = PAIR[S[k]][S[l]];
        if (!tk || T(qb, k, l) == 0.) continue;
        if (!SS(k - 1, k)) continue;
        double temp = prm_MLb;
        for (int ii = 1; ii <= k - 2; ii++)
          if (SS(ii, ii + 1)) temp += prml[ii] * T(qm, ii + 1, k - 1);
        temp *= exp_mlstem(P, tk, S[k - 1], S[l + 1]) * scale[2];
        T(out, k, l) += temp;
      }
    } else {
      for (int i = 0; i <= n; i++) prm_l[i] = 0.;
    }
    { double* tmp = prm_l1; prm_l1 = prm_l; prm_l = tmp; }

    if (cp > 0) {
      if (l >= cp) {
        double Qrout = 0.;
        for (int r = l + 1; r <= n; r++) Qrout += Qr[r] * T(q, l + 1, r - 1);
        if (Qrout != 0.)
          for (int k = cp; k < l - TURN; k++) {
            int tk = PAIR[S[k]][S[l]];
            if (!tk || T(qb, k, l) == 0.) continue;
            T(out, k, l) += Qrout * T(q, cp, k - 1) * exp_extstem(P, tk, k > cp ? S[k - 1] : -1, S[l + 1]);
          }
        double s = 0.;
        for (int p = 1; p < cp; p++) {
          int tp = PAIR[S[p]][S[l]];
          if (!tp || l - p <= TURN || T(out, p, l) == 0.) continue;
          s += T(out, p, l) * scale[2] * T(q, p + 1, cp - 1) *
               exp_extstem(P, RTYPE[tp], SS(l - 1, l) ? S[l - 1] : -1, SS(p, p + 1) ? S[p + 1] : -1);
        }
        Qr[l] = s;
      } else {
        if (!ql_ready) {
          for (int p = 1; p < cp; p++) {
            double s = 0.;
            for (int r = cp; r <= n; r++) {
              int tp = PAIR[S[p]][S[r]];
              if (!tp || r - p <= TURN || T(out, p, r) == 0.) continue;
              s += T(out, p, r) * scale[2] * T(q, cp, r - 1) *
                   exp_extstem(P, RTYPE[tp], SS(r - 1, r) ? S[r - 1] : -1, SS(p, p + 1) ? S[p + 1] : -1);
            }
            Ql[p] = s;
          }
          for (int k = 2; k < cp; k++) {
            double s = 0.;
            for (int p = 1; p < k; p++) s += Ql[p] * T(q, p + 1, k - 1);
            Qlout[k] = s;
          }
          ql_ready = 1;
        }
        for (int k = 2; k < l - TURN; k++) {
          int tk = PAIR[S[k]][S[l]];
          if (!tk || T(qb, k, l) == 0. || Qlout[k] == 0.) continue;
          T(out, k, l) += Qlout[k] * T(q, l + 1, cp - 1) * exp_extstem(P, tk, S[k - 1], l + 1 < cp ? S[l + 1] : -1);
        }
      }
    }
  }
  free(prml); free(prm_l); free(prm_l1); free(Ql); free(Qr); free(Qlout);
#undef SS
}

int orc_fold_soft(const orc_params* P, const char* seq, int n, int cp, const unsigned char* allow, const int* E,
                  double* pr, double* up, int max_w, double* logZ) {
  if (!P || n < 1) return 1;
  seq_t sq; tables_t t;
  seq_init(&sq, seq, n, cp);
  tables_alloc(&t, n, cp, P->pf_scale, P->expMLbase);
  double* f = stack_factors(P, E, n);
  inside_soft(P, &sq, &t, allow, f);
  if (logZ) *logZ = log(t.Z) + n * log(P->pf_scale);
  if (pr || up) outside_soft(P, &sq, &t, f);
  if (pr) {
    memset(pr, 0, sizeof(double) * (size_t)(n + 1) * (n + 1));
    const int ld = t.ld;
    for (int i = 1; i <= n; i++)
      for (int j = i + TURN + 1; j <= n; j++) pr[(size_t)i * (n + 1) + j] = T(t.out, i, j) * T(t.qb, i, j);
  }
  if (up && max_w > 0) unpaired_windows(P, &sq, &t, max_w, up);
  free(f);
  tables_free(&t);
  seq_free(&sq);
  return 0;
}

/* enum_eval() of rp_oracle.c, times the pseudo-energies of the structure's intramolecular stacks */
static const int* g_E;
static void enum_eval_soft(enum_t* E) {
  const orc_params* P = E->P;
  const int* S = E->sq->S;
  const int n = E->n, cp = E->cp;
  const int* pt = E->pt;
  double wgt = 1.;
  for (int x = 1; x <= n;) {
    if (pt[x] > x) {
      int k = x, l = pt[x];
      wgt *= exp_extstem(P, PAIR[S[k]][S[l]], (k > 1 && same_strand(cp, k - 1, k)) ? S[k - 1] : -1,
                         (l < n && same_strand(cp, l, l + 1)) ? S[l + 1] : -1);
      x = l + 1;
    } else x++;
  }
  for (int i = 1; i <= n && wgt != 0.; i++)
    if (pt[i] > i) wgt *= loop_weight_closed(E, i, pt[i]);
  if (wgt == 0.) return;
  int esum = 0;   /* a stack: (i,j) closes a loop whose only content is the pair (i+1,j-1) */
  for (int i = 1; i <= n && g_E; i++) {
    const int j = pt[i];
    if (j > i && pt[i + 1] == j - 1 && same_strand(cp, i, j)) esum += g_E[i - 1] + g_E[i] + g_E[j - 2] + g_E[j - 1];
  }
  wgt *= exp(-(double)esum * 10. / P->kT);
  E->Z += wgt;
  for (int i = 1; i <= n; i++)
    if (pt[i] > i) E->pr[(size_t)i * (n + 1) + pt[i]] += wgt;
  if (E->up)
    for (int i = 1; i <= n; i++)
      for (int d = 0; d < E->w && i + d <= n; d++) {
        if (pt[i + d]) break;
        E->up[(size_t)(i - 1) * E->w + d] += wgt;
      }
}

/* enum_rec_masked() of oracle_masked.c, evaluating with enum_eval_soft */
static void enum_rec_soft(enum_t* E, int pos, int* stack, int sp) {
  const int n = E->n;
  if (pos > n) { enum_eval_soft(E); return; }
  if (E->pt[pos]) {
    enum_rec_soft(E, pos + 1, stack, sp - 1);
    return;
  }
  enum_rec_soft(E, pos + 1, stack, sp);
  int limit = sp > 0 ? stack[sp - 1] - 1 : n;
  for (int j = pos + TURN + 1; j <= limit; j++) {
    if (E->pt[j] || !PAIR[E->sq->S[pos]][E->sq->S[j]] || !ALLOWED(g_allow, pos, j, n)) continue;
    E->pt[pos] = j; E->pt[j] = pos;
    int saved = stack[sp];
    stack[sp] = j;
    enum_rec_soft(E, pos + 1, stack, sp + 1);
    stack[sp] = saved;
    E->pt[pos] = 0; E->pt[j] = 0;
  }
}

int orc_enumerate_soft(const orc_params* P, const char* seq, int n, int cp, const unsigned char* allow, const int* Ev,
                       double* pr, double* up, int max_w, double* logZ) {
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
  g_E = Ev;
  enum_rec_soft(&E, 1, stack, 0);
  g_allow = NULL;
  g_E = NULL;
  for (size_t x = 0; x < (size_t)(n + 1) * (n + 1); x++) pr[x] /= E.Z;
  if (E.up) for (size_t x = 0; x < (size_t)n * max_w; x++) up[x] /= E.Z;
  if (logZ) *logZ = log(E.Z);
  free(stack); free(E.pt);
  seq_free(&sq);
  return 0;
}
