/* oracle_probed.c -- TEST INFRASTRUCTURE.  The soft oracle (oracle_soft.c: allowed-pair matrix and stacking
 * pseudo-energies) with unpaired pseudo-energies as well, the soft constraint of rp_batch_create_probed, applied
 * LITERALLY: U[0..n-1] holds one integer pseudo-energy per base in 0.01 kcal/mol (U == NULL: none), and every base a
 * structure leaves unpaired -- in a hairpin, an interior loop, a multiloop, the exterior loop -- multiplies its weight
 * by f(x) = exp(-U_x * 10 / kT).  In a two-strand problem a base paired with the other strand counts as unpaired: a
 * pair (i,j) that joins the strands multiplies by f(i) f(j).
 *   orc_fold_probed       McCaskill in which every scale factor of an unpaired run (scale[u], mlb[u]) is joined by
 *                         the product of f over that run, inside, outside and in the unpaired windows (pf_unstru).
 *                         An intermolecular pair's own factor sits in its qb and in the loops it closes.
 *   orc_enumerate_probed  exhaustive enumeration: a structure's weight times f over its unpaired bases.
 * With U == NULL (or all 0) orc_fold_probed equals orc_fold_soft bit for bit, which tests/test_unpaired.py checks.
 * Built by tests/test_unpaired.py. */
#include "oracle_soft.c"

/* f[0..n+1] = exp(-U * 10 / kT), 1 without data */
static double* unpaired_factors(const orc_params* P, const int* U, int n) {
  double* f = (double*)malloc(sizeof(double) * (size_t)(n + 2));
  for (int i = 0; i <= n + 1; i++) f[i] = 1.;
  if (U)
    for (int i = 1; i <= n; i++) f[i] = exp(-(double)U[i - 1] * 10. / P->kT);
  return f;
}

/* product of f over the run a..b (1 when empty) */
static double run_f(const double* f, int a, int b) {
  double r = 1.;
  for (int x = a; x <= b; x++) r *= f[x];
  return r;
}

/* the factor of a pair that joins the strands: both bases count as unpaired */
#define CROSS_F(uf, cp, i, j) (same_strand(cp, i, j) ? 1. : (uf)[i] * (uf)[j])

static void inside_probed(const orc_params* P, const seq_t* sq, tables_t* t, const unsigned char* allow,
                          const double* f, const double* uf) {
  const int n = t->n, cp = t->cp, ld = t->ld;
  const int* S = sq->S;
  double *q = t->q, *qb = t->qb, *qm = t->qm, *qm1 = t->qm1, *qm2 = t->qm2;
  const double* scale = t->scale;
  double* qq = (double*)calloc((size_t)(n + 2) * (n + 2), sizeof(double));
#define SS(a, b) same_strand(cp, a, b)
  for (int i = 1; i <= n + 1; i++) T(q, i, i - 1) = 1.0;
  for (int d = 0; d <= TURN && d < n; d++)
    for (int i = 1; i + d <= n; i++) T(q, i, i + d) = scale[d + 1] * run_f(uf, i, i + d);
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
        if (SS(i, j)) qbt += exp_hairpin(P, u, type, S[i + 1], S[j - 1], sq->str + i - 1) * scale[u + 2] * run_f(uf, i + 1, j - 1);
        for (int k = i + 1; k <= MIN2(i + P->maxloop + 1, j - TURN - 2); k++) {
          int u1 = k - i - 1;
          if (!SS(i, k)) break;
          for (int l = MAX2(k + TURN + 1, j - 1 - P->maxloop + u1); l < j; l++) {
            if (!SS(l, j)) continue;
            int t2 = PAIR[S[k]][S[l]];
            if (!t2) continue;
            double w = T(qb, k, l) * exp_intloop(P, u1, j - l - 1, type, RTYPE[t2], S[i + 1], S[j - 1], S[k - 1], S[l + 1]) * scale[u1 + j - l + 1];
            if (u1 == 0 && l == j - 1) w *= STACK_SC(f, cp, i, j);
            w *= run_f(uf, i + 1, k - 1) * run_f(uf, l + 1, j - 1);
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
        qbt *= CROSS_F(uf, cp, i, j);
      }
      T(qb, i, j) = qbt;
      double v = SS(j - 1, j) ? T(qm1, i, j - 1) * t->mlb[1] * uf[j] : 0.;
      if (type && SS(i - 1, i) && SS(j, j + 1))
        v += qbt * exp_mlstem(P, type, i > 1 ? S[i - 1] : -1, j < n ? S[j + 1] : -1);
      T(qm1, i, j) = v;
      double tm = 0.;
      for (int k = i + 1; k <= j; k++) {
        double a = 0.;
        if (SS(k - 1, k)) a += T(qm, i, k - 1);
        if (SS(i, k)) a += t->mlb[k - i] * run_f(uf, i, k - 1);
        tm += a * T(qm1, k, j);
      }
      T(qm, i, j) = tm + v;
      double e = T(qq, i, j - 1) * scale[1] * uf[j];
      if (type) e += qbt * exp_extstem(P, type, (i > 1 && SS(i - 1, i)) ? S[i - 1] : -1, (j < n && SS(j, j + 1)) ? S[j + 1] : -1);
      T(qq, i, j) = e;
      double tq = scale[j - i + 1] * run_f(uf, i, j) + e;
      for (int k = i + 1; k <= j; k++) tq += T(q, i, k - 1) * T(qq, k, j);
      T(q, i, j) = tq;
    }
  }
  t->Z = T(q, 1, n);
  free(qq);
#undef SS
}

/* outside_soft() with the unpaired runs' factors; an enclosing pair that joins the strands brings its own factor to
 * every loop it closes (interior loops, multiloops -- whose other stems lie on one strand -- and the loop with the nick) */
static void outside_probed(const orc_params* P, const seq_t* sq, tables_t* t, const double* f, const double* uf) {
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
          w *= run_f(uf, i + 1, k - 1) * run_f(uf, l + 1, j - 1) * CROSS_F(uf, cp, i, j);
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
            prmt1 = T(out, i, l + 1) * CROSS_F(uf, cp, i, l + 1) * P->expMLclosing * exp_mlstem(P, RTYPE[tt], S[l], S[i + 1]);
          for (int j = l + 2; j <= n; j++) {
            if (!SS(j - 1, j)) continue;
            tt = PAIR[S[i]][S[j]];
            if (!tt || T(out, i, j) == 0.) continue;
            prmt += T(out, i, j) * CROSS_F(uf, cp, i, j) * exp_mlstem(P, RTYPE[tt], S[j - 1], S[i + 1]) * T(qm, l + 1, j - 1);
          }
          prmt *= P->expMLclosing;
        }
        /* right run l+1..j-1 grows by base l+1, left run i+1..k-1 by base k-1 */
        prm_l[i] = prm_l1[i] * t->mlb[1] * uf[l + 1] + prmt1;
        if (SS(k - 1, k)) prm_MLb = prm_MLb * t->mlb[1] * uf[k - 1] + prmt;
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
          s += T(out, p, l) * CROSS_F(uf, cp, p, l) * scale[2] * T(q, p + 1, cp - 1) *
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
              s += T(out, p, r) * CROSS_F(uf, cp, p, r) * scale[2] * T(q, cp, r - 1) *
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

/* unpaired_windows() of rp_oracle.c with the unpaired runs' factors (single strand) */
static void unpaired_windows_probed(const orc_params* P, const seq_t* sq, const tables_t* t, int w, double* up,
                                    const double* uf) {
  const int n = t->n, ld = t->ld;
  const int* S = sq->S;
  const double *q = t->q, *qb = t->qb, *qm = t->qm, *qm2 = t->qm2, *out = t->out;
  const double* scale = t->scale;
  size_t sz = (size_t)(n + 2) * (n + 2);
  double* D = (double*)calloc(sz, sizeof(double));
  double* Mc = (double*)calloc(sz, sizeof(double));
  double* R = (double*)calloc(sz, sizeof(double));
  double* L = (double*)calloc(sz, sizeof(double));
  double* X = (double*)calloc(sz, sizeof(double));
  for (int p = 1; p <= n; p++)
    for (int o = p + TURN + 1; o <= n; o++) {
      int type = PAIR[S[p]][S[o]];
      double po = T(out, p, o);
      if (!type || po == 0.) continue;
      int u = o - p - 1;
      T(D, p, o) += po * exp_hairpin(P, u, type, S[p + 1], S[o - 1], sq->str + p - 1) * scale[u + 2] * run_f(uf, p + 1, o - 1);
      for (int k = p + 1; k <= MIN2(p + P->maxloop + 1, o - TURN - 2); k++) {
        int u1 = k - p - 1;
        for (int l = MAX2(k + TURN + 1, o - 1 - P->maxloop + u1); l < o; l++) {
          int t2 = PAIR[S[k]][S[l]];
          if (!t2) continue;
          double wgt = po * T(qb, k, l) * scale[u1 + o - l + 1] *
                       exp_intloop(P, u1, o - l - 1, type, RTYPE[t2], S[p + 1], S[o - 1], S[k - 1], S[l + 1]) *
                       run_f(uf, p + 1, k - 1) * run_f(uf, l + 1, o - 1);
          T(D, p, k) += wgt;
          T(D, l, o) += wgt;
        }
      }
      T(Mc, p, o) = po * P->expMLclosing * exp_mlstem(P, RTYPE[type], S[o - 1], S[p + 1]) * scale[2];
    }
  for (int a = 1; a <= n; a++)
    for (int b = n; b >= 1; b--)
      T(D, a, b) += T(D, a - 1, b) + (b < n ? T(D, a, b + 1) : 0.) - (b < n ? T(D, a - 1, b + 1) : 0.);
  for (int p = 1; p <= n; p++)
    for (int j = p + 1; j <= n; j++) {
      double s = 0.;
      for (int o = j + 2; o <= n; o++) s += T(Mc, p, o) * T(qm2, j + 1, o - 1);
      T(R, p, j) = s;
    }
  for (int o = 1; o <= n; o++)
    for (int i = 2; i < o; i++) {
      double s2 = 0., s1 = 0.;
      for (int p = 1; p <= i - 2; p++) {
        s2 += T(Mc, p, o) * T(qm2, p + 1, i - 1);
        s1 += T(Mc, p, o) * T(qm, p + 1, i - 1);
      }
      T(L, i, o) = s2;
      T(X, i, o) = s1;
    }
  for (int i = 1; i <= n; i++)
    for (int d = 0; d < w; d++) {
      int j = i + d;
      double v = 0.;
      if (j <= n) {
        v = T(q, 1, i - 1) * scale[j - i + 1] * run_f(uf, i, j) * T(q, j + 1, n) / t->Z;
        if (i > 1 && j < n) {
          v += T(D, i - 1, j + 1);
          double m1 = 0., m2 = 0., m3 = 0.;
          for (int p = 1; p < i; p++) m1 += t->mlb[j - p] * run_f(uf, p + 1, j) * T(R, p, j);
          for (int o = j + 1; o <= n; o++) m2 += t->mlb[o - i] * run_f(uf, i, o - 1) * T(L, i, o);
          for (int o = j + 2; o <= n; o++) m3 += T(qm, j + 1, o - 1) * T(X, i, o);
          v += m1 + m2 + m3 * t->mlb[j - i + 1] * run_f(uf, i, j);
        }
      }
      up[(size_t)(i - 1) * w + d] = v;
    }
  free(D); free(Mc); free(R); free(L); free(X);
}

int orc_fold_probed(const orc_params* P, const char* seq, int n, int cp, const unsigned char* allow, const int* E,
                    const int* U, double* pr, double* up, int max_w, double* logZ) {
  if (!P || n < 1) return 1;
  seq_t sq; tables_t t;
  seq_init(&sq, seq, n, cp);
  tables_alloc(&t, n, cp, P->pf_scale, P->expMLbase);
  double* f = stack_factors(P, E, n);
  double* uf = unpaired_factors(P, U, n);
  inside_probed(P, &sq, &t, allow, f, uf);
  if (logZ) *logZ = log(t.Z) + n * log(P->pf_scale);
  if (pr || up) outside_probed(P, &sq, &t, f, uf);
  if (pr) {
    memset(pr, 0, sizeof(double) * (size_t)(n + 1) * (n + 1));
    const int ld = t.ld;
    for (int i = 1; i <= n; i++)
      for (int j = i + TURN + 1; j <= n; j++) pr[(size_t)i * (n + 1) + j] = T(t.out, i, j) * T(t.qb, i, j);
  }
  if (up && max_w > 0) unpaired_windows_probed(P, &sq, &t, max_w, up, uf);
  free(f);
  free(uf);
  tables_free(&t);
  seq_free(&sq);
  return 0;
}

/* enum_eval_soft() of oracle_soft.c, times f over the structure's unpaired bases and the bases of its intermolecular
 * pairs */
static const int* g_U;
static void enum_eval_probed(enum_t* E) {
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
  int esum = 0;
  for (int i = 1; i <= n && g_E; i++) {
    const int j = pt[i];
    if (j > i && pt[i + 1] == j - 1 && same_strand(cp, i, j)) esum += g_E[i - 1] + g_E[i] + g_E[j - 2] + g_E[j - 1];
  }
  int usum = 0;   /* unpaired, or paired with the other strand */
  for (int i = 1; i <= n && g_U; i++) {
    const int j = pt[i];
    if (!j || !same_strand(cp, i < j ? i : j, i < j ? j : i)) usum += g_U[i - 1];
  }
  wgt *= exp(-(double)esum * 10. / P->kT) * exp(-(double)usum * 10. / P->kT);
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

static void enum_rec_probed(enum_t* E, int pos, int* stack, int sp) {
  const int n = E->n;
  if (pos > n) { enum_eval_probed(E); return; }
  if (E->pt[pos]) {
    enum_rec_probed(E, pos + 1, stack, sp - 1);
    return;
  }
  enum_rec_probed(E, pos + 1, stack, sp);
  int limit = sp > 0 ? stack[sp - 1] - 1 : n;
  for (int j = pos + TURN + 1; j <= limit; j++) {
    if (E->pt[j] || !PAIR[E->sq->S[pos]][E->sq->S[j]] || !ALLOWED(g_allow, pos, j, n)) continue;
    E->pt[pos] = j; E->pt[j] = pos;
    int saved = stack[sp];
    stack[sp] = j;
    enum_rec_probed(E, pos + 1, stack, sp + 1);
    stack[sp] = saved;
    E->pt[pos] = 0; E->pt[j] = 0;
  }
}

int orc_enumerate_probed(const orc_params* P, const char* seq, int n, int cp, const unsigned char* allow, const int* Ev,
                         const int* Uv, double* pr, double* up, int max_w, double* logZ) {
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
  g_U = Uv;
  enum_rec_probed(&E, 1, stack, 0);
  g_allow = NULL;
  g_E = NULL;
  g_U = NULL;
  for (size_t x = 0; x < (size_t)(n + 1) * (n + 1); x++) pr[x] /= E.Z;
  if (E.up) for (size_t x = 0; x < (size_t)n * max_w; x++) up[x] /= E.Z;
  if (logZ) *logZ = log(E.Z);
  free(stack); free(E.pt);
  seq_free(&sq);
  return 0;
}
