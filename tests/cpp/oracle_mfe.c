/* oracle_mfe.c -- TEST INFRASTRUCTURE.  A plain Zuker restatement of the minimum free energy rp_run_mfe computes, written
 * independently of the kernel (ractip_b200/csrc/mfe_core.h) and checked against exhaustive enumeration by
 * tests/test_mfe.py.
 *
 * Energy of a structure: the integer loop energies of rp_energy_of_structure (eval.cpp; dangles 2, special hairpins,
 * the loop that contains the nick scored as an exterior loop, DuplexInit once when a pair joins the strands), plus the
 * stacking pseudo-energies E (E(i)+E(i+1)+E(j-1)+E(j) per stack within one strand) and the unpaired pseudo-energies U,
 * applied literally: U(x) for every base x left unpaired in a hairpin, interior loop, multiloop, nick loop or the
 * exterior loop, and for both bases of a pair that joins the strands.  Structures: canonical pairs with j - i > 3,
 * interior loops up to 30 unpaired bases, pairs allowed by `allow` ((n+1) x (n+1), 1-based, NULL: all).
 *
 * The exterior loop of a co-fold is a prefix minimum with a flag for "a joining stem has been placed", and the multiloop
 * the classic unpaired-prefix form; no recursion is shared with the kernel's.
 */
#include <limits.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "ractip_prob.h"

#define INF 100000000

typedef struct {
  const rp_model* P;
  int n, cp;
  int* s;                   /* s[1..n] base codes, 0 outside */
  char* str;                /* letters for the special hairpins, 'X' for non-ACGU */
  const uint8_t* allow;
  const int* E;             /* E[1..n] or NULL */
  long long* Up;            /* prefix sums of U: Up[k] = U(1) + .. + U(k) */
  int* C;
  int* FM1;
  int* FML;
} Orc;

#define AT(t, i, j) ((t)[(size_t)(i) * (o->n + 2) + (j)])

static int mn(int a, int b) { return a < b ? a : b; }
static int ptype(int a, int b) {
  static const int T[5][5] = {{0, 0, 0, 0, 0}, {0, 0, 0, 0, 5}, {0, 0, 0, 1, 0}, {0, 0, 2, 0, 3}, {0, 6, 0, 4, 0}};
  return T[a][b];
}
static int rtyp(int t) { static const int R[8] = {0, 2, 1, 4, 3, 6, 5, 7}; return R[t]; }
/* the nick lies between a and b (a < b) */
static int nick(const Orc* o, int a, int b) { return o->cp > 0 && a < o->cp && b >= o->cp; }
static int same(const Orc* o, int a, int b) { return !nick(o, a, b); }
static long long useg(const Orc* o, int a, int b) { return b < a ? 0 : o->Up[b] - o->Up[a - 1]; }
static int can(const Orc* o, int i, int j) {
  if (j - i <= 3) return 0;
  if (!ptype(o->s[i], o->s[j])) return 0;
  return !o->allow || o->allow[(size_t)i * (o->n + 1) + j];
}

static int ext_stem(const rp_model* P, int type, int s5, int s3) {
  int e = 0;
  if (s5 >= 0 && s3 >= 0) e += P->mismatchExt37[type][s5][s3] < 0 ? P->mismatchExt37[type][s5][s3] : 0;
  else if (s5 >= 0) e += P->dangle5_37[type][s5] < 0 ? P->dangle5_37[type][s5] : 0;
  else if (s3 >= 0) e += P->dangle3_37[type][s3] < 0 ? P->dangle3_37[type][s3] : 0;
  if (type > 2) e += P->TerminalAU37;
  return e;
}
static int ml_stem(const rp_model* P, int type, int s5, int s3) {
  int e = 0;
  if (s5 >= 0 && s3 >= 0) e += P->mismatchM37[type][s5][s3] < 0 ? P->mismatchM37[type][s5][s3] : 0;
  else if (s5 >= 0) e += P->dangle5_37[type][s5] < 0 ? P->dangle5_37[type][s5] : 0;
  else if (s3 >= 0) e += P->dangle3_37[type][s3] < 0 ? P->dangle3_37[type][s3] : 0;
  if (type > 2) e += P->TerminalAU37;
  return e + P->ML_intern37;
}
static int hairpin(const Orc* o, int i, int j) {
  const rp_model* P = o->P;
  const int u = j - i - 1, type = ptype(o->s[i], o->s[j]);
  int e = u <= 30 ? P->hairpin37[u] : P->hairpin37[30] + (int)(P->lxc37 * log(u / 30.));
  if (P->special_hp && (u == 3 || u == 4 || u == 6)) {
    char loop[16];
    memcpy(loop, o->str + i - 1, (size_t)u + 2);
    loop[u + 2] = 0;
    const char* list = u == 4 ? P->Tetraloops : (u == 6 ? P->Hexaloops : P->Triloops);
    const int* en = u == 4 ? P->Tetraloop37 : (u == 6 ? P->Hexaloop37 : P->Triloop37);
    const char* hit = strstr(list, loop);
    if (hit) return en[(hit - list) / (u + 3)];
  }
  if (u == 3) return e + (type > 2 ? P->TerminalAU37 : 0);
  return e + P->mismatchH37[type][o->s[i + 1]][o->s[j - 1]];
}
static int int_loop(const rp_model* P, int n1, int n2, int type, int type2, int si1, int sj1, int sp1, int sq1) {
  const int nl = n1 > n2 ? n1 : n2, ns = n1 > n2 ? n2 : n1;
  if (nl == 0) return P->stack37[type][type2];
  if (ns == 0) {
    int e = P->bulge37[nl];
    if (nl == 1) e += P->stack37[type][type2];
    else {
      if (type > 2) e += P->TerminalAU37;
      if (type2 > 2) e += P->TerminalAU37;
    }
    return e;
  }
  int ninio = (nl - ns) * P->ninio37;
  if (ninio > P->MAX_NINIO) ninio = P->MAX_NINIO;
  if (ns == 1) {
    if (nl == 1) return P->int11_37[type][type2][si1][sj1];
    if (nl == 2) return n1 == 1 ? P->int21_37[type][type2][si1][sq1][sj1] : P->int21_37[type2][type][sq1][si1][sp1];
    return P->internal_loop37[nl + 1] + ninio + P->mismatch1nI37[type][si1][sj1] + P->mismatch1nI37[type2][sq1][sp1];
  }
  if (ns == 2) {
    if (nl == 2) return P->int22_37[type][type2][si1][sp1][sq1][sj1];
    if (nl == 3) return P->internal_loop37[5] + P->ninio37 + P->mismatch23I37[type][si1][sj1] + P->mismatch23I37[type2][sq1][sp1];
  }
  return P->internal_loop37[nl + ns] + ninio + P->mismatchI37[type][si1][sj1] + P->mismatchI37[type2][sq1][sp1];
}
/* exterior stem (k,l): dangles on its own strand */
static int ext_of(const Orc* o, int k, int l) {
  return ext_stem(o->P, ptype(o->s[k], o->s[l]), (k > 1 && same(o, k - 1, k)) ? o->s[k - 1] : -1,
                  (l < o->n && same(o, l, l + 1)) ? o->s[l + 1] : -1);
}

/* cell (i,j): C, FM1, FML.  Xs / Xp: the exterior minima of a..cp-1 and cp..b (joining cells only) */
static void fill(Orc* o, int i, int j, const int* Xs, const int* Xp) {
  const rp_model* P = o->P;
  const int n = o->n, cpx = o->cp;
  const int* E = o->E;
  int c = INF;
  if (can(o, i, j)) {
    const int type = ptype(o->s[i], o->s[j]);
    const int joins = nick(o, i, j);
    if (!joins) c = mn(c, hairpin(o, i, j) + (int)useg(o, i + 1, j - 1));
    for (int k = i + 1; k <= i + 31 && k < j; k++)
      for (int l = j - 1; l > k + 3; l--) {
        const int u1 = k - i - 1, u2 = j - l - 1;
        if (u1 + u2 > 30) break;
        if (!can(o, k, l) || AT(o->C, k, l) >= INF) continue;
        if (joins && !nick(o, k, l)) continue;   /* the nick would lie in the loop: a nick loop, not an interior one */
        int e = int_loop(P, u1, u2, type, rtyp(ptype(o->s[k], o->s[l])), o->s[i + 1], o->s[j - 1], o->s[k - 1], o->s[l + 1]);
        e += AT(o->C, k, l) + (int)(useg(o, i + 1, k - 1) + useg(o, l + 1, j - 1));
        if (u1 + u2 == 0 && !joins) e += E[i] + E[i + 1] + E[j - 1] + E[j];
        c = mn(c, e);
      }
    if (same(o, i, i + 1) && same(o, j - 1, j)) {   /* multiloop: two or more stems, none at the nick */
      int best = INF;
      for (int k = i + 6; k <= j - 5; k++) {
        if (nick(o, k - 1, k)) continue;
        const int a = AT(o->FML, i + 1, k - 1), b = AT(o->FM1, k, j - 1);
        if (a < INF && b < INF) best = mn(best, a + b);
      }
      if (best < INF) c = mn(c, best + P->ML_closing37 + ml_stem(P, rtyp(type), o->s[j - 1], o->s[i + 1]));
    }
    if (joins) {   /* the nick loop, scored as an exterior loop; both bases of (i,j) count as unpaired */
      const int a = i + 1 <= cpx - 1 ? Xs[i + 1] : 0, b = j - 1 >= cpx ? Xp[j - 1] : 0;
      if (a < INF && b < INF)
        c = mn(c, a + b + ext_stem(P, rtyp(type), same(o, j - 1, j) ? o->s[j - 1] : -1, same(o, i, i + 1) ? o->s[i + 1] : -1));
      if (c < INF) c += (int)(useg(o, i, i) + useg(o, j, j));
    }
  }
  AT(o->C, i, j) = c;
  /* FM1: stem (i,l), l+1..j unpaired, no nick from i-1 to the end of the stem's run */
  int m1 = INF;
  if (!nick(o, i - 1, i))
    for (int l = i + 4; l <= j; l++) {
      if (AT(o->C, i, l) >= INF || nick(o, l, l + 1) || nick(o, l, j)) continue;
      m1 = mn(m1, AT(o->C, i, l) + ml_stem(P, ptype(o->s[i], o->s[l]), i > 1 ? o->s[i - 1] : -1, l < n ? o->s[l + 1] : -1) +
                      P->ML_BASE37 * (j - l) + (int)useg(o, l + 1, j));
    }
  AT(o->FM1, i, j) = m1;
  /* FML: i..k-1 unpaired then one stem, or FML(i,k-1) then one stem */
  int ml = INF;
  for (int k = i; k <= j - 4; k++) {
    const int b = AT(o->FM1, k, j);
    if (b >= INF) continue;
    if (!nick(o, i, k)) ml = mn(ml, P->ML_BASE37 * (k - i) + (int)useg(o, i, k - 1) + b);
    if (k - 1 - i >= 4 && !nick(o, k - 1, k) && AT(o->FML, i, k - 1) < INF) ml = mn(ml, AT(o->FML, i, k - 1) + b);
  }
  AT(o->FML, i, j) = ml;
}

int orc_mfe(const rp_model* P, const char* seq, int n, int cp, const uint8_t* allow, const int* E0, const int* U0, int* mfe) {
  if (!P || !seq || n < 1 || !mfe) return 1;
  Orc O, *o = &O;
  memset(o, 0, sizeof O);
  o->P = P; o->n = n; o->cp = cp > 1 && cp <= n ? cp : 0; o->allow = allow;
  const size_t N2 = (size_t)(n + 2) * (n + 2);
  o->s = calloc((size_t)n + 2, sizeof(int));
  o->str = calloc((size_t)n + 2, 1);
  o->Up = calloc((size_t)n + 2, sizeof(long long));
  int* E = calloc((size_t)n + 2, sizeof(int));
  o->C = malloc(N2 * sizeof(int));
  o->FM1 = malloc(N2 * sizeof(int));
  o->FML = malloc(N2 * sizeof(int));
  int* Xs = malloc(((size_t)n + 3) * sizeof(int));   /* exterior minimum of a..cp-1 */
  int* Xp = malloc(((size_t)n + 3) * sizeof(int));   /* exterior minimum of cp..b */
  int* F = malloc(2 * ((size_t)n + 2) * sizeof(int));
  for (int i = 1; i <= n; i++) {
    const char ch = seq[i - 1];
    int code = 0;
    switch (ch) {
      case 'A': case 'a': code = 1; break;
      case 'C': case 'c': code = 2; break;
      case 'G': case 'g': code = 3; break;
      case 'U': case 'u': case 'T': case 't': code = 4; break;
      default: code = 0;
    }
    o->s[i] = code;
    o->str[i - 1] = (ch == 'A' || ch == 'C' || ch == 'G' || ch == 'U' || ch == 'a' || ch == 'c' || ch == 'g' || ch == 'u')
                        ? "NACGU"[code] : 'X';
    o->Up[i] = o->Up[i - 1] + (U0 ? U0[i - 1] : 0);
    E[i] = E0 ? E0[i - 1] : 0;
  }
  o->E = E;
  for (size_t x = 0; x < N2; x++) o->C[x] = o->FM1[x] = o->FML[x] = INF;
  /* same-strand cells first (they never depend on a joining one), then the exterior minima of the strand ends that
   * the nick loops need, then the cells whose span crosses the nick */
  for (int pass = 0; pass < (o->cp > 0 ? 2 : 1); pass++) {
    if (pass == 1) {
      const int cpx = o->cp;
      Xs[cpx] = 0;
      for (int a = cpx - 1; a >= 1; a--) {
        int v = Xs[a + 1] + (int)useg(o, a, a);
        for (int l = a + 4; l <= cpx - 1; l++)
          if (AT(o->C, a, l) < INF) v = mn(v, AT(o->C, a, l) + ext_of(o, a, l) + (l + 1 <= cpx - 1 ? Xs[l + 1] : 0));
        Xs[a] = v;
      }
      Xp[cpx - 1] = 0;
      for (int b = cpx; b <= n; b++) {
        int v = Xp[b - 1] + (int)useg(o, b, b);
        for (int k = cpx; k <= b - 4; k++)
          if (AT(o->C, k, b) < INF) v = mn(v, (k - 1 >= cpx ? Xp[k - 1] : 0) + AT(o->C, k, b) + ext_of(o, k, b));
        Xp[b] = v;
      }
    }
    for (int d = 4; d < n; d++)
      for (int i = 1; i + d <= n; i++)
        if (nick(o, i, i + d) == pass) fill(o, i, i + d, Xs, Xp);
  }
  /* exterior loop: F[j][f] = minimum over 1..j, f = 1 when one stem joins the strands (at most one can) */
  F[0] = 0;
  F[1] = INF;
  for (int j = 1; j <= n; j++) {
    int v0 = F[2 * (j - 1)] + (int)useg(o, j, j);
    int v1 = F[2 * (j - 1) + 1] < INF ? F[2 * (j - 1) + 1] + (int)useg(o, j, j) : INF;
    for (int k = 1; k <= j - 4; k++) {
      if (AT(o->C, k, j) >= INF) continue;
      const int stem = AT(o->C, k, j) + ext_of(o, k, j);
      if (nick(o, k, j)) {
        v1 = mn(v1, F[2 * (k - 1)] + stem);
      } else {
        v0 = mn(v0, F[2 * (k - 1)] + stem);
        if (F[2 * (k - 1) + 1] < INF) v1 = mn(v1, F[2 * (k - 1) + 1] + stem);
      }
    }
    F[2 * j] = v0;
    F[2 * j + 1] = v1;
  }
  {
    const int a = F[2 * n], b = F[2 * n + 1];
    *mfe = mn(a, b < INF ? b + P->DuplexInit37 : INF);
  }
  free(Xs); free(Xp);
  free(F);
  free(E);
  free(o->s); free(o->str); free(o->Up); free(o->C); free(o->FM1); free(o->FML);
  return 0;
}
