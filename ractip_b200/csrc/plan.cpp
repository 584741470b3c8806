// plan.cpp -- the host arithmetic of a batch (plan.h) and the planning entry points of the C ABI.
#include "plan.h"

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstring>

#include "mcc_band.h"
#include "seq_encode.h"

namespace rp {

size_t bp_len(int L) { return (size_t)(L + 1) * (size_t)(L + 2) / 2; }

int check_pairs(const rp_pair* pairs, int n_pairs, const rp_opts* opts) {
  if (!pairs || !opts || n_pairs < 0) return RP_ERR_ARG;
  for (int p = 0; p < n_pairs; p++)
    if (!pairs[p].s1 || pairs[p].n1 < 1 || pairs[p].n2 < 0 || (pairs[p].n2 > 0 && !pairs[p].s2)) return RP_ERR_ARG;   // n2 == 0: s1 alone
  return RP_OK;
}

// Structure constraints: c1 over s1, c2 over s2, in the alphabet of RactIP's joint structures --
//   .  no constraint      x  the base pairs with nothing
//   ( )  an intramolecular pair, bracket-matched within its string
//   [ (c1 only), ] (c2 only)  an intermolecular pair: the k-th '[' from the 3' end of s1 pairs with the k-th ']' from
//        the 5' end of s2 (nested, as RactIP's joint structures are)
// A constraint only removes pairs.  Each of a pair's problems sees the brackets of its own kind and keeps unpaired
// the bases the other kind pairs (a base paired on the other strand has no partner in its own strand's problem; a
// base paired within its strand forms no intermolecular pair):
//   s1:     bracket pairs () of c1,   unpaired x [
//   s2:     bracket pairs () of c2,   unpaired x ]
//   s1&s2:  bracket pairs [] across,  unpaired x ( )
// Pair (i,j) of a problem is allowed when neither base is unpaired, either base is bracketed only if they are each
// other's partner, and (i,j) crosses no bracket pair.
int check_constraints(const rp_pair* pairs, const rp_constraint* cons, int n_pairs, std::string* msg) {
  if (!cons) return RP_OK;
  char buf[200];
  auto bad = [&](int p, int s, int pos, const char* what) {
    std::snprintf(buf, sizeof buf, "pair %d, c%d, position %d: %s", p, s + 1, pos, what);
    if (msg) *msg = buf;
    return RP_ERR_ARG;
  };
  for (int p = 0; p < n_pairs; p++) {
    const char* cs[2] = {cons[p].c1, cons[p].c2};
    const int ns[2] = {pairs[p].n1, pairs[p].n2};
    std::vector<int> inter[2];   // positions of '[' in c1 / ']' in c2
    for (int s = 0; s < 2; s++) {
      const char* c = cs[s];
      if (!c) continue;
      const size_t len = strnlen(c, (size_t)ns[s] + 1);
      if (len != (size_t)ns[s]) {
        char what[96];
        std::snprintf(what, sizeof what, "the string is %s than s%d (%d nt)", len < (size_t)ns[s] ? "shorter" : "longer",
                      s + 1, ns[s]);
        return bad(p, s, (int)std::min(len, (size_t)ns[s]) + 1, what);
      }
      std::vector<int> open;
      for (int i = 0; i < ns[s]; i++) {
        switch (c[i]) {
          case '.': case 'x': break;
          case '(': open.push_back(i); break;
          case ')':
            if (open.empty()) return bad(p, s, i + 1, "')' closes no '('");
            open.pop_back();
            break;
          case '[':
            if (s == 1) return bad(p, s, i + 1, "'[' (an intermolecular pair's s1 end) may appear in c1 only");
            inter[s].push_back(i);
            break;
          case ']':
            if (s == 0) return bad(p, s, i + 1, "']' (an intermolecular pair's s2 end) may appear in c2 only");
            inter[s].push_back(i);
            break;
          default: {
            char what[64];
            std::snprintf(what, sizeof what, "character '%c' (code %d) is not one of .x()[]", std::isprint((unsigned char)c[i]) ? c[i] : '?',
                          (unsigned char)c[i]);
            return bad(p, s, i + 1, what);
          }
        }
      }
      if (!open.empty()) return bad(p, s, open.back() + 1, "'(' is never closed");
    }
    const size_t k1 = inter[0].size(), k2 = inter[1].size();
    if (k1 > k2) return bad(p, 0, inter[0][k1 - 1 - k2] + 1, "'[' has no partner ']' in c2");
    if (k2 > k1) return bad(p, 1, inter[1][k1] + 1, "']' has no partner '[' in c1");
  }
  return RP_OK;
}

// Stacking pseudo-energies: e1 over s1, e2 over s2, in kcal/mol (either may be null).
int check_stack_energies(const rp_pair* pairs, const rp_stack_energy* se, int n_pairs, std::string* msg) {
  if (!se) return RP_OK;
  for (int p = 0; p < n_pairs; p++) {
    const double* es[2] = {se[p].e1, se[p].e2};
    const int ns[2] = {pairs[p].n1, pairs[p].n2};
    for (int s = 0; s < 2; s++) {
      if (!es[s]) continue;
      for (int i = 0; i < ns[s]; i++)
        if (!std::isfinite(es[s][i])) {
          char buf[160];
          std::snprintf(buf, sizeof buf, "pair %d, e%d, position %d: %g kcal/mol is not finite", p, s + 1, i + 1, es[s][i]);
          if (msg) *msg = buf;
          return RP_ERR_ARG;
        }
    }
  }
  return RP_OK;
}

namespace {
// A pseudo-energy in kcal/mol as an integer number of 0.01 kcal/mol, half away from zero (as ViennaRNA stores
// soft-constraint energies): the one rounding of every pseudo-energy the stage takes.
double cal_units(double kcal) { return std::round(kcal * 100.0); }

int unpaired_not_finite(int p, int s, int i, double v, std::string* msg) {
  char buf[160];
  std::snprintf(buf, sizeof buf, "pair %d, u%d, position %d: %g kcal/mol is not finite", p, s + 1, i + 1, v);
  if (msg) *msg = buf;
  return RP_ERR_ARG;
}
}  // namespace

// Unpaired pseudo-energies: u1 over s1, u2 over s2, in kcal/mol (either may be null).  After rounding, a problem's
// weights move by at most a factor e^B either way against the same problem without data, B = sum_x |E_x| 10 / kT over
// the bases it applies; pf_scale is global, so B must leave the tables room in fp64 (UNPAIRED_MAX_B).
int check_unpaired_energies(const rp_pair* pairs, const rp_unpaired_energy* ue, int n_pairs, const rp_opts* opts,
                            std::string* msg) {
  if (!ue) return RP_OK;
  const double kT = (37.0 + RP_K0) * RP_GASCONST;
  char buf[200];
  for (int p = 0; p < n_pairs; p++) {
    const double* us[2] = {ue[p].u1, ue[p].u2};
    const int ns[2] = {pairs[p].n1, pairs[p].n2};
    double B[2] = {0., 0.};
    for (int s = 0; s < 2; s++) {
      if (!us[s]) continue;
      for (int i = 0; i < ns[s]; i++) {
        if (!std::isfinite(us[s][i])) return unpaired_not_finite(p, s, i, us[s][i], msg);
        B[s] += std::fabs(cal_units(us[s][i])) * 10.0 / kT;
      }
    }
    // s1's fold takes u1, s2's u2, the co-fold both (not under --duplex)
    const bool cofold = pairs[p].n2 > 0 && !opts->use_pf_duplex;
    const double Bs[3] = {B[0], B[1], cofold ? B[0] + B[1] : 0.};
    const char* names[3] = {"s1", "s2", "s1&s2"};
    for (int w = 0; w < 3; w++)
      if (Bs[w] > UNPAIRED_MAX_B) {
        std::snprintf(buf, sizeof buf,
                      "pair %d, problem %s: the unpaired pseudo-energies give B = sum |E| / kT = %.2f, beyond ln 10^150 "
                      "= %.2f, the range a batch's global pf_scale leaves",
                      p, names[w], Bs[w], UNPAIRED_MAX_B);
        if (msg) *msg = buf;
        return RP_ERR_UNSUPPORTED;
      }
  }
  return RP_OK;
}

int check_unpaired_finite(const rp_pair* pairs, const rp_unpaired_energy* ue, int n_pairs, std::string* msg) {
  if (!ue) return RP_OK;
  for (int p = 0; p < n_pairs; p++) {
    const double* us[2] = {ue[p].u1, ue[p].u2};
    const int ns[2] = {pairs[p].n1, pairs[p].n2};
    for (int s = 0; s < 2; s++)
      for (int i = 0; us[s] && i < ns[s]; i++)
        if (!std::isfinite(us[s][i])) return unpaired_not_finite(p, s, i, us[s][i], msg);
  }
  return RP_OK;
}

int check_samples(const rp_pair* pairs, int n_pairs, const rp_opts* opts, const rp_sample_opts* so, std::string* msg) {
  if (!so) return RP_OK;
  char buf[160];
  if (so->num < 0) {
    std::snprintf(buf, sizeof buf, "sample count %d is negative", so->num);
    if (msg) *msg = buf;
    return RP_ERR_ARG;
  }
  if (so->problems & ~(RP_SAMPLE_S1 | RP_SAMPLE_S2 | RP_SAMPLE_COFOLD)) {
    std::snprintf(buf, sizeof buf, "unknown bits 0x%x in the sampled problems", so->problems & ~7);
    if (msg) *msg = buf;
    return RP_ERR_ARG;
  }
  if (so->num > 0) {   // the sample buffer's size, and its size in bytes, must fit size_t (rp_sample_plan)
    std::vector<rp_sample_layout> lay(n_pairs > 0 ? n_pairs : 1);
    size_t total = 0;
    if (rp_sample_plan(pairs, n_pairs, so, lay.data(), &total) != RP_OK) {
      std::snprintf(buf, sizeof buf, "%d samples of the requested problems overflow the sample buffer's size", so->num);
      if (msg) *msg = buf;
      return RP_ERR_ARG;
    }
  }
  if (so->num > 0 && (so->problems & RP_SAMPLE_COFOLD) && opts->use_pf_duplex)
    for (int p = 0; p < n_pairs; p++)
      if (pairs[p].n2 > 0) {
        std::snprintf(buf, sizeof buf, "pair %d: --duplex has no co-fold ensemble to sample", p);
        if (msg) *msg = buf;
        return RP_ERR_UNSUPPORTED;
      }
  return RP_OK;
}

namespace {
// Stacking factors of one strand of length m from its pseudo-energies e[0..m-1] (kcal/mol): each value rounded to an
// integer number of 0.01 kcal/mol, half away from zero (as ViennaRNA stores soft-constraint energies), then
// f[i] = exp(-E_i * 10 / kT) at 37 C, the Boltzmann factor of every other integer energy of the model (dev_model.cpp).
// Returns whether any rounded value differs from 0 (whether the data changes anything).
bool fill_stack(const double* e, int m, double* f) {
  if (!e) return false;
  const double kT = (37.0 + RP_K0) * RP_GASCONST;
  bool any = false;
  for (int i = 1; i <= m; i++) {
    const double E = cal_units(e[i - 1]);
    f[i] = std::exp(-E * 10.0 / kT);
    any |= E != 0.;
  }
  return any;
}

// Pair factors of one strand of length m from its unpaired pseudo-energies u[0..m-1] (kcal/mol), rounded as fill_stack
// rounds: g[i] = exp(+E_i * 10 / kT), the inverse of the unpaired factor f (pair_sc, mcc_core.h), and *lnf = sum_i
// ln f(i) = -sum_i E_i * 10 / kT, what the data add to log Z.  Returns whether any rounded value differs from 0.
bool fill_unpaired(const double* u, int m, double* g, double* lnf) {
  *lnf = 0.;
  if (!u) return false;
  const double kT = (37.0 + RP_K0) * RP_GASCONST;
  bool any = false;
  for (int i = 1; i <= m; i++) {
    const double E = cal_units(u[i - 1]);
    g[i] = std::exp(E * 10.0 / kT);
    *lnf -= E * 10.0 / kT;
    any |= E != 0.;
  }
  return any;
}

// Keys of one problem of length m from its bracket pairs: partner[i] = j for the ends of a bracket pair (i,j), 0 for a
// base left free, -1 for a base kept unpaired (1-based).  Bracket pair number t (from 1, in the order they open) gets
// 2t+1 at both ends, a free base 2t for the innermost bracket pair around it (0 for none), an unpaired base
// 0x8000 + i, which no other base carries: then pair (i,j) is allowed iff key[i] == key[j].  n <= RP_MAX_N keeps
// every key below 2^16.  Returns whether any key differs from 0 (whether the constraint removes any pair).
bool fill_keys(const std::vector<int>& partner, int m, uint16_t* key) {
  std::vector<int> open;   // numbers of the bracket pairs around the current base
  int count = 0;
  bool any = false;
  for (int i = 1; i <= m; i++) {
    const int q = partner[i];
    int k;
    if (q < 0) k = 0x8000 + i;
    else if (q > i) { open.push_back(++count); k = 2 * count + 1; }
    else if (q > 0) { k = key[q]; open.pop_back(); }
    else k = open.empty() ? 0 : 2 * open.back();
    key[i] = (uint16_t)k;
    any |= k != 0;
  }
  return any;
}

// partners of the ( ) pairs of constraint string c (n bases), the bases of `unpaired` kept unpaired
void intra_partners(const char* c, int n, const char* unpaired, std::vector<int>& partner) {
  partner.assign(n + 1, 0);
  if (!c) return;
  std::vector<int> open;
  for (int i = 1; i <= n; i++) {
    if (c[i - 1] == '(') open.push_back(i);
    else if (c[i - 1] == ')') { partner[i] = open.back(); partner[open.back()] = i; open.pop_back(); }
    else if (std::strchr(unpaired, c[i - 1])) partner[i] = -1;
  }
}

// Keys of the three problems of a pair (s1 at k1[1..n1], s2 at k2[1..n2], the co-fold at k12[1..n1+n2]) from its
// constraint strings c1, c2 (either may be null), and in con[w] whether problem w is restricted.  `cofold`: the co-fold
// is constrained (not under --duplex, and n2 > 0).
void pair_keys(const rp_pair& pr, const char* c1, const char* c2, bool cofold, uint16_t* k1, uint16_t* k2, uint16_t* k12,
               int con[3]) {
  std::vector<int> partner;
  intra_partners(c1, pr.n1, "x[", partner);
  con[0] = fill_keys(partner, pr.n1, k1);
  intra_partners(c2, pr.n2, "x]", partner);
  con[1] = fill_keys(partner, pr.n2, k2);
  // s1&s2: the k-th '[' from the 3' end of c1 with the k-th ']' from the 5' end of c2
  const int n12 = pr.n1 + pr.n2;
  partner.assign(n12 + 1, 0);
  std::vector<int> ends;
  for (int i = pr.n1; i >= 1; i--)
    if (c1 && c1[i - 1] == '[') ends.push_back(i);
  size_t k = 0;
  for (int j = 1; j <= pr.n2; j++)
    if (c2 && c2[j - 1] == ']') { partner[ends[k]] = pr.n1 + j; partner[pr.n1 + j] = ends[k]; k++; }
  for (int i = 1; i <= n12; i++) {
    const char ch = i <= pr.n1 ? (c1 ? c1[i - 1] : '.') : (c2 ? c2[i - pr.n1 - 1] : '.');
    if (ch == 'x' || ch == '(' || ch == ')') partner[i] = -1;
  }
  con[2] = cofold && fill_keys(partner, n12, k12);
}
}  // namespace

}  // namespace rp

using rp::Problem;

extern "C" {

int rp_kernel_plan(int n, size_t smem_limit, size_t* smem_bytes) {
  if (smem_limit == 0) smem_limit = 232448;
  const size_t half_sm = (smem_limit + 1024) / 2 - 1024;   // two CTAs per SM, 1 KB reserved each
  if (n < 1) n = 1;
  const size_t s256 = rp::band_shared_bytes(n, 256, true), s512 = rp::band_shared_bytes(n, 512, true);
  if (s256 <= half_sm) { if (smem_bytes) *smem_bytes = s256; return RP_KERNEL_BAND_2CTA; }
  if (smem_bytes) *smem_bytes = s512;
  if (s512 <= smem_limit) return RP_KERNEL_BAND_1CTA;
  return n >= rp::MCC_LONG_N ? RP_KERNEL_GENERAL_WIDE : RP_KERNEL_GENERAL;
}

int rp_dense_plan(const rp_pair* pairs, int n_pairs, const rp_opts* opts, rp_dense_layout* layout,
                  size_t* total_floats) {
  int rc = rp::check_pairs(pairs, n_pairs, opts);
  if (rc) return rc;
  const size_t w = opts->max_w > 0 ? (size_t)opts->max_w : 0;
  size_t off = 0;
  for (int p = 0; p < n_pairs; p++) {
    rp_dense_layout l;
    l.n_bp1 = rp::bp_len(pairs[p].n1); l.n_bp2 = rp::bp_len(pairs[p].n2);
    l.n_up1 = (size_t)pairs[p].n1 * w; l.n_up2 = (size_t)pairs[p].n2 * w;
    l.n_hp = (size_t)(pairs[p].n1 + 1) * (size_t)(pairs[p].n2 + 1);
    l.bp1 = off; off += l.n_bp1;
    l.bp2 = off; off += l.n_bp2;
    l.up1 = off; off += l.n_up1;
    l.up2 = off; off += l.n_up2;
    l.hp = off; off += l.n_hp;
    if (layout) layout[p] = l;
  }
  if (total_floats) *total_floats = off;
  return RP_OK;
}

int rp_square_plan(const rp_pair* pairs, int n_pairs, const rp_opts* opts, rp_square_layout* layout) {
  int rc = rp::check_pairs(pairs, n_pairs, opts);
  if (rc) return rc;
  if (!layout) return RP_ERR_ARG;
  rp_square_layout s = {};
  s.B = n_pairs;
  s.W = std::max(opts->max_w, 0);
  for (int p = 0; p < n_pairs; p++) {
    s.N1 = std::max(s.N1, pairs[p].n1);
    s.N2 = std::max(s.N2, pairs[p].n2);
  }
  // B * rows * cols elements, and their size in bytes, must fit size_t
  bool overflow = false;
  auto count = [&](size_t rows, size_t cols) {
    size_t n = 0;
    overflow |= __builtin_mul_overflow((size_t)s.B, rows, &n) || __builtin_mul_overflow(n, cols, &n) ||
                n > SIZE_MAX / sizeof(float);
    return n;
  };
  const size_t m1 = (size_t)s.N1 + 1, m2 = (size_t)s.N2 + 1;
  s.n_bp1 = count(m1, m1);
  s.n_bp2 = count(m2, m2);
  s.n_up1 = count(s.N1, s.W);
  s.n_up2 = count(s.N2, s.W);
  s.n_hp = count(m1, m2);
  if (overflow) return RP_ERR_ARG;
  *layout = s;
  return RP_OK;
}

int rp_sample_plan(const rp_pair* pairs, int n_pairs, const rp_sample_opts* so, rp_sample_layout* per_pair, size_t* total) {
  if (!pairs || n_pairs < 0 || !so || so->num < 0 || !total || (n_pairs > 0 && !per_pair)) return RP_ERR_ARG;
  size_t off = 0;
  bool overflow = false;
  // num pair tables of n int16 each, or none; the running offset and its size in bytes must fit size_t
  auto take = [&](bool on, size_t n, size_t* at, size_t* len) {
    size_t m = 0;
    if (on) overflow |= __builtin_mul_overflow((size_t)so->num, n, &m);
    *at = off;
    *len = m;
    overflow |= __builtin_add_overflow(off, m, &off) || off > SIZE_MAX / sizeof(int16_t);
  };
  for (int p = 0; p < n_pairs; p++) {
    const size_t n1 = (size_t)std::max(pairs[p].n1, 0), n2 = (size_t)std::max(pairs[p].n2, 0);
    rp_sample_layout& L = per_pair[p];
    take((so->problems & RP_SAMPLE_S1) != 0, n1, &L.s1, &L.len_s1);
    take((so->problems & RP_SAMPLE_S2) != 0, n2, &L.s2, &L.len_s2);
    take((so->problems & RP_SAMPLE_COFOLD) != 0 && n2 > 0, n1 + n2, &L.co, &L.len_co);
  }
  if (overflow) return RP_ERR_ARG;
  *total = off;
  return RP_OK;
}

int rp_shape_deigan(const double* r, int n, double slope, double intercept, double* e) {
  if (n < 0 || (n > 0 && (!r || !e))) return RP_ERR_ARG;
  for (int i = 0; i < n; i++) e[i] = r[i] >= 0. ? slope * std::log(r[i] + 1.) + intercept : 0.;   // r < 0, NaN: missing
  return RP_OK;
}

int rp_sparse_plan(const rp_pair* pairs, int n_pairs, const rp_opts* opts, rp_sparse_layout* layout, size_t* total_recs,
                   size_t* total_floats) {
  int rc = rp::check_pairs(pairs, n_pairs, opts);
  if (rc) return rc;
  const size_t w = opts->max_w > 0 ? (size_t)opts->max_w : 0;
  // Each base pairs with total probability <= 1, so fewer than 1/th partners
  // exceed th: at most n/(2 th) pairs inside one RNA, min(n1,n2)/th across.
  auto cap_in = [&](int n) -> size_t {
    size_t all = (size_t)n * (size_t)(n - 1) / 2;
    if (!(opts->th_ss > 0.f)) return all;
    return std::min(all, (size_t)std::floor(n / (2.0 * opts->th_ss)) + 1);
  };
  size_t roff = 0, foff = 0;
  for (int p = 0; p < n_pairs; p++) {
    rp_sparse_layout l;
    l.cap_x = cap_in(pairs[p].n1);
    l.cap_y = cap_in(pairs[p].n2);
    size_t all = (size_t)pairs[p].n1 * (size_t)pairs[p].n2;
    l.cap_z = !(opts->th_hy > 0.f) ? all
                                   : std::min(all, (size_t)std::min(pairs[p].n1, pairs[p].n2) *
                                                       ((size_t)std::floor(1.0 / opts->th_hy) + 1));
    // accessible regions: one variable per (start, length) with length in min_w..max_w, when the
    // reference creates them at all (enable_accessibility, src/ractip.cpp:526)
    const bool acc = opts->min_w > 1 && opts->max_w >= opts->min_w;
    const size_t nlen = acc ? (size_t)(opts->max_w - opts->min_w + 1) : 0;
    l.cap_v = (size_t)pairs[p].n1 * nlen;
    l.cap_w = (size_t)pairs[p].n2 * nlen;
    l.x = roff; roff += l.cap_x;
    l.y = roff; roff += l.cap_y;
    l.z = roff; roff += l.cap_z;
    l.v = roff; roff += l.cap_v;
    l.w = roff; roff += l.cap_w;
    l.n_up1 = (size_t)pairs[p].n1 * w; l.n_up2 = (size_t)pairs[p].n2 * w;
    l.up1 = foff; foff += l.n_up1;
    l.up2 = foff; foff += l.n_up2;
    if (layout) layout[p] = l;
  }
  if (total_recs) *total_recs = roff;
  if (total_floats) *total_floats = foff;
  return RP_OK;
}

static double alg_flops_mcc_uncached(int n);
double rp_alg_flops_mcc(int n) {
  // memoised: the O(n^2) count below used to be recomputed for all 3 problems of every pair of
  // every one-shot call (tens of milliseconds per 1000-pair batch, more than the copies)
  static thread_local std::vector<std::pair<int, double>> memo;
  for (const auto& kv : memo)
    if (kv.first == n) return kv.second;
  const double v = alg_flops_mcc_uncached(n);
  if (memo.size() < 4096) memo.emplace_back(n, v);
  return v;
}
static double alg_flops_mcc_uncached(int n) {
  // SURVEY.md 8(d): F_mcc(n) = 6 I(n) + 2 S_in(n) + 2 S_out(n), TURN=3, MAXLOOP=30
  if (n < 5) return 0.;
  double I = 0, Sin = 0, Sout = 0;
  for (int d = 4; d <= n - 1; d++) {
    const int m = std::min(30, d - 6);
    if (m >= 0) I += (double)(n - d) * (m + 1) * (m + 2) / 2.0;
    Sin += (double)(n - d) * ((d - 2) + d + d);
  }
  for (int l = 5; l <= n; l++)
    for (int k = 2; k <= l - 4; k++) Sout += std::max(0, n - l - 1) + (k - 2);
  return 6. * I + 2. * Sin + 2. * Sout;
}

}  // extern "C"

namespace rp {

int plan_batch(const rp_pair* pairs, int n_pairs, const rp_opts* opts, const DeviceFacts& dev, const RouteSettings& rs,
               BatchPlan* out, const rp_constraint* cons, const rp_stack_energy* se, const rp_sample_opts* so,
               const rp_unpaired_energy* ue) {
  BatchPlan& b = *out;
  b = BatchPlan{};
  // sampled problems (CON_SAMPLE): those with room in the sample buffer
  if (so && so->num > 0) {
    b.sample_layout.resize(n_pairs);
    rp_sample_plan(pairs, n_pairs, so, b.sample_layout.data(), &b.sample_total);   // cannot fail: check_samples
    b.sample_num = so->num;
    b.sample_seed = so->seed;
  }
  size_t mem = 0;   // DeviceFacts::memory, asked once
  auto memory = [&]() {
    if (!mem) mem = std::max<size_t>(1, dev.memory());
    return mem;
  };
  b.layout.resize(n_pairs);
  rp_dense_plan(pairs, n_pairs, opts, b.layout.data(), &b.total_floats);

  // problems and their encoded sequences: per pair  0 s1 0 s2 0 s1s2 0
  size_t bytes = 0;
  for (int p = 0; p < n_pairs; p++) bytes += 2 * ((size_t)pairs[p].n1 + pairs[p].n2) + 4;
  std::vector<uint8_t>& seq = b.seq;
  seq.reserve(bytes + 16);
  std::vector<uint16_t>& key = b.key;   // (filled only for batches with constraints, then dropped if none restricts)
  bool any_constrained = false;
  std::vector<double>& stack = b.stack;   // (the same for the stacking factors)
  bool any_stack = false;
  std::vector<double>& unp = b.unpaired;   // (and for the unpaired pseudo-energies' pair factors)
  bool any_unp = false;
  const int w = opts->max_w > 0 ? opts->max_w : 0;
  size_t ws_need = 0;
  for (int p = 0; p < n_pairs; p++) {
    const rp_pair& pr = pairs[p];
    const rp_dense_layout& L = b.layout[p];
    seq.push_back(0);
    const int off1 = (int)seq.size();
    for (int i = 0; i < pr.n1; i++) seq.push_back(encode_base(pr.s1[i]));
    seq.push_back(0);
    const int off2 = (int)seq.size();
    for (int i = 0; i < pr.n2; i++) seq.push_back(encode_base(pr.s2[i]));
    seq.push_back(0);
    const int off12 = (int)seq.size();
    for (int i = 0; i < pr.n1; i++) seq.push_back(encode_base(pr.s1[i]));
    for (int i = 0; i < pr.n2; i++) seq.push_back(encode_base(pr.s2[i]));
    seq.push_back(0);
    int con[3] = {0, 0, 0};   // s1, s2, s1&s2 restricted by the constraint
    if (cons && (cons[p].c1 || cons[p].c2)) {
      key.resize(seq.size(), 0);
      // --duplex: the co-fold is unconstrained
      pair_keys(pr, cons[p].c1, cons[p].c2, pr.n2 > 0 && !opts->use_pf_duplex, &key[off1 - 1], &key[off2 - 1],
                &key[off12 - 1], con);
      any_constrained |= con[0] || con[1] || con[2];
    }
    // stacking pseudo-energies: s1's fold takes e1, s2's e2, the co-fold both (stack_sc, mcc_core.h, leaves out the
    // stacks that join the strands); --duplex takes none
    int stk[2] = {0, 0};
    if (se && (se[p].e1 || se[p].e2)) {
      stack.resize(seq.size(), 1.0);
      stk[0] = fill_stack(se[p].e1, pr.n1, &stack[off1 - 1]) ? CON_STACK : 0;
      stk[1] = fill_stack(se[p].e2, pr.n2, &stack[off2 - 1]) ? CON_STACK : 0;
      std::copy(&stack[off1], &stack[off1] + pr.n1, &stack[off12]);
      std::copy(&stack[off2], &stack[off2] + pr.n2, &stack[off12] + pr.n1);
      any_stack |= stk[0] || stk[1];
    }
    // unpaired pseudo-energies: s1's fold takes u1, s2's u2, the co-fold both (pair_sc, mcc_core.h, gives the pairs
    // that join the strands no factor); --duplex takes none
    int unf[2] = {0, 0};
    double lnf[2] = {0., 0.};
    if (ue && (ue[p].u1 || ue[p].u2)) {
      unp.resize(seq.size(), 1.0);
      b.unpaired_lz.resize(3 * (size_t)n_pairs, 0.);
      unf[0] = fill_unpaired(ue[p].u1, pr.n1, &unp[off1 - 1], &lnf[0]) ? CON_UNPAIRED : 0;
      unf[1] = fill_unpaired(ue[p].u2, pr.n2, &unp[off2 - 1], &lnf[1]) ? CON_UNPAIRED : 0;
      std::copy(&unp[off1], &unp[off1] + pr.n1, &unp[off12]);
      std::copy(&unp[off2], &unp[off2] + pr.n2, &unp[off12] + pr.n1);
      b.unpaired_lz[3 * (size_t)p] = lnf[0];
      b.unpaired_lz[3 * (size_t)p + 1] = lnf[1];
      b.unpaired_lz[3 * (size_t)p + 2] = lnf[0] + lnf[1];
      any_unp |= unf[0] || unf[1];
    }
    Problem q;
    std::memset(&q, 0, sizeof q);
    q.pair = p; q.max_w = w; q.n1 = pr.n1; q.n2 = pr.n2; q.th_hy = opts->th_hy;
    q.out_bp = q.out_up = q.out_hp = -1;
    q.ws_off = -1;
    // rnafold(fa1, ...), rnafold(fa2, ...)  src/ractip.cpp:546-547
    Problem a = q;
    const rp_sample_layout* sl = b.sample_total ? &b.sample_layout[p] : nullptr;
    a.kind = KIND_LINEAR; a.which = 0; a.seq_off = off1; a.n = pr.n1; a.cp = 0; a.constrained = con[0] | stk[0] | unf[0];
    if (sl && sl->len_s1) a.constrained |= CON_SAMPLE;
    a.out_bp = (long long)L.bp1; a.out_up = w > 0 ? (long long)L.up1 : -1;
    b.probs.push_back(a);
    a.which = 1; a.seq_off = off2; a.n = pr.n2; a.constrained = con[1] | stk[1] | unf[1];
    if (sl && sl->len_s2) a.constrained |= CON_SAMPLE;
    a.out_bp = (long long)L.bp2; a.out_up = w > 0 ? (long long)L.up2 : -1;
    b.probs.push_back(a);
    if (pr.n2 == 0) {   // a lone sequence (RactIP::rnafold on its own, src/ractip.cpp:1599-1601): no second fold, no hybridization
      Problem none = q;
      none.kind = KIND_LINEAR; none.which = 2; none.n = 0;
      b.probs.push_back(none);
      b.alg_flops += rp_alg_flops_mcc(pr.n1);
      b.has_single = true;
      continue;
    }
    // rnaduplex(fa1, fa2, hp_)  src/ractip.cpp:548
    Problem c = q;
    c.which = 2; c.seq_off = off12; c.out_hp = (long long)L.hp;
    if (opts->use_pf_duplex) {
      c.kind = KIND_DUPLEX; c.n = pr.n1 + pr.n2; c.cp = pr.n1 + 1;
      b.n_duplex++;
      ws_need = std::max(ws_need, 2 * (size_t)(pr.n1 + 2) * (size_t)(pr.n2 + 2));
    } else {
      c.kind = KIND_COFOLD; c.n = pr.n1 + pr.n2; c.cp = pr.n1 + 1; c.constrained = con[2] | stk[0] | stk[1] | unf[0] | unf[1];
      if (sl && sl->len_co) c.constrained |= CON_SAMPLE;
      b.alg_flops += rp_alg_flops_mcc(c.n);
    }
    b.probs.push_back(c);
    b.alg_flops += rp_alg_flops_mcc(pr.n1) + rp_alg_flops_mcc(pr.n2);
  }
  if (any_constrained) key.resize(seq.size(), 0);
  else std::vector<uint16_t>().swap(key);
  if (any_stack) stack.resize(seq.size(), 1.0);
  else std::vector<double>().swap(stack);
  if (any_unp) {
    unp.resize(seq.size(), 1.0);
  } else {
    std::vector<double>().swap(unp);
    std::vector<double>().swap(b.unpaired_lz);
  }

  // Band class of a problem: 0 = L (512 threads, ring needs more than half an SM), 1 = S (256 threads, 2 CTAs/SM),
  // -1 = the general kernel, which alone applies structure constraints, stacking and unpaired pseudo-energies and samples.
  auto cls = [&](const Problem& q) {
    if (!rs.band || q.kind == KIND_DUPLEX || q.constrained) return -1;
    const int k = rp_kernel_plan(q.n, dev.smem_optin, nullptr);
    return k >= RP_KERNEL_GENERAL ? -1 : k;
  };
  // LPT cost.  Band-kernel lengths (measured, profiles/r01b_phase_ablation.txt): ~30 k cycles per unit of
  // length for the two wavefronts (fixed cost per diagonal) + ~160 n^2 for the unpaired-window pass.
  auto cost = [&](const Problem& q) {
    if (q.kind == KIND_DUPLEX) return 0.0;
    if (cls(q) >= 0) return 3.0e4 * q.n + ((q.kind == KIND_LINEAR && q.max_w > 0) ? 160.0 * q.n * q.n : 0.0);
    return (double)q.n * q.n * (q.n + 1500.0);
  };
  // most expensive first (LPT), ties by index for determinism; then split into [class L | class S | general]
  std::vector<int> lpt;
  for (size_t k = 0; k < b.probs.size(); k++)
    if (b.probs[k].n > 0) lpt.push_back((int)k);
  std::stable_sort(lpt.begin(), lpt.end(), [&](int x, int y) { return cost(b.probs[x]) > cost(b.probs[y]); });
  std::vector<int> part[3];
  int band_maxn[2] = {0, 0};
  for (int k : lpt) {
    const int c = cls(b.probs[k]);
    part[c < 0 ? 2 : c].push_back(k);
    if (c >= 0) band_maxn[c] = std::max(band_maxn[c], b.probs[k].n);
  }
  b.n_band[0] = (int)part[0].size();
  b.n_band[1] = (int)part[1].size();
  b.n_general = (int)part[2].size();

  // Unpaired-window passes of the band classes, three ways:
  //   mode 1 (large batches, >= 4.5 single-strand problems per SM): a launch of their own after the wavefront kernels
  //           (unstru_kernel: one 768-thread CTA per SM -- the pass needs no shared-memory ring, and the tables of 148
  //           resident problems stay in the L2);
  //   mode 2 (batches with at least three problems per SM): JOBS of their own in the band kernel's queue, after all
  //           wavefront jobs, each waiting for its problem's completion flag -- finer jobs shorten the tail;
  //   mode 0 (a handful of problems, or no room for private workspaces): fused with the wavefronts.
  // (measured, MicA x ompA shuffles, kernel ms fused / own launch / jobs of their own: 125 pairs 5.09 / 5.13 / 5.29,
  //  180 pairs 7.70 / 8.05 / 7.15, 250 pairs 10.40 / 9.89 / 9.83, 350 pairs 13.94 / 13.34 / 13.45, 500 pairs - / 18.3 / 19.1,
  //  1000 pairs 39.0 / 36.2 / -)
  std::vector<int> up;
  int up_maxn = 0;
  for (int c = 0; c < 2; c++)
    for (int k : part[c]) {
      const Problem& q = b.probs[k];
      if (q.kind == KIND_LINEAR && q.max_w > 0 && q.out_up >= 0) { up.push_back(k); up_maxn = std::max(up_maxn, q.n); }
    }
  const size_t up_slot = up.empty() ? 0 : slot_doubles(up_maxn);
  const size_t up_bytes = up_slot * sizeof(double) * up.size();
  if (!up.empty() && (double)up_bytes <= 24e9) {
    if (2 * (int)up.size() >= 9 * dev.sm_count && dev.up_ctas_per_sm > 0) b.up_mode = 1;
    else if (b.n_band[0] + b.n_band[1] >= 3 * dev.sm_count) b.up_mode = 2;
    // the private workspaces are part of the context's workspace; if the device cannot hold them, the pass stays fused
    if (b.up_mode && up_bytes > dev.ws_bytes && up_bytes > memory() / 10 * 6) b.up_mode = 0;
  }
  if (b.up_mode) {
    b.n_defer = (int)up.size();
    b.defer_slot = up_slot;
    for (size_t k = 0; k < up.size(); k++) {
      b.probs[up[k]].defer_up = 1;
      b.probs[up[k]].ws_off = (long long)(k * up_slot);
    }
    // the deferred passes, costliest (longest) first
    std::stable_sort(up.begin(), up.end(), [&](int x, int y) { return b.probs[x].n > b.probs[y].n; });
  }
  for (int c = 0; c < 2; c++) {
    if (b.up_mode == 2) {
      // wavefront jobs with a dependent job first (their successor should start early), then the others, then the
      // unpaired-window jobs
      for (int k : part[c])
        if (b.probs[k].defer_up) b.order.push_back(k);
      for (int k : part[c])
        if (!b.probs[k].defer_up) b.order.push_back(k);
      for (int k : up)
        if (cls(b.probs[k]) == c) b.order.push_back(k | RP_JOB_UNPAIRED);
      b.n_band[c] = (int)b.order.size() - (c ? b.n_band[0] : 0);
    } else {
      b.order.insert(b.order.end(), part[c].begin(), part[c].end());
    }
  }
  b.order.insert(b.order.end(), part[2].begin(), part[2].end());
  if (b.up_mode == 1) b.order.insert(b.order.end(), up.begin(), up.end());   // queue of unstru_kernel

  // general kernel: build, grid and workspace slots
  int gen_maxn = 0;
  for (int k : part[2])
    if (b.probs[k].kind != KIND_DUPLEX) { gen_maxn = std::max(gen_maxn, b.probs[k].n); b.n_mcc++; }
  b.slot_doubles = std::max(b.n_mcc ? slot_doubles(gen_maxn) : (size_t)0, ws_need);
  b.mcc_minb = (gen_maxn >= rs.mcc_long_n && dev.ctas_per_sm1 > 0) ? 1 : 2;
  if (b.n_general > 0) {
    const size_t slot_bytes = std::max<size_t>(b.slot_doubles * sizeof(double), 8);
    int g = dev.sm_count * std::max(1, b.mcc_minb >= 2 ? dev.ctas_per_sm : dev.ctas_per_sm1);
    g = std::min(g, b.n_general);
    // keep the workspace within a budget (long sequences: fewer, fatter slots)
    if ((size_t)g * slot_bytes > dev.ws_bytes) g = (int)std::min<size_t>(g, std::max<size_t>(1, memory() / 10 * 7 / slot_bytes));
    b.grid = g;
  }
  // Few long problems (a single long pair, not a shuffle batch): one problem per thread-block cluster, so
  // that its wavefront runs on several SMs -- 16 CTAs per problem while that leaves no cluster waiting,
  // 8 up to ~5 rounds of clusters.  Beyond that one CTA per problem has the higher throughput (a 1500-nt
  // problem: 57 ms on 16 SMs, 76 ms on 8, ~400 ms on one; DESIGN.md section 8).
  if (b.n_mcc > 0) {
    if (rs.cluster >= 0) b.cluster = rs.cluster;
    else if (b.n_mcc * 16 <= dev.sm_count) b.cluster = 16;                   // any general-kernel length (measured: one 250 x 100 pair 17.2 -> 9.3 ms)
    else if (b.n_mcc * 8 <= dev.sm_count * (b.mcc_minb == 1 ? 5 : 4)) b.cluster = 8;   // up to 4-5 rounds of clusters (20 pairs of 400 x 300: 87 -> 56 ms; 40 pairs: 93 vs 106 ms)
  }

  // band classes: grid = resident CTAs, one workspace slot each, placed after the general kernel's slots
  size_t ws = (size_t)b.grid * b.slot_doubles;
  for (int c = 0; c < 2; c++) {
    b.ws_band[c] = ws;
    if (!b.n_band[c]) continue;
    b.band_smem[c] = band_shared_bytes(band_maxn[c], BAND_THREADS[c], true);
    b.band_slot[c] = slot_doubles(band_maxn[c]);
    const int occ = dev.band_occupancy(BAND_THREADS[c], b.band_smem[c]);
    if (occ < 1) return RP_ERR_CUDA;
    b.band_grid[c] = std::min(b.n_band[c], dev.sm_count * occ);
    ws += (size_t)b.band_grid[c] * b.band_slot[c];
  }
  b.ws_up = ws;
  b.ws_doubles = ws + b.defer_slot * (size_t)b.n_defer;
  if (b.up_mode == 1) b.up_grid = std::min(b.n_defer, dev.sm_count * std::max(1, dev.up_ctas_per_sm));

  // the launch that carries most of the algorithmic flops (an unpaired-window job carries none)
  double f[3] = {0, 0, 0};
  const int cnt[3] = {b.n_band[0], b.n_band[1], b.n_general};
  for (int k = 0, x = 0; k < 3; x += cnt[k], k++)
    for (int y = x; y < x + cnt[k]; y++) {
      if (b.order[y] & RP_JOB_UNPAIRED) continue;
      const Problem& q = b.probs[b.order[y]];
      if (q.kind != KIND_DUPLEX) f[k] += rp_alg_flops_mcc(q.n);
    }
  b.dom_kind = f[0] >= f[1] && f[0] >= f[2] ? 0 : (f[1] >= f[2] ? 1 : 2);
  b.dom_flops = f[b.dom_kind];
  if (b.dom_flops <= 0) b.dom_kind = -1;

  // Split fetch.  The short band class runs last (side stream, on the SMs the long class leaves), so everything the
  // long class wrote can cross PCIe meanwhile.  Needs a uniform batch (the z-score shuffle batch: every pair has the
  // lengths of the original pair) so that the sections are strided 2-D copies.
  if (rs.split_fetch && rs.band && n_pairs >= 2 && b.n_band[0] > 0 && b.n_band[1] > 0 && b.n_general == 0) {
    bool uniform = true;
    for (int p = 1; p < n_pairs && uniform; p++) uniform = pairs[p].n1 == pairs[0].n1 && pairs[p].n2 == pairs[0].n2;
    if (uniform) {
      const rp_dense_layout& L = b.layout[0];
      b.pair_stride = b.layout[1].bp1 - L.bp1;
      auto is_short = [&](int n) { return rp_kernel_plan(n, dev.smem_optin, nullptr) == RP_KERNEL_BAND_2CTA; };
      const bool s1 = is_short(pairs[0].n1), s2 = is_short(pairs[0].n2), s12 = is_short(pairs[0].n1 + pairs[0].n2);
      struct Sec { size_t off, len; bool sh; };
      const bool late = b.up_mode == 1;   // the deferred unpaired-window launch writes the up sections last
      const Sec secs[5] = {{L.bp1, L.n_bp1, s1}, {L.bp2, L.n_bp2, s2}, {L.up1, L.n_up1, s1 || late}, {L.up2, L.n_up2, s2 || late}, {L.hp, L.n_hp, s12}};
      for (const Sec& x : secs) {   // sections are in layout order: merge neighbours of the same class
        if (!x.len) continue;
        auto& v = x.sh ? b.sect_short : b.sect_long;
        if (!v.empty() && v.back().first + v.back().second == x.off) v.back().second += x.len;
        else v.push_back({x.off - L.bp1, x.len});
      }
      b.split_fetch = !b.sect_long.empty() && !b.sect_short.empty();
    }
  }
  return RP_OK;
}

int check_mfe(const rp_pair* pairs, int n_pairs, const rp_constraint* cons, const rp_stack_energy* se,
              const rp_unpaired_energy* ue, int problems, std::string* msg) {
  const rp_opts o = {15, 5, 0.5f, 0.1f, 0.003f, 0};   // rp_opts plays no part; check_pairs only needs one
  if (check_pairs(pairs, n_pairs, &o)) {
    if (msg) *msg = "bad pairs";
    return RP_ERR_ARG;
  }
  for (int p = 0; p < n_pairs; p++)
    if ((long long)pairs[p].n1 + pairs[p].n2 > RP_MAX_N) {
      if (msg) *msg = "n1+n2 exceeds the 32-bit workspace indexing limit (12000 nt)";
      return RP_ERR_TOO_LONG;
    }
  if (problems & ~(RP_SAMPLE_S1 | RP_SAMPLE_S2 | RP_SAMPLE_COFOLD)) {
    char buf[96];
    std::snprintf(buf, sizeof buf, "unknown bits 0x%x in the requested problems", problems & ~7);
    if (msg) *msg = buf;
    return RP_ERR_ARG;
  }
  int rc;
  if ((rc = check_constraints(pairs, cons, n_pairs, msg)) != RP_OK) return rc;
  if ((rc = check_stack_energies(pairs, se, n_pairs, msg)) != RP_OK) return rc;
  return check_unpaired_finite(pairs, ue, n_pairs, msg);
}

int plan_mfe(const rp_pair* pairs, int n_pairs, const rp_constraint* cons, const rp_stack_energy* se,
             const rp_unpaired_energy* ue, int problems, const DeviceFacts& dev, MfePlan* out, std::string* msg) {
  MfePlan& m = *out;
  m = MfePlan{};
  rp_sample_opts so = {1, 0, problems};
  m.layout.resize(n_pairs);
  if (rp_sample_plan(pairs, n_pairs, &so, m.layout.data(), &m.total) != RP_OK) return RP_ERR_ARG;
  size_t bytes = 0;
  for (int p = 0; p < n_pairs; p++) bytes += 2 * ((size_t)pairs[p].n1 + pairs[p].n2) + 4;
  m.seq.reserve(bytes + 16);
  bool any_key = false, any_es = false, any_eu = false;
  const char* names[3] = {"s1", "s2", "s1&s2"};
  int maxn = 0;
  for (int p = 0; p < n_pairs; p++) {
    const rp_pair& pr = pairs[p];
    const rp_sample_layout& L = m.layout[p];
    m.seq.push_back(0);
    const int off1 = (int)m.seq.size();
    for (int i = 0; i < pr.n1; i++) m.seq.push_back(encode_base(pr.s1[i]));
    m.seq.push_back(0);
    const int off2 = (int)m.seq.size();
    for (int i = 0; i < pr.n2; i++) m.seq.push_back(encode_base(pr.s2[i]));
    m.seq.push_back(0);
    const int off12 = (int)m.seq.size();
    for (int i = 0; i < pr.n1; i++) m.seq.push_back(encode_base(pr.s1[i]));
    for (int i = 0; i < pr.n2; i++) m.seq.push_back(encode_base(pr.s2[i]));
    m.seq.push_back(0);
    int flags[3] = {0, 0, 0};
    if (cons && (cons[p].c1 || cons[p].c2)) {
      m.key.resize(m.seq.size(), 0);
      int con[3];
      pair_keys(pr, cons[p].c1, cons[p].c2, pr.n2 > 0, &m.key[off1 - 1], &m.key[off2 - 1], &m.key[off12 - 1], con);
      for (int w = 0; w < 3; w++) flags[w] |= con[w] ? CON_KEYS : 0;
    }
    // rounded pseudo-energies of s1 and s2, copied into the co-fold's concatenation; |E| summed per strand
    double sum[2][2] = {{0., 0.}, {0., 0.}};   // [strand][stack, unpaired]
    long long eu_sum[2] = {0, 0};
    auto fill = [&](std::vector<int32_t>& v, const double* e1, const double* e2, int kind, bool& any) {
      if (!e1 && !e2) return;
      v.resize(m.seq.size(), 0);
      const double* es[2] = {e1, e2};
      const int ns[2] = {pr.n1, pr.n2}, offs[2] = {off1, off2}, offc[2] = {off12, off12 + pr.n1};
      for (int s = 0; s < 2; s++)
        for (int i = 0; es[s] && i < ns[s]; i++) {
          const double E = cal_units(es[s][i]);
          sum[s][kind] += std::fabs(E);
          if (std::fabs(E) > MFE_MAX_PSEUDO) continue;   // rejected below; keeps the conversion defined
          v[offs[s] + i] = v[offc[s] + i] = (int32_t)E;
          if (kind) eu_sum[s] += (int32_t)E;
          if (E != 0.) {
            any = true;
            flags[s] |= kind ? CON_UNPAIRED : CON_STACK;
            flags[2] |= kind ? CON_UNPAIRED : CON_STACK;
          }
        }
    };
    if (se) fill(m.es, se[p].e1, se[p].e2, 0, any_es);
    if (ue) fill(m.eu, ue[p].u1, ue[p].u2, 1, any_eu);
    any_key |= (flags[0] | flags[1] | flags[2]) & CON_KEYS;
    const long long lens[3] = {(long long)L.len_s1, (long long)L.len_s2, (long long)L.len_co};
    const long long outs[3] = {(long long)L.s1, (long long)L.s2, (long long)L.co};
    const int offs[3] = {off1, off2, off12}, ns[3] = {pr.n1, pr.n2, pr.n1 + pr.n2};
    for (int w = 0; w < 3; w++) {
      if (!lens[w]) continue;
      const double total = w < 2 ? sum[w][0] + sum[w][1] : sum[0][0] + sum[0][1] + sum[1][0] + sum[1][1];
      if (total > MFE_MAX_PSEUDO) {
        char buf[200];
        std::snprintf(buf, sizeof buf,
                      "pair %d, problem %s: the pseudo-energies give sum |E| = %.2f kcal/mol, beyond %.2f kcal/mol, the "
                      "range of the MFE kernel's int32 energies",
                      p, names[w], total / 100.0, MFE_MAX_PSEUDO / 100.0);
        if (msg) *msg = buf;
        return RP_ERR_UNSUPPORTED;
      }
      MfeJob j;
      j.seq_off = offs[w];
      j.n = ns[w];
      j.cp = w == 2 ? pr.n1 + 1 : 0;
      j.flags = flags[w];
      j.out = outs[w];
      j.energy_at = 3 * p + w;
      j.eu_const = (int)(w < 2 ? eu_sum[w] : eu_sum[0] + eu_sum[1]);
      m.jobs.push_back(j);
      maxn = std::max(maxn, j.n);
    }
  }
  if (!any_key) std::vector<uint16_t>().swap(m.key);
  else m.key.resize(m.seq.size(), 0);
  if (!any_es) std::vector<int32_t>().swap(m.es);
  else m.es.resize(m.seq.size(), 0);
  if (!any_eu) std::vector<int32_t>().swap(m.eu);
  else m.eu.resize(m.seq.size(), 0);
  for (MfeJob& j : m.jobs) {   // a problem without nonzero data of a kind does not bind it
    if (m.key.empty()) j.flags &= ~CON_KEYS;
    if (m.es.empty()) j.flags &= ~CON_STACK;
    if (m.eu.empty()) j.flags &= ~CON_UNPAIRED;
  }
  std::stable_sort(m.jobs.begin(), m.jobs.end(), [](const MfeJob& x, const MfeJob& y) { return x.n > y.n; });
  if (m.jobs.empty()) return RP_OK;
  // one workspace slot per resident CTA, within the device's memory (long problems: fewer, fatter slots)
  m.slot_ints = mfe_slot_ints(maxn);
  const size_t slot_bytes = m.slot_ints * sizeof(int32_t);
  int g = dev.sm_count * std::max(1, dev.mfe_ctas_per_sm);
  g = std::min<int>(g, (int)m.jobs.size());
  if ((size_t)g * slot_bytes > dev.ws_bytes) g = (int)std::min<size_t>(g, std::max<size_t>(1, std::max<size_t>(1, dev.memory()) / 10 * 7 / slot_bytes));
  m.grid = g;
  return RP_OK;
}

}  // namespace rp
