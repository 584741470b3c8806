// dev_model.cpp -- integer energy model (rp_model) -> fp64 Boltzmann tables.
//
// Product-side restatement of ViennaRNA's parameter scaling as the reference's
// hot path sees it (pf_fold / co_pf_fold called at src/ractip.cpp:356,444 with
// temperature 37, dangles 2, pf_scale = -1; scale_parameters() called at
// src/pf_duplex.c:79).  At 37 C every table is exp(-E*10/kT) of its *37 value;
// dangles and exterior/multiloop mismatches go through the SMOOTH() clamp.
#include "dev_model.h"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace rp {
namespace {

struct Boltz {
  double kT;
  double operator()(int e) const { return std::exp(-static_cast<double>(e) * 10.0 / kT); }
};

// ViennaRNA params.c SMOOTH(X), X = -energy: keeps favourable values, maps
// unfavourable ones smoothly onto 0 so that dangles never penalise.
double smooth_neg(const rp_model& m, double x) {
  if (!m.pf_smooth) return x < 0 ? 0.0 : x;
  const double y = x / 10.0;
  if (y < -1.2283697) return 0.0;
  if (y > 0.8660254) return x;
  const double s = std::sin(y - 0.34242663) + 1.0;
  return 10.0 * 0.38490018 * s * s;
}

int base_of(char c) {
  switch (c) {
    case 'A': return 1;
    case 'C': return 2;
    case 'G': return 3;
    case 'U': return 4;
    default: return -1;  // list entries with other letters can never match an ACGU window
  }
}

// Blank-separated k-mer list -> base-8 codes (position-major, first char most significant).
int parse_special(const char* list, int mer, int max_entries, int* codes) {
  int n = 0;
  const size_t len = std::strlen(list);
  for (size_t off = 0; off + mer <= len && n < max_entries; off += mer + 1, n++) {
    int code = 0;
    bool ok = true;
    for (int k = 0; k < mer; k++) {
      int b = base_of(list[off + k]);
      if (b < 0) ok = false;
      code = code * 8 + (b < 0 ? 0 : b);
    }
    codes[n] = ok ? code : -1;
  }
  return n;
}

}  // namespace

int build_dev_model(const rp_model& m, DevModel* out) {
  if (!out) return RP_ERR_ARG;
  if (m.temperature != 37.0) return RP_ERR_UNSUPPORTED;  // *_dH tables are not carried
  if (m.dangles != 2) return RP_ERR_UNSUPPORTED;
  DevModel& D = *out;
  std::memset(&D, 0, sizeof D);
  Boltz bf{(m.temperature + RP_K0) * RP_GASCONST};
  D.kT = bf.kT;
  // pf_scale = -1 at every call site (src/ractip.cpp:325,392,442): ViennaRNA
  // then estimates it from -185 cal/mol per nucleotide times sfact.
  D.pf_scale = std::max(1.0, std::exp(-(m.sfact * (-185.0 + (m.temperature - 37.0) * 7.27)) / bf.kT));
  D.scale1 = 1.0 / D.pf_scale;
  D.expMLbase = bf(m.ML_BASE37);
  D.mlb1 = D.expMLbase * D.scale1;
  D.lxc = m.lxc37;
  D.expMLclosing = bf(m.ML_closing37);
  D.expMLintern = bf(m.ML_intern37);
  D.expTermAU = bf(m.TerminalAU37);
  D.scale_small[0] = 1.0;
  for (int k = 1; k < 40; k++) D.scale_small[k] = D.scale_small[k - 1] * D.scale1;
  for (int u = 0; u <= 30; u++) {
    D.exphairpin[u] = bf(m.hairpin37[u]);
    D.expbulge[u] = bf(m.bulge37[u]);
    D.expinternal[u] = bf(m.internal_loop37[u]);
    D.expninio[u] = bf(std::min(m.MAX_NINIO, u * m.ninio37));
    D.i_bulge[u] = m.bulge37[u];
    D.i_internal[u] = m.internal_loop37[u];
  }
  for (int t = 0; t < 8; t++) {
    for (int t2 = 0; t2 < 8; t2++) {
      D.expstack[t][t2] = bf(m.stack37[t][t2]);
      D.i_stack[t][t2] = m.stack37[t][t2];
      for (int a = 0; a < 5; a++)
        for (int b = 0; b < 5; b++) {
          D.int11[t][t2][a][b] = bf(m.int11_37[t][t2][a][b]);
          D.i_int11[t][t2][a][b] = m.int11_37[t][t2][a][b];
          for (int c = 0; c < 5; c++) {
            D.int21[t][t2][a][b][c] = bf(m.int21_37[t][t2][a][b][c]);
            D.i_int21[t][t2][a][b][c] = m.int21_37[t][t2][a][b][c];
            for (int d = 0; d < 5; d++) {
              D.int22[t][t2][a][b][c][d] = bf(m.int22_37[t][t2][a][b][c][d]);
              D.i_int22[t][t2][a][b][c][d] = m.int22_37[t][t2][a][b][c][d];
            }
          }
        }
    }
    for (int a = 0; a < 5; a++) {
      D.dangle5[t][a] = std::exp(smooth_neg(m, -static_cast<double>(m.dangle5_37[t][a])) * 10.0 / bf.kT);
      D.dangle3[t][a] = std::exp(smooth_neg(m, -static_cast<double>(m.dangle3_37[t][a])) * 10.0 / bf.kT);
      D.i_dangle5[t][a] = std::min(0, m.dangle5_37[t][a]);
      D.i_dangle3[t][a] = std::min(0, m.dangle3_37[t][a]);
      for (int b = 0; b < 5; b++) {
        D.mmI[t][a][b] = bf(m.mismatchI37[t][a][b]);
        D.mmH[t][a][b] = bf(m.mismatchH37[t][a][b]);
        D.mm1n[t][a][b] = bf(m.mismatch1nI37[t][a][b]);
        D.mm23[t][a][b] = bf(m.mismatch23I37[t][a][b]);
        D.mmM[t][a][b] = std::exp(smooth_neg(m, -static_cast<double>(m.mismatchM37[t][a][b])) * 10.0 / bf.kT);
        D.mmExt[t][a][b] = std::exp(smooth_neg(m, -static_cast<double>(m.mismatchExt37[t][a][b])) * 10.0 / bf.kT);
        D.i_mmExt[t][a][b] = std::min(0, m.mismatchExt37[t][a][b]);
        D.i_mmI[t][a][b] = m.mismatchI37[t][a][b];
        D.i_mm1n[t][a][b] = m.mismatch1nI37[t][a][b];
        D.i_mm23[t][a][b] = m.mismatch23I37[t][a][b];
      }
    }
  }
  // finished weights of the table-driven small loops, multiplied in the order the kernels used to
  for (int t = 0; t < 8; t++)
    for (int t2 = 0; t2 < 8; t2++) {
      D.spw[SPW_STACK + t * 8 + t2] = D.expstack[t][t2] * D.scale_small[2];
      D.spw[SPW_BULGE1 + t * 8 + t2] = D.expbulge[1] * D.expstack[t][t2] * D.scale_small[3];
      for (int a = 0; a < 5; a++)
        for (int b = 0; b < 5; b++) {
          D.spw[SPW_INT11 + ((t * 8 + t2) * 5 + a) * 5 + b] = D.int11[t][t2][a][b] * D.scale_small[4];
          // SPW_23 [type=t][si1=a][sj1=b][t2r=t2][sq1][sp1]
          for (int q = 0; q < 5; q++)
            for (int pp = 0; pp < 5; pp++)
              D.spw[SPW_23 + ((((t * 5 + a) * 5 + b) * 8 + t2) * 5 + q) * 5 + pp] =
                  D.expinternal[5] * D.expninio[1] * D.mm23[t][a][b] * D.mm23[t2][q][pp] * D.scale_small[7];
          for (int c = 0; c < 5; c++) {
            D.spw[SPW_INT21 + (((t * 8 + t2) * 5 + a) * 5 + b) * 5 + c] = D.int21[t][t2][a][b][c] * D.scale_small[5];
            for (int d = 0; d < 5; d++)
              D.spw[SPW_INT22 + ((((t * 8 + t2) * 5 + a) * 5 + b) * 5 + c) * 5 + d] = D.int22[t][t2][a][b][c][d] * D.scale_small[6];
          }
        }
    }
  D.i_TermAU = m.TerminalAU37;
  D.i_ninio = m.ninio37;
  D.i_MAX_NINIO = m.MAX_NINIO;
  D.i_DuplexInit = m.DuplexInit37;
  for (int u = 0; u <= 30; u++) D.i_hairpin[u] = m.hairpin37[u];
  for (int t = 0; t < 8; t++)
    for (int a = 0; a < 5; a++)
      for (int b = 0; b < 5; b++) {
        D.i_mmH[t][a][b] = m.mismatchH37[t][a][b];
        D.i_mmM[t][a][b] = std::min(0, m.mismatchM37[t][a][b]);
      }
  D.i_MLbase = m.ML_BASE37;
  D.i_MLclosing = m.ML_closing37;
  D.i_MLintern = m.ML_intern37;
  for (int i = 0; i < 200; i++) D.i_tetra[i] = m.Tetraloop37[i];
  for (int i = 0; i < 40; i++) D.i_tri[i] = m.Triloop37[i];
  for (int i = 0; i < 200; i++) D.i_hex[i] = m.Hexaloop37[i];
  for (int u = 31; u <= HP_LONG_MAX; u++) D.i_hairpin_long[u] = m.hairpin37[30] + (int)(m.lxc37 * std::log(u / 30.));

  D.special_hp = m.special_hp;
  D.n_tetra = parse_special(m.Tetraloops, 6, 200, D.tetra_code);
  D.n_tri = parse_special(m.Triloops, 5, 40, D.tri_code);
  D.n_hex = parse_special(m.Hexaloops, 8, 200, D.hex_code);
  for (int i = 0; i < D.n_tetra; i++) D.exptetra[i] = bf(m.Tetraloop37[i]);
  for (int i = 0; i < D.n_tri; i++) D.exptri[i] = bf(m.Triloop37[i]);
  for (int i = 0; i < D.n_hex; i++) D.exphex[i] = bf(m.Hexaloop37[i]);

  // Factorised interior loops (see dev_model.h for the classes).
  for (int u1 = 0; u1 <= MAXLOOP; u1++)
    for (int u2 = 0; u2 < GROW_LD; u2++) {
      D.grow[u1][u2] = 0.;
      D.gfull[u1][u2] = 0.;
      D.gcls[u1][u2] = CLS_NONE;
      if (u1 + u2 > MAXLOOP) continue;
      const int ul = std::max(u1, u2), us = std::min(u1, u2);
      int cls = CLS_SPECIAL;
      double g = 0;
      if (us == 0) {
        if (ul >= 2) { cls = CLS_BULGE; g = D.expbulge[ul]; }
      } else if (us == 1) {
        if (ul >= 3) { cls = CLS_1N; g = D.expinternal[ul + us] * D.expninio[ul - us]; }
      } else if (!(us == 2 && (ul == 2 || ul == 3))) {
        cls = CLS_GENERIC;
        g = D.expinternal[ul + us] * D.expninio[ul - us];
      }
      g *= D.scale_small[u1 + u2 + 2];
      D.gcls[u1][u2] = static_cast<uint8_t>(cls);
      if (cls == CLS_SPECIAL) continue;
      D.gfull[u1][u2] = g;
      const int row_cls = u1 == 0 ? CLS_BULGE : (u1 == 1 ? CLS_1N : CLS_GENERIC);
      if (cls == row_cls) D.grow[u1][u2] = g;
      else if (u2 == 0) D.ghead_b[u1] = g;  // rows >= 2: bulge (u1,0)
      else D.ghead_1[u1] = g;               // rows >= 3: 1xn (u1,1)
    }
  for (int sdiag = 0; sdiag <= MAXLOOP; sdiag++)
    for (int t = 0; t <= sdiag; t++)
      D.gpack[sdiag * (sdiag + 1) / 2 + t] = D.gcls[t][sdiag - t] == CLS_GENERIC ? D.gfull[t][sdiag - t] : 0.;
  for (int sdiag = 0; sdiag < 32; sdiag++) {
    D.gA[sdiag] = (sdiag >= 2 && sdiag <= MAXLOOP) ? D.gfull[0][sdiag] : 0.;
    D.g1[sdiag] = (sdiag >= 4 && sdiag <= MAXLOOP) ? D.gfull[1][sdiag - 1] : 0.;
  }
  return RP_OK;
}

}  // namespace rp
