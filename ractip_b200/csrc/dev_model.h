// dev_model.h -- fp64 Boltzmann tables as the kernels consume them, and the
// host routine that builds them from the integer model.
//
// Replaces ViennaRNA's get_scaled_pf_parameters()/scale_parameters() as used
// inside pf_fold / co_pf_fold (reference call sites src/ractip.cpp:356,444) and
// by src/pf_duplex.c:78-81.  Plain-old-data: uploaded to HBM once per context.
#ifndef RP_DEV_MODEL_H
#define RP_DEV_MODEL_H

#include <stdint.h>

#include "ractip_prob.h"

namespace rp {

constexpr int TURN = RP_TURN;
constexpr int MAXLOOP = RP_MAXLOOP;

// Factorised interior loops.  Outside the table-driven small cases the weight
// of the loop (u1 unpaired on the 5' side, u2 on the 3' side) splits into
//     f(closing pair) * f(inner pair) * g(u1,u2)
// with three classes of pair factors:
//   GENERIC (us>=2, not 2x2/2x3): g = expinternal[u]*expninio[|u1-u2|], f = expmismatchI
//   ONE_N   (us==1, ul>=3)      : g = expinternal[u]*expninio[ul-1],   f = expmismatch1nI
//   BULGE   (us==0, ul>=2)      : g = expbulge[ul],                    f = expTermAU^[type>2]
// so the sum over inner pairs becomes, per class, a weighted sum over a table
// that already carries the inner pair's factor.  All g below include
// scale[u1+u2+2].  Stack, 1-bulge, 1x1, 1x2, 2x2 and 2x3 loops do not factorise
// (class SPECIAL) and are evaluated directly.
enum { CLS_GENERIC = 0, CLS_1N = 1, CLS_BULGE = 2, CLS_SPECIAL = 3, CLS_NONE = 255 };
constexpr int GROW_LD = 32;
constexpr int HP_LONG_MAX = 12000;   // longest hairpin loop of DevModel::i_hairpin_long (= RP_MAX_N, mcc_core.h)

// Table-driven small loops (the nine shapes that do not factorise: stack, 1-bulge, 1x1, 1x2, 2x1, 2x2, 2x3,
// 3x2): ONE flat table of finished weights, scale included, so that a look-up is an index computation and
// a single load (DevModel::spw; index arithmetic in special_loop, mcc_core.h).
//   SPW_STACK  [type][t2r]                          expstack * scale[2]
//   SPW_BULGE1 [type][t2r]                          expbulge[1] * expstack * scale[3]
//   SPW_INT11  [type][t2r][si1][sj1]                int11 * scale[4]
//   SPW_INT21  [type][t2r][a][b][c]                 int21 * scale[5]   (index order of ViennaRNA's int21)
//   SPW_INT22  [type][t2r][si1][sp1][sq1][sj1]      int22 * scale[6]
//   SPW_23     [type][si1][sj1][t2r][sq1][sp1]      expinternal[5]*expninio[1]*mm23*mm23*scale[7]
constexpr int SPW_STACK = 0, SPW_BULGE1 = 64, SPW_INT11 = 128, SPW_INT21 = SPW_INT11 + 1600,
              SPW_INT22 = SPW_INT21 + 8000, SPW_23 = SPW_INT22 + 40000, SPW_SIZE = SPW_23 + 40000;

struct DevModel {
  double pf_scale, scale1, mlb1;  // scale1 = 1/pf_scale, mlb1 = expMLbase*scale1
  double kT, lxc;
  double expMLclosing, expMLintern, expTermAU, expMLbase;
  double scale_small[40];  // scale1^k
  double exphairpin[31], expbulge[31], expinternal[31], expninio[MAXLOOP + 1];
  double expstack[8][8];
  double mmI[8][5][5], mmH[8][5][5], mmM[8][5][5], mmExt[8][5][5], mm1n[8][5][5], mm23[8][5][5];
  double dangle5[8][5], dangle3[8][5];
  double int11[8][8][5][5];
  double int21[8][8][5][5][5];
  double int22[8][8][5][5][5][5];
  double spw[SPW_SIZE];   // finished weights of the table-driven small loops (see above)
  // Band kernel's view of the factorised weights, ready to be copied into shared memory:
  //   gpack[s*(s+1)/2 + t] = g(t, s-t) where (t, s-t) is GENERIC, else 0;  gA[s] = g(0,s) (bulge, s >= 2);
  //   g1[s] = g(1,s-1) (1xn, s >= 4)
  double gpack[(MAXLOOP + 1) * (MAXLOOP + 2) / 2 + 8];
  double gA[32], g1[32];
  // special hairpins: k-mers as base-8 codes of the 1..4 encoding
  int n_tetra, n_tri, n_hex;
  int tetra_code[200], tri_code[40], hex_code[200];
  double exptetra[200], exptri[40], exphex[200];
  int special_hp;
  // Row view of the factorised loops: row u1 is scanned along u2.
  //   row 0 runs over the BULGE table, row 1 over the ONE_N table, rows >=2 over GENERIC;
  //   grow[u1][u2] is the run weight (0 where (u1,u2) is SPECIAL or handled as a head);
  //   rows >= 2 have two heads in other tables: u2=0 (BULGE, ghead_b[u1]) and
  //   u2=1 (ONE_N, ghead_1[u1], rows >= 3).
  double grow[MAXLOOP + 1][GROW_LD];
  double ghead_b[GROW_LD], ghead_1[GROW_LD];
  // Full (u1,u2) view for the unpaired-window gap sums.
  double gfull[MAXLOOP + 1][GROW_LD];
  uint8_t gcls[MAXLOOP + 1][GROW_LD];
  // integer view for pf_duplex (scale_parameters semantics at 37 C)
  int i_dangle5[8][5], i_dangle3[8][5], i_mmExt[8][5][5];
  int i_stack[8][8], i_bulge[31], i_internal[31], i_mmI[8][5][5], i_mm1n[8][5][5], i_mm23[8][5][5];
  int i_int11[8][8][5][5], i_int21[8][8][5][5][5], i_int22[8][8][5][5][5][5];
  int i_TermAU, i_ninio, i_MAX_NINIO, i_DuplexInit;
  // Integer view for the MFE kernel (mfe_core.h), appended so that every field above keeps its offset.  Exactly the
  // values rp_energy_of_structure (eval.cpp) uses: mismatchM clipped to <= 0 like the dangles, the rest as is.
  // i_hairpin_long[u] = hairpin37[30] + (int)(lxc37 * ln(u / 30)) for 30 < u <= HP_LONG_MAX, computed on the host with
  // eval.cpp's expression, so that the truncation to int does not hinge on the device's log().
  int i_hairpin[31], i_mmH[8][5][5], i_mmM[8][5][5];
  int i_MLbase, i_MLclosing, i_MLintern;
  int i_tetra[200], i_tri[40], i_hex[200];
  int i_hairpin_long[HP_LONG_MAX + 1];
};

// Host: integer model -> DevModel.  Returns RP_OK or an error code.
int build_dev_model(const rp_model& m, DevModel* out);

}  // namespace rp
#endif
