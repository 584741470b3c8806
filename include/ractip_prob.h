/*
 * ractip_prob.h -- C ABI of the B200-native probability stage for RactIP.
 *
 * This is the drop-in boundary for the three calls RactIP::solve makes to fill
 * its probability matrices (reference src/ractip.cpp:546-548):
 *     rnafold (fa1, bp1_, offset1_, up1_, max_w)    src/ractip.cpp:308-382
 *     rnafold (fa2, bp2_, offset2_, up2_, max_w)    src/ractip.cpp:308-382
 *     rnaduplex(fa1, fa2, hp_)                      src/ractip.cpp:384-459
 * and for the batch of those calls made by the --zscore shuffle loop
 * (src/ractip.cpp:1638-1657).  Everything is plain C: pointers, sizes, ints.
 * No torch types, no C++ types, no exceptions cross this boundary.
 *
 * All compute entry points run hand-written sm_100a CUDA kernels.  There is NO
 * CPU fallback: without a usable CUDA device they return RP_ERR_NO_DEVICE.
 * Host-only helpers (model loading, shuffling, layout queries) work anywhere.
 */
#ifndef RACTIP_PROB_H
#define RACTIP_PROB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------ */
/* constants of the energy model (ViennaRNA energy_const.h; used by name in  */
/* reference src/pf_duplex.c:73,100,142,148-154)                             */
/* ------------------------------------------------------------------------ */
#define RP_NBPAIRS 7
#define RP_MAXLOOP 30
#define RP_TURN 3
#define RP_INF 10000000
#define RP_K0 273.15
#define RP_GASCONST 1.98717 /* cal/(K mol) */

/* error codes (0 = success) */
enum {
  RP_OK = 0,
  RP_ERR_ARG = 1,        /* bad argument (NULL, negative size, ...)           */
  RP_ERR_NO_DEVICE = 2,  /* no CUDA device / driver: there is no CPU fallback */
  RP_ERR_CUDA = 3,       /* a CUDA call failed; see rp_last_error()           */
  RP_ERR_IO = 4,         /* file missing / unreadable                         */
  RP_ERR_FORMAT = 5,     /* parameter file malformed                          */
  RP_ERR_NO_DEFAULTS = 6,/* requested tables that are not embedded            */
  RP_ERR_SEQ = 7,        /* sequence has a character outside ACGUT (any case) */
  RP_ERR_TOO_LONG = 8,   /* sequence longer than the context was created for  */
  RP_ERR_CAPACITY = 9,   /* caller-provided output buffer too small           */
  RP_ERR_UNSUPPORTED = 10
};

/* ------------------------------------------------------------------------ */
/* rp_model: the integer energy tables (units 0.01 kcal/mol, 37 C) with the  */
/* exact names, index order and extents of ViennaRNA's energy_par.h globals. */
/* Replaces: the ViennaRNA globals that copy_boltzmann_parameters()          */
/* (src/boltzmann_param.c:5908-6026) and read_parameter_file()               */
/* (src/ractip.cpp:63,1568-1569) prime before the hot path runs.             */
/* A RactIP build that links ViennaRNA can memcpy its globals into this      */
/* struct field by field (INTEGRATION.md shows the stub).                    */
/* The *_dH enthalpy tables are deliberately absent: RactIP never changes    */
/* `temperature` from 37 C, where they cancel exactly.                       */
/* ------------------------------------------------------------------------ */
typedef struct rp_model {
  double temperature;     /* must be 37.0                                    */
  int dangles;            /* must be 2 (ViennaRNA default; pf treats 1 as 2) */
  int special_hp;         /* tetra_loop flag, default 1                      */
  int pf_smooth;          /* default 1                                       */
  double sfact;           /* pf_scale heuristic factor, default 1.07         */

  int stack37[RP_NBPAIRS + 1][RP_NBPAIRS + 1];
  int hairpin37[31];
  int bulge37[31];
  int internal_loop37[31];
  int mismatchI37[RP_NBPAIRS + 1][5][5];
  int mismatchH37[RP_NBPAIRS + 1][5][5];
  int mismatchM37[RP_NBPAIRS + 1][5][5];
  int mismatchExt37[RP_NBPAIRS + 1][5][5];
  int mismatch1nI37[RP_NBPAIRS + 1][5][5];
  int mismatch23I37[RP_NBPAIRS + 1][5][5];
  int dangle5_37[RP_NBPAIRS + 1][5];
  int dangle3_37[RP_NBPAIRS + 1][5];
  int int11_37[RP_NBPAIRS + 1][RP_NBPAIRS + 1][5][5];
  int int21_37[RP_NBPAIRS + 1][RP_NBPAIRS + 1][5][5][5];
  int int22_37[RP_NBPAIRS + 1][RP_NBPAIRS + 1][5][5][5][5];
  int ML_BASE37, ML_closing37, ML_intern37;
  int TerminalAU37;
  int ninio37, MAX_NINIO;
  int DuplexInit37;
  double lxc37;
  /* special hairpins: blank-separated lists exactly as ViennaRNA keeps them */
  char Tetraloops[1401];
  int Tetraloop37[200];
  char Triloops[241];
  int Triloop37[40];
  char Hexaloops[1801];
  int Hexaloop37[200];
} rp_model;

/* Fill *m with the tables a default `ractip` run uses: ViennaRNA's Turner-2004
 * defaults for the tables BL* leaves alone (embedded copy: see
 * params/turner2004_residual.par for provenance) and, if use_bl != 0, the
 * Andronescu BL* values with the copy semantics of
 * src/boltzmann_param.c:5908-6026.  use_bl == 0 (--no-bl) needs the full
 * Turner-2004 set, which is not embedded: returns RP_ERR_NO_DEFAULTS unless a
 * complete parameter file is loaded afterwards.  Host only. */
int rp_model_default(rp_model* m, int use_bl);

/* Overlay a ViennaRNA "## RNAfold parameter file v2.0" on *m (replaces
 * Vienna::read_parameter_file, src/ractip.cpp:1568-1569).  Only the sections
 * present in the file are overwritten.  Host only. */
int rp_model_read_par(rp_model* m, const char* path);

/* FNV-1a digest of every table in *m (tests pin the embedded defaults). */
uint64_t rp_model_digest(const rp_model* m);

/* ------------------------------------------------------------------------ */
/* problems                                                                  */
/* ------------------------------------------------------------------------ */
typedef struct rp_pair {
  const char* s1; int n1;   /* first RNA, 5'->3', ACGU/T any case, not NUL-terminated-dependent */
  const char* s2; int n2;   /* second RNA; n2 == 0 (s2 may be NULL): s1 alone, */
                            /* only its bp/up sections are computed           */
} rp_pair;

/* options that change the probability stage (src/ractip.cpp:546-548,390,447) */
typedef struct rp_opts {
  int max_w;          /* accessibility window: callers pass std::max(1,max_w_) */
  int min_w;          /* only used by the sparse path (src/ractip.cpp:622)     */
  float th_ss;        /* -t, default 0.5   (src/ractip.cpp:562,583)            */
  float th_hy;        /* -u, default 0.1   (src/ractip.cpp:447,452,603)        */
  float th_ac;        /* -s, default 0.003 (src/ractip.cpp:623,643)            */
  int use_pf_duplex;  /* --duplex: pf_duplex instead of co_pf_fold (:390)      */
} rp_opts;

void rp_opts_default(rp_opts* o);   /* max_w 15, min_w 5, 0.5, 0.1, 0.003, 0 */

/* Flat dense output layout for one pair; offsets are in floats from the start
 * of the batch buffer.  Sections use the reference's own layouts:
 *   bp : (L+1)(L+2)/2 floats, bp[offset[i]+j], offset[i]=i*(2L+1-i)/2, 1<=i<j<=L
 *        (src/ractip.cpp:314-317,365-367); entries never written by the
 *        reference (i==j, index 0) are 0.
 *   up : L*max_w floats row-major, up[i*max_w+d] = P(bases i+1..i+1+d unpaired)
 *        with 0-based start i (src/ractip.cpp:370-375); windows running past
 *        the 3' end are 0.
 *   hp : (L1+1)*(L2+1) floats row-major, 1-based both.  Default branch: p if
 *        p>th_hy else 0 (src/ractip.cpp:404-405,451-453); --duplex branch:
 *        dense (src/ractip.cpp:393-397). */
typedef struct rp_dense_layout {
  size_t bp1, bp2, up1, up2, hp;      /* offsets (floats)                    */
  size_t n_bp1, n_bp2, n_up1, n_up2, n_hp; /* section lengths (floats)       */
} rp_dense_layout;

/* Compute per-pair layouts (layout[n_pairs]) and the total float count. */
int rp_dense_plan(const rp_pair* pairs, int n_pairs, const rp_opts* opts,
                  rp_dense_layout* layout, size_t* total_floats);

/* Sparse (thresholded) records in the reference's variable-creation order
 * (src/ractip.cpp:557-567 x: j ascending then i descending; :598-609 z: i
 * ascending then j ascending; :619-628 v and :639-648 w: start i ascending,
 * then window-length index j = min_w-1 .. max_w-1 ascending, the region being
 * bases i..i+j), 0-based like the consumer's loops.  v/w are empty when the
 * reference would not create them (min_w <= 1 or max_w < min_w, :526). */
typedef struct rp_rec { int32_t i, j; float p; } rp_rec;

typedef struct rp_sparse_layout {
  size_t x, y, z;            /* offsets into the rp_rec buffer               */
  size_t cap_x, cap_y, cap_z;/* capacities (records)                         */
  size_t up1, up2;           /* offsets (floats) into the OPTIONAL float     */
  size_t n_up1, n_up2;       /* buffer of the dense window tables            */
  size_t v, w;               /* offsets into the rp_rec buffer               */
  size_t cap_v, cap_w;
} rp_sparse_layout;

typedef struct rp_sparse_counts { int32_t n_x, n_y, n_z, overflow, n_v, n_w; } rp_sparse_counts;

int rp_sparse_plan(const rp_pair* pairs, int n_pairs, const rp_opts* opts,
                   rp_sparse_layout* layout, size_t* total_recs, size_t* total_floats);

/* ------------------------------------------------------------------------ */
/* context: one per process per GPU                                          */
/* ------------------------------------------------------------------------ */
typedef struct rp_ctx rp_ctx;

/* Builds the fp64 Boltzmann tables from *m (replaces ViennaRNA's
 * get_scaled_pf_parameters / scale_parameters as used by pf_fold, co_pf_fold
 * and src/pf_duplex.c:78-81) and uploads them to `device`.
 * Returns RP_ERR_NO_DEVICE when no CUDA device can be used. */
int rp_create(rp_ctx** ctx, const rp_model* m, int device);
int rp_destroy(rp_ctx* ctx);
const char* rp_last_error(const rp_ctx* ctx);   /* ctx may be NULL            */
const char* rp_strerror(int code);

/* Use an externally owned cudaStream_t (e.g. torch's current stream). NULL
 * restores the context's own stream. */
int rp_set_stream(rp_ctx* ctx, void* cuda_stream);
/* The stream the context enqueues on now (its own one unless rp_set_stream
 * chose another), so that a caller can set it back after borrowing it. */
int rp_get_stream(const rp_ctx* ctx, void** cuda_stream);

/* Pinned host memory for output buffers (plain malloc'd buffers also work). */
void* rp_host_alloc(size_t bytes);
void rp_host_free(void* p);

/* One-shot calls with HOST buffers: H2D of the sequences, kernels, D2H of the
 * results, synchronous.  `out` must hold total_floats from rp_dense_plan. */
int rp_run_dense(rp_ctx* ctx, const rp_pair* pairs, int n_pairs,
                 const rp_opts* opts, float* out, size_t out_floats);

/* `ups` (the dense window tables next to the lists) may be NULL: the v/w lists
 * carry every up[i][j] the integer programme reads (src/ractip.cpp:621-627). */
int rp_run_sparse(rp_ctx* ctx, const rp_pair* pairs, int n_pairs,
                  const rp_opts* opts, rp_rec* recs, size_t n_recs,
                  float* ups, size_t n_floats, rp_sparse_counts* counts);

/* All GPUs of one box behind one handle (host threads over the single-device entry points): the batch is cut
 * into contiguous blocks, pair k of n going to device k*G/n, and every device writes its block straight into
 * the caller's one host buffer, in the layouts of rp_dense_plan / rp_sparse_plan for the WHOLE batch.  This is
 * what the z-score loop of src/ractip.cpp:1638-1657 needs to use a multi-GPU box from one process.
 * devices == NULL: devices 0 .. n_devices-1 (n_devices <= 0: every visible device). */
typedef struct rp_multi rp_multi;
int rp_multi_create(rp_multi** multi, const rp_model* m, const int* devices, int n_devices);
int rp_multi_destroy(rp_multi* multi);
int rp_multi_devices(const rp_multi* multi);
const char* rp_multi_last_error(const rp_multi* multi);   /* multi may be NULL */
int rp_multi_run_dense(rp_multi* multi, const rp_pair* pairs, int n_pairs,
                       const rp_opts* opts, float* out, size_t out_floats);
int rp_multi_run_sparse(rp_multi* multi, const rp_pair* pairs, int n_pairs,
                        const rp_opts* opts, rp_rec* recs, size_t n_recs,
                        rp_sparse_counts* counts);

/* Device-resident batch (bench "value": inputs already in HBM). */
typedef struct rp_batch rp_batch;
int rp_batch_create(rp_ctx* ctx, const rp_pair* pairs, int n_pairs,
                    const rp_opts* opts, rp_batch** batch);

/* Structure constraints of one pair (RactIP -c, the FASTA record's structure
 * line): c1 over s1 (n1 chars), c2 over s2 (n2 chars), NUL-terminated; NULL
 * means unconstrained.  Alphabet of RactIP's joint structures:
 *   .      no constraint
 *   x      the base pairs with nothing
 *   ( )    intramolecular pair, bracket-matched within the same string
 *   [ ]    intermolecular pair, '[' in c1 only, ']' in c2 only: the k-th '['
 *          from the 3' end of s1 pairs with the k-th ']' from the 5' end of s2
 * A constraint only removes pairs (no base is forced to pair, no energy
 * changes).  s1's fold sees the () of c1 and keeps x and [ unpaired; s2's fold
 * the () of c2, x and ] unpaired; the s1&s2 co-fold the [] pairs, x ( )
 * unpaired; the --duplex branch is unconstrained.  A pair (i,j) of a problem is
 * allowed when neither base is unpaired there, a bracketed base pairs only with
 * its partner, and (i,j) crosses no bracket pair.  A bracket pair that cannot
 * form leaves both bases unpaired. */
typedef struct rp_constraint {
  const char* c1;
  const char* c2;
} rp_constraint;
/* rp_batch_create with one rp_constraint per pair (cons == NULL, or an entry
 * with both strings NULL: unconstrained).  The problems a constraint restricts
 * run on the general kernel.  RP_ERR_ARG, with rp_last_error naming the pair,
 * the string and the position, for a string whose length differs from its
 * sequence's, a character outside .x()[], unbalanced (), ] in c1 or [ in c2,
 * or different numbers of [ in c1 and ] in c2.  Everything that takes an
 * rp_batch works on the result unchanged. */
int rp_batch_create_constrained(rp_ctx* ctx, const rp_pair* pairs,
                                const rp_constraint* cons, int n_pairs,
                                const rp_opts* opts, rp_batch** batch);

/* Stacking pseudo-energies of one pair (chemical probing data, e.g. SHAPE
 * reactivities through rp_shape_deigan): e1[0..n1-1] over s1, e2[0..n2-1]
 * over s2, in kcal/mol; NULL means none.  ViennaRNA's vrna_sc_set_stack
 * semantics, to which RNAfold --shape (Deigan method) reduces:
 *   - each value is rounded to an integer number of 0.01 kcal/mol, half away
 *     from zero: E_i;
 *   - every stack, an interior loop closed by (i,j) around (i+1,j-1), has its
 *     Boltzmann weight multiplied by f(i) f(i+1) f(j-1) f(j), where
 *     f(x) = exp(-E_x * 10 / kT) at the model's kT (37 C);
 *   - nothing else changes: no other loop (bulges of one base included), no
 *     pf_scale, no energy of rp_energy_of_structure (-e, z-scores).
 * s1's fold takes e1, s2's fold e2.  The s1&s2 co-fold applies them to the
 * stacks within one strand, with that strand's values; a stack that joins the
 * strands gets no pseudo-energy (data measured on each RNA alone describe its
 * own structure).  The --duplex branch takes none. */
typedef struct rp_stack_energy {
  const double* e1;
  const double* e2;
} rp_stack_energy;
/* rp_batch_create with structure constraints (cons, as
 * rp_batch_create_constrained; NULL: none) and stacking pseudo-energies (se,
 * one rp_stack_energy per pair; NULL, or an entry with both NULL: none).  A
 * problem whose rounded values are all 0 has no data: it is planned and
 * computed exactly as without them.  Problems with data run on the general
 * kernel.  RP_ERR_ARG, with rp_last_error naming the pair, the vector and
 * the position, for a value that is not finite; constraint errors as
 * rp_batch_create_constrained.  Everything that takes an rp_batch works on
 * the result unchanged. */
int rp_batch_create_soft(rp_ctx* ctx, const rp_pair* pairs,
                         const rp_constraint* cons, const rp_stack_energy* se,
                         int n_pairs, const rp_opts* opts, rp_batch** batch);
/* Deigan et al. (2009) pseudo-energies from probing reactivities, host only:
 * e[i] = slope * ln(r[i] + 1) + intercept for r[i] >= 0, 0 for r[i] < 0 or
 * NaN (missing data).  RNAfold --shapeMethod=D uses slope 1.8 and intercept
 * -0.6 kcal/mol.  RP_ERR_ARG for n < 0 or a NULL array with n > 0. */
int rp_shape_deigan(const double* r, int n, double slope, double intercept,
                    double* e);
/* Stochastic sampling of secondary structures (RNAfold -p --stochBT,
 * RNAsubopt -p): `num` structures per requested problem, each drawn with
 * probability exp(-E/kT) / Z from exactly the ensemble whose log Z
 * rp_batch_fetch_logz reports (dangles = 2, MAXLOOP, special hairpins, -P
 * tables; the batch's constraints and stacking pseudo-energies apply; the
 * co-fold without DuplexInit).  `problems` is a mask of RP_SAMPLE_*; --duplex
 * has no co-fold ensemble to sample (RP_ERR_UNSUPPORTED), a pair with n2 == 0
 * only s1.  Random numbers: Philox4x64-10, key (seed, 3 pair + problem),
 * counter (sample, decision / 4, 0, 0): a pair's samples do not depend on the
 * other pairs of the batch, and one seed gives the same samples. */
enum { RP_SAMPLE_S1 = 1, RP_SAMPLE_S2 = 2, RP_SAMPLE_COFOLD = 4 };
typedef struct rp_sample_opts {
  int num;          /* samples per requested problem, >= 0 */
  uint64_t seed;
  int problems;     /* RP_SAMPLE_* mask */
} rp_sample_opts;
/* Where a pair's samples live in the batch's sample buffer, in int16
 * elements: num pair tables of n1 at s1, of n2 at s2, of n1+n2 at co (the
 * concatenation s1 s2: base b of s2 is n1 + b); a problem that is not
 * sampled has length 0.  Pair table t: t[k-1] = partner of base k (1-based),
 * 0 if k is unpaired. */
typedef struct rp_sample_layout {
  size_t s1, s2, co;          /* offsets */
  size_t len_s1, len_s2, len_co;
} rp_sample_layout;
/* Host arithmetic: per_pair[p] and *total (int16 elements).  RP_ERR_ARG for a
 * bad argument or when a size overflows size_t. */
int rp_sample_plan(const rp_pair* pairs, int n_pairs, const rp_sample_opts* so,
                   rp_sample_layout* per_pair, size_t* total);
/* rp_batch_create_soft plus samples, drawn by every rp_batch_run between the
 * inside and the outside pass of the sampled problems, which run on the
 * general kernel (so == NULL or num == 0: exactly rp_batch_create_soft).
 * RP_ERR_ARG for num < 0 or an unknown bit in problems, RP_ERR_UNSUPPORTED for
 * RP_SAMPLE_COFOLD with use_pf_duplex; rp_last_error names the pair. */
int rp_batch_create_sampled(rp_ctx* ctx, const rp_pair* pairs,
                            const rp_constraint* cons, const rp_stack_energy* se,
                            int n_pairs, const rp_opts* opts,
                            const rp_sample_opts* so, rp_batch** batch);

/* Unpaired pseudo-energies of one pair (probing data that reward or penalise a
 * base for staying unpaired, e.g. DMS or SHAPE perturbation vectors): u1[0..n1-1]
 * over s1, u2[0..n2-1] over s2, in kcal/mol; NULL means none.  ViennaRNA's
 * vrna_sc_set_up semantics (RNAfold --shapeMethod=W):
 *   - each value is rounded to an integer number of 0.01 kcal/mol, half away
 *     from zero: E_x;
 *   - every base x a structure leaves unpaired, in hairpins, interior loops,
 *     bulges, multiloops and the exterior loop alike, multiplies the
 *     structure's Boltzmann weight by f(x) = exp(-E_x * 10 / kT) (37 C);
 *   - nothing else changes: no pf_scale, no energy of rp_energy_of_structure.
 * s1's fold takes u1, s2's fold u2.  The s1&s2 co-fold takes both; a base paired
 * with the partner counts as unpaired there (data measured on each RNA alone
 * describe only its own structure).  The --duplex branch takes none.  log Z
 * (rp_batch_fetch_logz) is that of the ensemble with the factors.
 * Range: pf_scale is not adapted to the data, so a problem whose
 * B = sum_x |E_x| * 10 / kT over the bases it applies exceeds ln 10^150 is
 * RP_ERR_UNSUPPORTED (about 425 nt at 0.5 kcal/mol per base). */
typedef struct rp_unpaired_energy {
  const double* u1;
  const double* u2;
} rp_unpaired_energy;
/* rp_batch_create_sampled with unpaired pseudo-energies as well (ue, one
 * rp_unpaired_energy per pair; NULL, or an entry with both NULL: none; ue ==
 * NULL is exactly rp_batch_create_sampled).  A problem whose rounded values are
 * all 0 has no such data and is planned and computed exactly as without it;
 * problems with data run on the general kernel.  RP_ERR_ARG, with rp_last_error
 * naming the pair, the vector and the position, for a value that is not
 * finite; RP_ERR_UNSUPPORTED, naming the pair, the problem and B, for a problem
 * beyond the range above. */
int rp_batch_create_probed(rp_ctx* ctx, const rp_pair* pairs,
                           const rp_constraint* cons, const rp_stack_energy* se,
                           const rp_unpaired_energy* ue, int n_pairs,
                           const rp_opts* opts, const rp_sample_opts* so,
                           rp_batch** batch);
/* The samples of the last run, in the layout of rp_sample_plan: to the host
 * (synchronous), or device to device into memory the caller owns (the stream
 * rules of rp_batch_dense_device).  RP_ERR_CAPACITY when n < total. */
int rp_batch_fetch_samples(rp_batch* batch, int16_t* out, size_t n);
int rp_batch_samples_device(rp_batch* batch, void* out_dev, size_t n);
/* Minimum free energy (MFE) structures (RNAfold / RNAcofold's first line):
 * for each requested problem of each pair, the minimum over every structure S
 * of exactly the ensemble the partition function sums over (canonical pairs
 * with j-i > TURN across the nick too, interior loops up to MAXLOOP, the
 * pair's constraint keys as rp_batch_create_constrained builds them; s1 takes
 * e1/u1, s2 e2/u2, the co-fold both) of
 *   E(S) = rp_energy_of_structure(seq, S, cut_point)     (0.01 kcal/mol)
 *        + sum over stacks (i,j),(i+1,j-1) of S within one strand of
 *          Es(i) + Es(i+1) + Es(j-1) + Es(j)
 *        + sum over bases x unpaired in S of Eu(x)
 * with Es, Eu rounded as rp_batch_create_soft / rp_batch_create_probed round
 * them; in the co-fold a stack that joins the strands gets no Es, and a base
 * paired with the partner counts as unpaired.  The co-fold (cut_point =
 * n1+1) adds DuplexInit once when a pair joins the strands, as
 * rp_energy_of_duplex and -e count it, so that
 *   MFE(s1&s2) = min(MFE of the unjoined structures, i.e. s1's and s2's folds
 *                under the co-fold's constraint,
 *                min over joined structures + DuplexInit);
 * the partition function (log Z, probabilities, samples) leaves DuplexInit
 * out.  The result is exact integer arithmetic.  One structure that reaches
 * the minimum is returned; ties are broken by a fixed candidate order.
 *
 * `problems` is a mask of RP_SAMPLE_* (unknown bits: RP_ERR_ARG); a pair with
 * n2 == 0 has s1 only.  structures: the layout of rp_sample_plan with num = 1
 * and the same mask (RP_ERR_CAPACITY when n_structures is smaller); energies:
 * 3 int32 per pair (s1, s2, s1&s2) in 0.01 kcal/mol, RP_INF for a problem not
 * computed.  cons, se, ue (each may be NULL) are checked as
 * rp_batch_create_probed checks them, with the same messages, except that the
 * pf_scale range of unpaired pseudo-energies does not apply.  Instead a
 * problem whose sum over its bases of |Es| + |Eu| (0.01 kcal/mol, after
 * rounding) exceeds RP_INF / 4 (25000 kcal/mol) is RP_ERR_UNSUPPORTED,
 * naming the pair and the problem: every energy then stays far from the
 * int32 range next to the kernel's INF sentinel.  rp_opts plays no part
 * (--duplex changes how hp is computed, not the co-fold's MFE).  Synchronous,
 * host buffers, on the context's stream. */
int rp_run_mfe(rp_ctx* ctx, const rp_pair* pairs, const rp_constraint* cons,
               const rp_stack_energy* se, const rp_unpaired_energy* ue,
               int n_pairs, int problems, int16_t* structures,
               size_t n_structures, int32_t* energies);
int rp_batch_run(rp_batch* batch);                 /* async on the ctx stream */
int rp_batch_sync(rp_batch* batch);
int rp_batch_fetch_dense(rp_batch* batch, float* out, size_t out_floats);
int rp_batch_fetch_sparse(rp_batch* batch, rp_rec* recs, size_t n_recs,
                          float* ups, size_t n_floats, rp_sparse_counts* counts);
/* Same records, but left in DEVICE memory the caller owns (e.g. torch CUDA
 * tensors handed to one ncclAllGather): no host copy, asynchronous on the
 * context stream.  counts_dev receives n_pairs rp_sparse_counts. */
int rp_batch_sparse_device(rp_batch* batch, void* recs_dev, size_t n_recs,
                           void* ups_dev, size_t n_floats, void* counts_dev);
/* The dense outputs left in DEVICE memory the caller owns, in the layout of
 * rp_dense_plan (the bytes rp_batch_fetch_dense delivers): one device-to-device
 * copy, asynchronous on the context's current stream.  If the batch last ran
 * on another stream, the current stream first waits for it (no host
 * synchronisation).  RP_ERR_CAPACITY when out_floats < total_floats. */
int rp_batch_dense_device(rp_batch* batch, void* out_dev, size_t out_floats);

/* Padded square layout of a batch: the dense outputs of every pair expanded
 * into five fp32 tensors, row-major, 1-based like the reference (index 0 and
 * everything past a pair's own lengths are 0):
 *   bp1 [B][N1+1][N1+1]   symmetric: P[i][j] = P[j][i] = bp[offset[i]+j], 1<=i<j<=n1
 *   bp2 [B][N2+1][N2+1]
 *   up1 [B][N1][W]        up[i][d] as in rp_dense_layout, rows past n1 are 0
 *   up2 [B][N2][W]
 *   hp  [B][N1+1][N2+1]   hp[i][j] as in rp_dense_layout (thresholded zeros kept)
 * with N1 = max n1, N2 = max n2 over the batch and W = max(max_w, 0).  A pair
 * with n2 == 0 has all-zero bp2, up2 and hp slices.  n_* are element counts;
 * RP_ERR_ARG if one of them (or its size in bytes) overflows size_t.  Host
 * arithmetic only. */
typedef struct rp_square_layout {
  int B, N1, N2, W;
  size_t n_bp1, n_bp2, n_up1, n_up2, n_hp;
} rp_square_layout;
int rp_square_plan(const rp_pair* pairs, int n_pairs, const rp_opts* opts,
                   rp_square_layout* layout);
/* Expand the batch's dense outputs into the square tensors of rp_square_plan,
 * in DEVICE memory the caller owns (each sized as rp_square_plan says; NULL
 * skips that tensor).  Every element, padding included, is written: the
 * buffers need no clearing.  Same stream rules as rp_batch_dense_device. */
int rp_batch_square_device(rp_batch* batch, float* bp1, float* bp2, float* up1,
                           float* up2, float* hp);
/* log of the (unscaled) partition function per problem: 3 doubles per pair
 * (s1, s2, s1&s2); parity / debugging aid. */
int rp_batch_fetch_logz(rp_batch* batch, double* logz, size_t n);
int rp_batch_destroy(rp_batch* batch);

/* CUDA-event timing of the last rp_batch_run / rp_run_* on this context. */
typedef struct rp_timing {
  float ms_total;      /* first kernel start -> last kernel end              */
  float ms_h2d, ms_d2h;/* 0 for rp_batch_run                                 */
  int kernel_launches; /* kernels launched by the call                       */
  double alg_flops;    /* dense algorithmic flops (SURVEY 8d F_pair summed)  */
  /* the launch that carries most of those flops, timed by itself (events around it on its stream):
   * 0 = band kernel, long class (<512,1>), 1 = band kernel, short class (<256,2>), 2 = general kernel */
  int dominant_kind;
  float ms_dominant;
  double alg_flops_dominant;   /* F_mcc summed over the problems of that launch */
} rp_timing;
int rp_last_timing(const rp_ctx* ctx, rp_timing* t);

/* Micro-benchmarks used as roofline denominators (fp64 FMA pipe, TFLOP/s;
 * shared-memory read bandwidth, GB/s).  Measured live on the context's GPU. */
int rp_measure_peaks(rp_ctx* ctx, double* fp64_tflops, double* smem_gbs);

/* ------------------------------------------------------------------------ */
/* z-score shuffle batch (host).  Replaces the generator side of the loop at */
/* src/ractip.cpp:1636-1643: srandom(seed); per iteration shuffle(s1,k=2)    */
/* then shuffle(s2,k=2), both always from the ORIGINAL sequences, uShuffle   */
/* semantics (src/ushuffle.c:139-275) on glibc random().  mode is the        */
/* --zscore value: 1 (shuffle s1 only), 2 (s2 only), 12 (both).              */
/* out1/out2: num * n1 / num * n2 chars, shuffle r at out1 + r*n1.           */
/* ------------------------------------------------------------------------ */
int rp_zscore_shuffles(const char* s1, int n1, const char* s2, int n2,
                       int mode, unsigned int seed, int num, int k,
                       char* out1, char* out2);

/* Dense algorithmic flop count F_mcc(n) of SURVEY.md section 8(d). */
double rp_alg_flops_mcc(int n);

/* Which kernel a McCaskill problem of length n (n1+n2 for the two-strand     */
/* problem of rnaduplex, src/ractip.cpp:400-458) runs on, given the per-CTA   */
/* shared-memory limit of the device (bytes; 0 = B200's 232448).  Host        */
/* arithmetic only.  Returns RP_KERNEL_*; *smem_bytes (may be NULL) receives   */
/* the dynamic shared memory the band kernel would need for that length.      */
enum {
  RP_KERNEL_BAND_1CTA = 0,  /* shared-memory band kernel, 512 threads, 1 CTA/SM */
  RP_KERNEL_BAND_2CTA = 1,  /* shared-memory band kernel, 256 threads, 2 CTA/SM */
  RP_KERNEL_GENERAL = 2,    /* HBM-table wavefront kernel (any length), 2 CTA/SM */
  RP_KERNEL_GENERAL_WIDE = 3 /* the same with 128 registers, 1 CTA/SM and split  */
                            /* sums in bands of 10 diagonals: n >= 700.  A batch */
                            /* runs ALL its general-kernel problems in this build */
                            /* when its longest one qualifies; with few such      */
                            /* problems (<= ~90) each runs on a thread-block       */
                            /* cluster of 8 or 16 CTAs (multi-CTA wavefront).      */
};
int rp_kernel_plan(int n, size_t smem_limit, size_t* smem_bytes);

const char* rp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RACTIP_PROB_H */
