// kernels.h -- launch interface between the C-ABI host layer and kernels.cu
#ifndef RP_KERNELS_H
#define RP_KERNELS_H

#include <cuda_runtime.h>
#include <stdint.h>

#include "mcc_band.h"
#include "mcc_core.h"
#include "mfe_core.h"
#include "ractip_prob.h"

namespace rp {

constexpr int RP_MCC_THREADS = 512;   // threads per CTA of the general kernel
constexpr int RP_MCC_MIN_CTAS = 2;    // CTAs per SM of its 64-register build

struct BatchDev {
  const DevModel* model;
  const uint8_t* seq;      // encoded sequences, one zero byte of padding around each
  const Problem* probs;
  const int* order;        // problem indices by decreasing cost
  int nprob;
  int* counter;            // work-queue head
  double* ws;              // nslots workspace slots
  size_t slot_stride;      // doubles per slot
  int nslots;
  int* done;               // per problem: set when a deferred problem's wavefronts are complete (its unpaired-window job waits on it)
  double* ws_up;           // per-problem workspaces of the problems whose unpaired-window pass is deferred (Problem::ws_off)
  float* dense;            // dense fp32 outputs (reference layouts)
  double* logz;            // 3 per pair, may be null
  long long* prof;         // 64 counters (cycles, calls per phase id) or null
  int dbg;                 // RP_DEBUG_SKIP bits (tuning aid; results are wrong when set)
  unsigned stack_off;      // doubles from perbase to the stacking factors
  // Per-base data of the batch, or null: a PerBaseHead (below), structure-constraint keys (uint16) laid out like seq
  // after it (Problem::constrained & CON_KEYS), stacking pseudo-energy factors (double) laid out like seq at stack_off
  // (CON_STACK), the sample offsets, the unpaired pseudo-energies' pair factors (CON_UNPAIRED).  One pointer, so that the parameter block of every kernel keeps the layout it had
  // before factors and samples.
  const void* perbase;
};

// Head of the per-base block (BatchDev::perbase): the batch's stochastic samples (Problem::constrained & CON_SAMPLE):
// `num` pair tables per sampled problem, problem `which` of pair p at samples + off[3p + which] (rp_sample_plan), where
// off = (const long long*)perbase + off_doubles.  The structure-constraint keys follow the head, at PB_HEAD doubles.
// Unpaired pseudo-energies (Problem::constrained & CON_UNPAIRED): the pair factors upf (double) laid out like seq at
// unp_off, and at unp_lz_off one log-Z term per problem, problem `which` of pair p at [3p + which].
struct PerBaseHead {
  int16_t* samples;   // null: nothing sampled
  unsigned long long seed;
  long long off_doubles;
  long long num;
  long long unp_off;
  long long unp_lz_off;
};
constexpr int PB_HEAD = sizeof(PerBaseHead) / sizeof(double);

struct SparsePair {
  int n1, n2;
  long long bp1, bp2, hp;              // float offsets into the dense buffer
  long long x, y, z;                   // record offsets
  int cap_x, cap_y, cap_z;
  long long up1_src, up2_src, up1_dst, up2_dst;
  int n_up1, n_up2;
  long long v, w;                      // record offsets of the accessible-region lists
  int cap_v, cap_w;
};

struct SparseDev {
  const SparsePair* pairs;
  const float* dense;
  rp_rec* recs;
  float* ups;
  rp_sparse_counts* counts;
  float th_ss, th_hy, th_ac;
  int min_w, max_w;                    // window-length indices min_w-1 .. max_w-1 are scanned (src/ractip.cpp:622)
};

// rp_batch_square_device: the dense outputs of a batch (three problems per pair, in pair order: s1, s2, s1&s2, whose
// out_* offsets locate the pair's sections) expanded into the padded square tensors of rp_square_plan
enum { SQ_BP1 = 0, SQ_BP2, SQ_UP1, SQ_UP2, SQ_HP, SQ_SECTIONS };
struct SquareDev {
  const Problem* probs;
  const float* dense;
  float* out[SQ_SECTIONS];             // null: section skipped
  int N1, N2, W;
  int tiles;                           // 32-row tiles per pair: ceil((max(N1, N2) + 1) / 32)
};

// general kernel, RP_MCC_THREADS threads.  minb = 2: 64-register build, two CTAs per SM; 1: 128 registers, one CTA
// per SM, split sums in bands of 10 diagonals.  Both launches run the instances that apply per-base data (structure
// constraints, stacking and unpaired pseudo-energies, samples) when b.perbase is set, else the ones that compile it out.
int mcc_max_ctas_per_sm(int minb);
cudaError_t launch_mcc(const BatchDev& b, int grid, int minb, cudaStream_t st);
// multi-CTA wavefront: `nclusters` clusters of `ctas` (8 or 16) CTAs, one problem (and one workspace slot) per cluster
cudaError_t launch_mcc_cluster(const BatchDev& b, int nclusters, int ctas, cudaStream_t st);
// mfe_kernel (rp_run_mfe): one CTA per problem of the queue `jobs` (longest first), RP_MFE_THREADS threads, int32
// workspace slots of slot_ints; per-base arrays laid out like seq, null when no problem carries them
constexpr int RP_MFE_THREADS = 512;
struct MfeDev {
  const DevModel* model;
  const uint8_t* seq;
  const uint16_t* key;
  const int32_t* es;
  const int32_t* eu;
  const MfeJob* jobs;
  int njobs;
  int* counter;
  int32_t* ws;
  size_t slot_ints;
  int16_t* structures;
  int32_t* energies;   // 3 per pair; RP_INF stays where no problem writes
};
int mfe_max_ctas_per_sm();
cudaError_t launch_mfe(const MfeDev& m, int grid, cudaStream_t st);
int band_max_ctas_per_sm(int threads, size_t smem);   // threads = 256 (2 CTAs/SM) or 512 (1 CTA/SM)
cudaError_t launch_band(const BatchDev& b, int grid, int threads, size_t smem, cudaStream_t st);
cudaError_t launch_duplex(const BatchDev& b, int grid, cudaStream_t st);
int unstru_max_ctas_per_sm();
cudaError_t launch_unstru(const BatchDev& b, int grid, cudaStream_t st);   // deferred unpaired-window passes: b.order/nprob = their queue
cudaError_t launch_sparse(const SparseDev& s, int n_pairs, bool with_ups, cudaStream_t st);
cudaError_t launch_square(const SquareDev& s, int n_pairs, cudaStream_t st);
cudaError_t launch_peak_fp64(double* out, int grid, int iters, cudaStream_t st);
cudaError_t launch_peak_smem(double* out, int grid, int iters, cudaStream_t st);

}  // namespace rp
#endif
