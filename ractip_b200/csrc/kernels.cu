// kernels.cu -- sm_100a kernels of the probability stage.
//
// mcc_persistent: one CTA per problem *slot*.  Each CTA pulls problems (one
// RNA, or one two-strand concatenation) from a global queue ordered by
// decreasing cost, runs the whole inside/outside/unpaired-window pipeline of
// mcc_driver.h on it inside its private HBM workspace slot, writes the fp32
// results in the reference's layouts, and pulls the next one.  The grid is
// sized to the number of CTAs that are simultaneously resident
// (SMs x occupancy), so the whole shuffle batch is ONE launch.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include "kernels.h"
#include "mcc_driver.h"

#ifdef RP_TUNE
#define RP_EXPROF(p) (p)
#else
#define RP_EXPROF(p) false
#endif

namespace rp {

namespace {

// executor of the phase schedules (mcc_driver.h) on the G CTAs that share one problem: one CTA (G = 1) or the CTAs of
// a thread-block cluster (G > 1, launched with __cluster_dims__(G, 1, 1))
template <int G = 1, int NB = 4, int W = BAND>
struct CtaExecT {
  static constexpr int kCtas = G;
  static constexpr bool kShfl = true;   // the split sums run the warp-shuffle forms
  static constexpr int kBatch = NB;   // load-batch depth of the split-sum band phases (mcc_band_shfl.cuh)
  static constexpr int kWide = W;     // diagonals per split-sum band of the general kernel (solve_mcc_wide when > BAND)
  long long* prof;  // optional per-phase cycle counters (RP_PROFILE=1), else null
  __device__ __forceinline__ int nthreads() const { return blockDim.x; }
  template <class F>
  __device__ __forceinline__ void phase(int id, F f) {
    long long t0 = 0;
    if (RP_EXPROF(prof) && threadIdx.x == 0) t0 = clock64();
    f(threadIdx.x);
    __syncthreads();
    if (RP_EXPROF(prof) && threadIdx.x == 0) {
      atomicAdd(reinterpret_cast<unsigned long long*>(prof + id), (unsigned long long)(clock64() - t0));
      atomicAdd(reinterpret_cast<unsigned long long*>(prof + 32 + id), 1ull);
    }
  }
  // G > 1 only: this CTA's rank in the cluster, and the cluster barrier
  __device__ __forceinline__ int rank_begin() const { return (int)cooperative_groups::this_cluster().block_rank(); }
  __device__ __forceinline__ int rank_end() const { return rank_begin() + 1; }
  __device__ __forceinline__ void sync() { cooperative_groups::this_cluster().sync(); }
};

using CtaExec = CtaExecT<>;

}  // namespace

// Instantiated for two register budgets: <2> two CTAs per SM at 64 registers (many short problems
// in flight) and <1> one CTA per SM at 128 registers (long problems: the split-sum band phases keep
// their accumulators, operand windows and four steps' loads in registers without spilling, and half
// as many problem histories compete for the L2).
// <1, W> with W > BAND sums the split sums in wide bands (solve_mcc_wide): W-fold reuse of every element
// streamed from HBM.
template <int MINB, int W>
__global__ void __launch_bounds__(RP_MCC_THREADS, MINB) mcc_persistent(BatchDev b) {
  extern __shared__ double smem_raw[];
  __shared__ int s_next;
  CtaExecT<1, (MINB >= 2 ? 2 : 4), W> ex;
  ex.prof = b.prof;
  Shared sh;
  carve_shared(sh, smem_raw, blockDim.x, W);
  for (;;) {
    if (threadIdx.x == 0) s_next = atomicAdd(b.counter, 1);
    __syncthreads();
    const int q = s_next;
    __syncthreads();
    if (q >= b.nprob) break;
    const Problem p = b.probs[b.order[q]];
    if (p.kind == KIND_DUPLEX) continue;  // handled by duplex_kernel
    Ctx c;
    bind_ctx(c, b.model, b.seq + p.seq_off - 1, p, b.ws + (size_t)blockIdx.x * b.slot_stride);
    c.dbg = b.dbg;
    if (W > BAND) solve_mcc_wide(ex, c, p, b.dense, b.logz, sh);
    else solve_mcc(ex, c, p, b.dense, b.logz, sh);
  }
}

// mcc_cluster_kernel: the multi-CTA wavefront for long problems when there are few of them (a single long
// pair rather than a shuffle batch).  A cluster of G CTAs works on one problem (solve_mcc_wide); clusters
// pull problems from the same cost-ordered queue, one workspace slot each.  G = 16 (beyond the portable
// cluster size, opted in at launch) when there are at most sm_count/16 problems, else 8.
template <int W, int G>
__global__ void __cluster_dims__(G, 1, 1) __launch_bounds__(RP_MCC_THREADS, 1) mcc_cluster_kernel(BatchDev b) {
  namespace cg = cooperative_groups;
  extern __shared__ double smem_raw[];
  __shared__ int s_next;
  cg::cluster_group cl = cg::this_cluster();
  CtaExecT<G, 4, W> ex;
  ex.prof = b.prof;
  Shared sh;
  carve_shared(sh, smem_raw, blockDim.x, W);
  const int cid = blockIdx.x / G;
  for (;;) {
    if (cl.block_rank() == 0 && threadIdx.x == 0) s_next = atomicAdd(b.counter, 1);
    cl.sync();
    const int q = *cl.map_shared_rank(&s_next, 0);   // rank 0's copy, through distributed shared memory
    cl.sync();                                       // everybody has read it before rank 0 draws again
    if (q >= b.nprob) break;
    const Problem p = b.probs[b.order[q]];
    if (p.kind == KIND_DUPLEX) continue;
    Ctx c;
    bind_ctx(c, b.model, b.seq + p.seq_off - 1, p, b.ws + (size_t)cid * b.slot_stride);
    c.dbg = b.dbg;
    solve_mcc_wide(ex, c, p, b.dense, b.logz, sh);
  }
}

// mcc_band_kernel: the shared-memory band formulation (mcc_band.h).  Same persistent-CTA queue as
// mcc_persistent, but the interior-loop operands of the last 32 diagonals live in a shared-memory
// ring and are summed densely, 8 cells per thread, from registers.  Dynamic shared memory =
// band_shared_bytes(longest problem of the launch, T).  Instantiated for the two launch shapes:
// <512,1> one CTA per SM (rings of up to ~215 nt) and <256,2> two CTAs per SM (short problems).
template <int T, int MINB>
__global__ void __launch_bounds__(T, MINB) mcc_band_kernel(BatchDev b) {
  extern __shared__ double smem_raw[];
  __shared__ int s_next;
  CtaExec ex;
  ex.prof = b.prof;
  for (;;) {
    if (threadIdx.x == 0) s_next = atomicAdd(b.counter, 1);
    __syncthreads();
    const int q = s_next;
    __syncthreads();
    if (q >= b.nprob) break;
    const int job = b.order[q], pi = job & (RP_JOB_UNPAIRED - 1);
    const Problem p = b.probs[pi];
    Ctx c;
    bind_ctx(c, b.model, b.seq + p.seq_off - 1, p, p.ws_off >= 0 ? b.ws_up + p.ws_off : b.ws + (size_t)blockIdx.x * b.slot_stride);
    c.dbg = b.dbg;
    c.prof = b.prof;
    if (job & RP_JOB_UNPAIRED) {
      // The unpaired-window pass of a problem whose wavefronts ran as an earlier job (maybe on another SM; its tables sit
      // in the problem's private workspace).  Such jobs come after ALL wavefront jobs in the queue, so the job waited for
      // is running or done: no deadlock.  Finer jobs = a shorter tail when there are few problems per SM.
      if (threadIdx.x == 0) {
        while (atomicAdd(b.done + pi, 0) == 0) __nanosleep(500);
        __threadfence();
      }
      __syncthreads();
      solve_band_unpaired(ex, c, p, b.dense, smem_raw);
      continue;
    }
    solve_band(ex, c, p, b.dense, b.logz, smem_raw);
    if (p.defer_up) {   // publish: the tables are complete (release; the unpaired-window job acquires)
      __threadfence();
      __syncthreads();
      if (threadIdx.x == 0) atomicExch(b.done + pi, 1);
    }
  }
}

// unstru_kernel: the unpaired-window pass (pf_unstru, src/ractip.cpp:371-375) of the single-strand problems the
// band kernel has finished, as a launch of its own.  The pass needs no shared-memory ring and is bound by its
// table walks, every table several times: ONE 768-thread CTA per SM (80 registers) keeps 24 warps in flight -- the
// band kernel's shape allows 16 -- and 148 problems' tables (about 1 MB each) resident, which the 126 MB L2 nearly
// holds; three 256-thread CTAs per SM have the same warps but three times the resident problems, and every re-read
// of a table goes to DRAM (38.1 against 36.2 ms per 1000-pair step; 512 x 1: 36.9, 1024 x 1 at 64 registers: 36.4,
// 256 x 2: 39.0, 128 x 6: 41.5).  Each problem's tables sit in its private workspace (Problem::ws_off).
constexpr int RP_UP_THREADS = 768;
__global__ void __launch_bounds__(RP_UP_THREADS, 1) unstru_kernel(BatchDev b) {
  __shared__ int s_next;
  __shared__ double s_gfull[(MAXLOOP + 1) * GROW_LD];
  __shared__ uint8_t s_seq[RP_SMEM_SEQ + 8];
  CtaExec ex;
  ex.prof = b.prof;
  const int T = blockDim.x;
  for (int x = threadIdx.x; x < (MAXLOOP + 1) * GROW_LD; x += T) s_gfull[x] = (&b.model->gfull[0][0])[x];
  for (;;) {
    if (threadIdx.x == 0) s_next = atomicAdd(b.counter, 1);
    __syncthreads();
    const int q = s_next;
    __syncthreads();
    if (q >= b.nprob) break;
    const Problem p = b.probs[b.order[q]];
    Ctx c;
    bind_ctx(c, b.model, b.seq + p.seq_off - 1, p, b.ws_up + p.ws_off);
    c.dbg = b.dbg;
    c.prof = b.prof;
    if (p.n + 2 <= RP_SMEM_SEQ) stage_sequence(ex, c, s_seq, [](int) {});
    inside_end(c);   // 1/Z from the finished inside table
    emit_unpaired(ex, c, p, b.dense, *b.model, s_gfull);
  }
}

// ---------------------------------------------------------------------------
// pf_duplex (--duplex): log-space forward/backward over pure duplexes.
// Restates reference src/pf_duplex.c:128-164 (fw), :166-206 (bk), :97-103 (pr)
// with LogAdd of :34-40.  One CTA per problem; cells on the wavefront
// w = i + (n2 - j) are independent (every predecessor (k,l) has k<i, l>j).
// The backward table is computed in the equivalent pull form
//   bk(k,l) = logsum( close(k,l), bk(i,j) - E(k,l;i,j)  for i>k, j<l ).
// ---------------------------------------------------------------------------
namespace {

__device__ __forceinline__ double log_add(double x, double y) {
  if (x == -INFINITY) return y;
  if (y == -INFINITY) return x;
  return x > y ? log1p(exp(y - x)) + x : log1p(exp(x - y)) + y;
}

__device__ __forceinline__ int i_ext_loop(const DevModel& M, int type, int s5, int s3) {
  int e = 0;
  if (s5 >= 0 && s3 >= 0) e += M.i_mmExt[type][s5][s3];
  else if (s5 >= 0) e += M.i_dangle5[type][s5];
  else if (s3 >= 0) e += M.i_dangle3[type][s3];
  if (type > 2) e += M.i_TermAU;
  return e;
}

__device__ __forceinline__ int i_int_loop(const DevModel& M, int n1, int n2, int type, int type2, int si1, int sj1,
                                          int sp1, int sq1) {
  const int nl = n1 > n2 ? n1 : n2, ns = n1 > n2 ? n2 : n1;
  if (nl == 0) return M.i_stack[type][type2];
  if (ns == 0) {
    int e = M.i_bulge[nl];
    if (nl == 1) e += M.i_stack[type][type2];
    else {
      if (type > 2) e += M.i_TermAU;
      if (type2 > 2) e += M.i_TermAU;
    }
    return e;
  }
  if (ns == 1) {
    if (nl == 1) return M.i_int11[type][type2][si1][sj1];
    if (nl == 2) return n1 == 1 ? M.i_int21[type][type2][si1][sq1][sj1] : M.i_int21[type2][type][sq1][si1][sp1];
    int e = M.i_internal[nl + 1];
    e += min(M.i_MAX_NINIO, (nl - ns) * M.i_ninio);
    return e + M.i_mm1n[type][si1][sj1] + M.i_mm1n[type2][sq1][sp1];
  }
  if (ns == 2) {
    if (nl == 2) return M.i_int22[type][type2][si1][sp1][sq1][sj1];
    if (nl == 3) return M.i_internal[5] + M.i_ninio + M.i_mm23[type][si1][sj1] + M.i_mm23[type2][sq1][sp1];
  }
  int e = M.i_internal[nl + ns];
  e += min(M.i_MAX_NINIO, (nl - ns) * M.i_ninio);
  return e + M.i_mmI[type][si1][sj1] + M.i_mmI[type2][sq1][sp1];
}

}  // namespace

__global__ void __launch_bounds__(256) duplex_kernel(BatchDev b) {
  __shared__ double red[256];
  const DevModel& M = *b.model;
  for (int q = blockIdx.x; q < b.nprob; q += gridDim.x) {
    const Problem p = b.probs[b.order[q]];
    if (p.kind != KIND_DUPLEX) continue;
    const int n1 = p.n1, n2 = p.n2;
    const uint8_t* A = b.seq + p.seq_off - 1;       // A[1..n1]
    const uint8_t* B = A + n1;                      // B[1..n2] (stored right after s1)
    double* ws = b.ws + (size_t)(blockIdx.x % b.nslots) * b.slot_stride;
    const int ld = n2 + 2;
    double* fw = ws;
    double* bk = ws + (size_t)(n1 + 2) * ld;
    const double kT = M.kT;
    const int tid = threadIdx.x, T = blockDim.x;
    for (int x = tid; x < (n1 + 2) * ld; x += T) { fw[x] = -INFINITY; bk[x] = -INFINITY; }
    __syncthreads();
    // forward: wavefront w = i + (n2 - j), i in 1..n1, j in 1..n2
    double esum = -INFINITY;
    for (int w = 1; w <= n1 + n2 - 1; w++) {
      for (int i = 1 + tid; i <= n1; i += T) {
        const int j = n2 - (w - i);
        if (j < 1 || j > n2) continue;
        const int type = pair_type(A[i] & 7, B[j] & 7);
        if (!type) continue;
        int E = M.i_DuplexInit + i_ext_loop(M, type, i > 1 ? (A[i - 1] & 7) : -1, j < n2 ? (B[j + 1] & 7) : -1);
        double f = -E * 10. / kT;
        for (int k = i - 1; k > 0 && k > i - MAXLOOP - 2; k--)
          for (int l = j + 1; l <= n2; l++) {
            if (i - k + l - j - 2 > MAXLOOP) break;
            const int type2 = pair_type(A[k] & 7, B[l] & 7);
            if (!type2) continue;
            E = i_int_loop(M, i - k - 1, l - j - 1, type2, rtype(type), A[k + 1] & 7, B[l - 1] & 7, A[i - 1] & 7,
                           B[j + 1] & 7);
            f = log_add(f, fw[k * ld + l] - E * 10. / kT);
          }
        fw[i * ld + j] = f;
        E = i_ext_loop(M, rtype(type), j > 1 ? (B[j - 1] & 7) : -1, i < n1 ? (A[i + 1] & 7) : -1);
        esum = log_add(esum, f - E * 10. / kT);
      }
      __syncthreads();
    }
    // reduce the per-thread partial log-sums (fixed order: deterministic)
    red[tid] = esum;
    __syncthreads();
    if (tid == 0) {
      double s = -INFINITY;
      for (int t = 0; t < T; t++) s = log_add(s, red[t]);
      red[0] = s;
    }
    __syncthreads();
    const double Esum = red[0];
    __syncthreads();
    // backward, pull form: wavefront from the far corner (i=n1, j=1) inwards
    for (int w = n1 + n2 - 1; w >= 1; w--) {
      for (int k = 1 + tid; k <= n1; k += T) {
        const int l = n2 - (w - k);
        if (l < 1 || l > n2) continue;
        const int type2 = pair_type(A[k] & 7, B[l] & 7);
        if (!type2) continue;
        int E = i_ext_loop(M, rtype(type2), l > 1 ? (B[l - 1] & 7) : -1, k < n1 ? (A[k + 1] & 7) : -1);
        double v = -E * 10. / kT;
        for (int i = k + 1; i <= n1 && i < k + MAXLOOP + 2; i++)
          for (int j = l - 1; j >= 1; j--) {
            if (i - k + l - j - 2 > MAXLOOP) break;
            const int type = pair_type(A[i] & 7, B[j] & 7);
            if (!type) continue;
            E = i_int_loop(M, i - k - 1, l - j - 1, type2, rtype(type), A[k + 1] & 7, B[l - 1] & 7, A[i - 1] & 7,
                           B[j + 1] & 7);
            v = log_add(v, bk[i * ld + j] - E * 10. / kT);
          }
        bk[k * ld + l] = v;
      }
      __syncthreads();
    }
    if (p.out_hp >= 0) {
      float* hp = b.dense + p.out_hp;
      for (int x = tid; x < (n1 + 1) * (n2 + 1); x += T) {
        const int i = x / (n2 + 1), j = x % (n2 + 1);
        hp[x] = (i >= 1 && j >= 1) ? (float)exp(fw[i * ld + j] + bk[i * ld + j] - Esum) : 0.f;
      }
    }
    if (b.logz && tid == 0) b.logz[(size_t)p.pair * 3 + 2] = Esum;
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// thresholded records in the reference's variable-creation order
// (src/ractip.cpp:557-567 for x/y: j ascending, i descending; :598-609 for z:
// i ascending, j ascending; :619-628,639-648 for v/w: start ascending, length ascending).
// One CTA per (pair, list).  The scan order of a list is a flat index k; every thread takes a contiguous range of
// k, counts its hits (pass 1), the CTA turns the counts into offsets, and the thread writes its hits in place
// (pass 2) -- the order is the scan order whatever the thread count, and the loads of a range are independent.
// ---------------------------------------------------------------------------
constexpr int RP_SPARSE_THREADS = 128;
struct SparseList {
  int kind;            // 0 x, 1 y, 2 z, 3 v, 4 w
  const float* src;
  int L, n2, nj, j0, max_w;
  float th;
};
// element k of the scan: (i, j) as stored in the record, and its probability
__device__ __forceinline__ float sparse_at(const SparseList& q, int cj, int ci, int k, int& ri, int& rj) {
  if (q.kind < 2) {          // (column cj, row ci), both 0-based, ci < cj
    ri = ci; rj = cj;
    const int I = ci + 1, J = cj + 1;
    return q.src[(size_t)I * (2 * q.L + 1 - I) / 2 + J];
  }
  if (q.kind == 2) {
    ri = k / q.n2; rj = k - ri * q.n2;
    return q.src[(size_t)(ri + 1) * (q.n2 + 1) + (rj + 1)];
  }
  ri = k / q.nj; rj = q.j0 + (k - ri * q.nj);
  return q.src[(size_t)ri * q.max_w + rj];
}
__global__ void __launch_bounds__(RP_SPARSE_THREADS) sparse_kernel(SparseDev s) {
  __shared__ int s_cnt[RP_SPARSE_THREADS];
  const int pair = blockIdx.x, kind = blockIdx.y, tid = threadIdx.x, T = RP_SPARSE_THREADS;
  const SparsePair sp = s.pairs[pair];
  SparseList q;
  q.kind = kind;
  rp_rec* out;
  int cap, total;
  if (kind < 2) {
    q.L = kind == 0 ? sp.n1 : sp.n2;
    q.src = s.dense + (kind == 0 ? sp.bp1 : sp.bp2);
    q.th = s.th_ss;
    out = s.recs + (kind == 0 ? sp.x : sp.y);
    cap = kind == 0 ? sp.cap_x : sp.cap_y;
    total = q.L * (q.L - 1) / 2;
  } else if (kind == 2) {
    q.n2 = sp.n2;
    q.src = s.dense + sp.hp;
    q.th = s.th_hy;
    out = s.recs + sp.z;
    cap = sp.cap_z;
    total = sp.n1 * sp.n2;
  } else {
    q.L = kind == 3 ? sp.n1 : sp.n2;
    q.src = s.dense + (kind == 3 ? sp.up1_src : sp.up2_src);
    q.th = s.th_ac;
    out = s.recs + (kind == 3 ? sp.v : sp.w);
    cap = kind == 3 ? sp.cap_v : sp.cap_w;
    q.j0 = s.min_w - 1;
    q.max_w = s.max_w;
    q.nj = cap > 0 ? s.max_w - q.j0 : 0;   // cap == 0: accessibility is off, no variables
    total = q.nj > 0 ? q.L * q.nj : 0;
  }
  const int per = (total + T - 1) / T;
  const int k0 = tid * per < total ? tid * per : total, k1 = k0 + per < total ? k0 + per : total;
  // x / y: column of k0 (column cj holds the cj scan positions cj(cj-1)/2 .. ; rows cj-1 down to 0)
  int cj0 = 1, ci0 = 0;
  if (kind < 2 && k0 < k1) {
    cj0 = (int)((1.0 + sqrt(1.0 + 8.0 * (double)k0)) * 0.5);
    while (cj0 * (cj0 - 1) / 2 > k0) cj0--;
    while ((cj0 + 1) * cj0 / 2 <= k0) cj0++;
    ci0 = cj0 - 1 - (k0 - cj0 * (cj0 - 1) / 2);
  }
  int mine = 0;
  for (int pass = 0; pass < 2; pass++) {
    int pos = 0;
    if (pass == 1) {
      __syncthreads();
      for (int t = 0; t < tid; t++) pos += s_cnt[t];
    }
    int cj = cj0, ci = ci0, n = 0;
    for (int k = k0; k < k1; k += 4) {   // four independent loads per round trip
      float p[4];
      int ri[4], rj[4];
      int tj = cj, ti = ci;
#pragma unroll
      for (int u = 0; u < 4; u++) {
        p[u] = 0.f; ri[u] = rj[u] = 0;
        if (k + u < k1) {
          p[u] = sparse_at(q, tj, ti, k + u, ri[u], rj[u]);
          if (--ti < 0) { tj++; ti = tj - 1; }
        }
      }
      cj = tj; ci = ti;
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (k + u < k1 && p[u] > q.th) {
          if (pass == 1 && pos + n < cap) { out[pos + n].i = ri[u]; out[pos + n].j = rj[u]; out[pos + n].p = p[u]; }
          n++;
        }
      }
    }
    if (pass == 0) { mine = n; s_cnt[tid] = n; }
  }
  (void)mine;
  if (tid == T - 1) {
    int count = 0;
    for (int t = 0; t < T; t++) count += s_cnt[t];
    int* cnt = reinterpret_cast<int*>(&s.counts[pair]);   // {n_x, n_y, n_z, overflow, n_v, n_w}
    cnt[kind < 3 ? kind : kind + 1] = count;
    if (count > cap) atomicOr(&cnt[3], 1);
  }
}


// gather the up sections of the dense buffer into the compact float buffer
__global__ void gather_up_kernel(SparseDev s) {
  const SparsePair sp = s.pairs[blockIdx.x];
  for (int x = threadIdx.x; x < sp.n_up1; x += blockDim.x) s.ups[sp.up1_dst + x] = s.dense[sp.up1_src + x];
  for (int x = threadIdx.x; x < sp.n_up2; x += blockDim.x) s.ups[sp.up2_dst + x] = s.dense[sp.up2_src + x];
}

// ---------------------------------------------------------------------------
// roofline denominators measured live: fp64 FMA pipe and shared-memory reads
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) peak_fp64_kernel(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

__global__ void __launch_bounds__(256) peak_smem_kernel(double* out, int iters) {
  __shared__ double buf[4096];
  for (int x = threadIdx.x; x < 4096; x += blockDim.x) buf[x] = x;
  __syncthreads();
  double acc = 0;
  int idx = threadIdx.x;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int u = 0; u < 16; u++) acc += buf[(idx + u * 256) & 4095];
    idx = (idx + 1) & 4095;
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}

// ---------------------------------------------------------------------------
// host-callable launchers
// ---------------------------------------------------------------------------
namespace {
using MccKernel = void (*)(BatchDev);
// minb = 2: 64-register build, BAND-wide sums; minb = 1: 128 registers, bands of 10 diagonals
MccKernel mcc_kernel(int minb, int* w_out) {
  if (minb >= 2) { *w_out = BAND; return mcc_persistent<RP_MCC_MIN_CTAS, BAND>; }
  *w_out = 10;
  return mcc_persistent<1, 10>;
}
}  // namespace

int mcc_max_ctas_per_sm(int minb) {
  int n = 0, w = BAND;
  MccKernel k = mcc_kernel(minb, &w);
  size_t smem = shared_bytes(RP_MCC_THREADS, w);
  if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return 0; }
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, RP_MCC_THREADS, smem) != cudaSuccess) return 0;
  return minb >= 2 ? n : (n > 1 ? 1 : n);
}

cudaError_t launch_mcc(const BatchDev& b, int grid, int minb, cudaStream_t st) {
  int w = BAND;
  MccKernel k = mcc_kernel(minb, &w);
  size_t smem = shared_bytes(RP_MCC_THREADS, w);
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k<<<grid, RP_MCC_THREADS, smem, st>>>(b);
  return cudaGetLastError();
}

cudaError_t launch_mcc_cluster(const BatchDev& b, int nclusters, int ctas, cudaStream_t st) {
  size_t smem = shared_bytes(RP_MCC_THREADS, 10);
  MccKernel k = ctas >= 16 ? mcc_cluster_kernel<10, 16> : mcc_cluster_kernel<10, 8>;
  const int G = ctas >= 16 ? 16 : 8;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (G > 8) {   // beyond the portable cluster size
    e = cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
  }
  k<<<nclusters * G, RP_MCC_THREADS, smem, st>>>(b);
  return cudaGetLastError();
}

namespace {
// launch shapes of the band kernel: 256 threads x 2 CTAs/SM (short problems), 512 threads x 1 CTA/SM.
// (Wider CTAs were measured: <640,1> at 96 registers and <768,1> at 80 compile with 32 / 256 bytes of
// spills and run the 100..137-nt class 6 % / 14 % SLOWER -- the phases have no parallelism left for the
// extra warps.)
MccKernel band_kernel(int threads) { return threads == 256 ? mcc_band_kernel<256, 2> : mcc_band_kernel<512, 1>; }
}  // namespace

int band_max_ctas_per_sm(int threads, size_t smem) {
  int n = 0;
  MccKernel k = band_kernel(threads);
  if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return 0; }
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, threads, smem) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

cudaError_t launch_band(const BatchDev& b, int grid, int threads, size_t smem, cudaStream_t st) {
  MccKernel k = band_kernel(threads);
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  k<<<grid, threads, smem, st>>>(b);
  return cudaGetLastError();
}

int unstru_max_ctas_per_sm() {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, unstru_kernel, RP_UP_THREADS, 0) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
cudaError_t launch_unstru(const BatchDev& b, int grid, cudaStream_t st) {
  unstru_kernel<<<grid, RP_UP_THREADS, 0, st>>>(b);
  return cudaGetLastError();
}

cudaError_t launch_duplex(const BatchDev& b, int grid, cudaStream_t st) {
  duplex_kernel<<<grid, 256, 0, st>>>(b);
  return cudaGetLastError();
}

cudaError_t launch_sparse(const SparseDev& s, int n_pairs, bool with_ups, cudaStream_t st) {
  sparse_kernel<<<dim3(n_pairs, 5), RP_SPARSE_THREADS, 0, st>>>(s);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || !with_ups) return e;
  gather_up_kernel<<<n_pairs, 256, 0, st>>>(s);
  return cudaGetLastError();
}

cudaError_t launch_peak_fp64(double* out, int grid, int iters, cudaStream_t st) {
  peak_fp64_kernel<<<grid, 256, 0, st>>>(out, iters);
  return cudaGetLastError();
}
cudaError_t launch_peak_smem(double* out, int grid, int iters, cudaStream_t st) {
  peak_smem_kernel<<<grid, 256, 0, st>>>(out, iters);
  return cudaGetLastError();
}

}  // namespace rp
