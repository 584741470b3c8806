// api.cu -- the C ABI of include/ractip_prob.h over the CUDA kernels.
//
// Host-side mirror of what RactIP::solve does before it builds the IP
// (reference src/ractip.cpp:546-548): for every pair, two single-strand
// problems (rnafold: pair probabilities + unpaired windows) and one two-strand
// problem (rnaduplex), batched over all pairs of a call -- the --zscore shuffle
// loop (src/ractip.cpp:1638-1657) hands its whole batch over at once.
//
// There is no CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "dev_model.h"
#include "kernels.h"
#include "plan.h"
#include "ractip_prob.h"

using rp::Problem;

struct rp_ctx {
  int device = 0;
  int sm_count = 0;
  int ctas_per_sm = 0;       // general kernel, 64-register build (two CTAs per SM)
  int ctas_per_sm1 = 0;      // general kernel, 128-register build (one CTA per SM: long problems)
  int up_ctas_per_sm = 0;    // unstru_kernel occupancy
  int mfe_ctas_per_sm = 0;   // mfe_kernel occupancy
  size_t smem_optin = 0;     // max dynamic shared memory per CTA
  rp::RouteSettings route;   // read from the environment at rp_create
  rp::DevModel* d_model = nullptr;
  cudaStream_t own_stream = nullptr;
  cudaStream_t side_stream = nullptr;   // the second band launch shape runs here, so that its CTAs fill the SMs the first one leaves
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaStream_t copy_stream = nullptr;   // rp_batch_fetch_dense: outputs of the long band class leave while the short class still runs
  cudaEvent_t ev_main = nullptr, ev_copy = nullptr;
  cudaEvent_t ev_handoff = nullptr;     // rp_batch_*_device: the reading stream waits for the stream the batch ran on
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[6] = {};
  cudaEvent_t ev_dom[2] = {};   // around the launch that carries most of the algorithmic flops (rp_timing::ms_dominant)
  bool dom_timed = false;
  double* ws = nullptr;       // workspace slots (grow-only)
  size_t ws_bytes = 0;
  rp_timing timing = {};
  bool timing_pending = false;
  bool timed_copies = false;
  std::string err;
  // device buffers of destroyed batches, reused by the next batch (cudaMalloc/cudaFree cost
  // milliseconds and cudaFree synchronises the device: fatal for the one-shot host calls)
  std::vector<std::pair<void*, size_t>> pool_free;
  std::vector<std::pair<void*, size_t>> pool_live;
  // lifetime: batches hold a reference; rp_destroy with batches alive only marks the context closed, the last
  // rp_batch_destroy tears it down (a batch handle never outlives the memory it points into)
  int live_batches = 0;
  bool closing = false;
  cudaStream_t ws_stream = nullptr;   // stream of the last launch that used the workspace / a pooled buffer
#ifdef RP_TUNE
  bool profile = false;               // RP_PROFILE: per-phase cycle counters, printed after each run
  int debug_skip = 0;                 // RP_DEBUG_SKIP bits (results are wrong when set)
  long long* d_prof = nullptr;        // RP_PROFILE counters (per context: per device)
#endif
};

struct rp_batch {
  rp_ctx* ctx = nullptr;
  int n_pairs = 0;
  rp_opts opts = {};
  rp::BatchPlan plan;
  // device
  uint8_t* d_seq = nullptr;
  // per-base data (BatchDev::perbase): PerBaseHead, BatchPlan::key, then BatchPlan::stack from stack_off doubles on, then
  // the sample offsets; null when no problem is constrained, carries pseudo-energies or is sampled
  double* d_perbase = nullptr;
  unsigned stack_off = 0;
  Problem* d_probs = nullptr;
  int* d_order = nullptr;
  int* d_counter = nullptr;
  float* d_dense = nullptr;
  double* d_logz = nullptr;
  int* d_done = nullptr;      // completion flags of the deferred problems (indexed by problem)
  int16_t* d_samples = nullptr;   // stochastic samples (BatchPlan::sample_total int16), null when nothing is sampled
  cudaStream_t last_stream = nullptr;   // stream the batch last ran on (rp_set_stream may have moved the context on)
  // sparse
  std::vector<rp_sparse_layout> slayout;
  size_t total_recs = 0, total_upf = 0;
  rp::SparsePair* d_spairs = nullptr;
  rp_rec* d_recs = nullptr;
  float* d_ups = nullptr;
  rp_sparse_counts* d_counts = nullptr;
};

namespace {

thread_local std::string g_err;

int fail(rp_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  g_err = msg;
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(ctx, RP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));     \
  } while (0)

int ensure_workspace(rp_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->ws_bytes) return RP_OK;
  if (ctx->ws) {
    if (ctx->ws_stream && ctx->ws_stream != ctx->stream) CU(cudaStreamSynchronize(ctx->ws_stream));
    CU(cudaStreamSynchronize(ctx->stream));
    CU(cudaFree(ctx->ws));
    ctx->ws = nullptr;
    ctx->ws_bytes = 0;
  }
  cudaError_t e = cudaMalloc(&ctx->ws, bytes);
  if (e != cudaSuccess) {   // give the cached buffers of destroyed batches back to the driver and retry once
    cudaGetLastError();
    for (auto& f : ctx->pool_free) cudaFree(f.first);
    ctx->pool_free.clear();
    e = cudaMalloc(&ctx->ws, bytes);
  }
  if (e != cudaSuccess) { ctx->ws = nullptr; return fail(ctx, RP_ERR_CUDA, std::string("cudaMalloc workspace: ") + cudaGetErrorString(e)); }
  ctx->ws_bytes = bytes;
  return RP_OK;
}

size_t pool_cached_bytes(const rp_ctx* ctx) {
  size_t t = 0;
  for (const auto& f : ctx->pool_free) t += f.second;
  return t;
}

size_t pool_cached_bytes(const rp_ctx* ctx);
cudaError_t pool_alloc(rp_ctx* ctx, void** out, size_t bytes) {
  bytes = std::max<size_t>(bytes, 256);
  int best = -1;
  for (size_t k = 0; k < ctx->pool_free.size(); k++)
    if (ctx->pool_free[k].second >= bytes && (best < 0 || ctx->pool_free[k].second < ctx->pool_free[best].second)) best = (int)k;
  if (best >= 0 && ctx->pool_free[best].second <= 4 * bytes + (1 << 20)) {
    *out = ctx->pool_free[best].first;
    ctx->pool_live.push_back(ctx->pool_free[best]);
    ctx->pool_free.erase(ctx->pool_free.begin() + best);
    return cudaSuccess;
  }
  cudaError_t e = cudaMalloc(out, bytes);
  if (e != cudaSuccess) {  // give cached buffers back to the driver and retry once
    for (auto& f : ctx->pool_free) cudaFree(f.first);
    ctx->pool_free.clear();
    e = cudaMalloc(out, bytes);
  }
  if (e == cudaSuccess) ctx->pool_live.emplace_back(*out, bytes);
  return e;
}
template <class T>
cudaError_t pool_alloc(rp_ctx* ctx, T** out, size_t bytes) {
  return pool_alloc(ctx, reinterpret_cast<void**>(out), bytes);
}
void pool_release(rp_ctx* ctx, void* p) {
  if (!p) return;
  for (size_t k = 0; k < ctx->pool_live.size(); k++)
    if (ctx->pool_live[k].first == p) {
      ctx->pool_free.push_back(ctx->pool_live[k]);
      ctx->pool_live.erase(ctx->pool_live.begin() + k);
      // keep the cache bounded: beyond 64 buffers or 8 GB the oldest entries go back to the driver
      while (ctx->pool_free.size() > 64 || pool_cached_bytes(ctx) > ((size_t)8 << 30)) {
        cudaFree(ctx->pool_free.front().first);
        ctx->pool_free.erase(ctx->pool_free.begin());
      }
      return;
    }
  cudaFree(p);
}

// The context's settings from the environment, read once (rp_create).  RP_BAND=0, RP_MCC_LONG_N, RP_CLUSTER=0|8|16 and
// RP_NO_SPLIT_FETCH force routes for tests and A/B comparisons; the tuning build adds RP_PROFILE and RP_DEBUG_SKIP.
void read_settings(rp_ctx* ctx) {
  rp::RouteSettings& s = ctx->route;
  if (const char* e = std::getenv("RP_BAND")) s.band = std::atoi(e) != 0;
  if (const char* e = std::getenv("RP_MCC_LONG_N")) s.mcc_long_n = std::atoi(e);
  if (const char* e = std::getenv("RP_CLUSTER")) {
    const int v = std::atoi(e);
    s.cluster = v >= 16 ? 16 : v > 0 ? 8 : 0;
  }
  s.split_fetch = std::getenv("RP_NO_SPLIT_FETCH") == nullptr;
#ifdef RP_TUNE
  ctx->profile = std::getenv("RP_PROFILE") != nullptr;
  if (const char* e = std::getenv("RP_DEBUG_SKIP")) ctx->debug_skip = std::atoi(e);
#endif
}

rp::DeviceFacts device_facts(rp_ctx* ctx) {
  rp::DeviceFacts f;
  f.sm_count = ctx->sm_count;
  f.smem_optin = ctx->smem_optin;
  f.ctas_per_sm = ctx->ctas_per_sm;
  f.ctas_per_sm1 = ctx->ctas_per_sm1;
  f.up_ctas_per_sm = ctx->up_ctas_per_sm;
  f.mfe_ctas_per_sm = ctx->mfe_ctas_per_sm;
  f.ws_bytes = ctx->ws_bytes;
  f.band_occupancy = rp::band_max_ctas_per_sm;
  f.memory = [ctx]() -> size_t {   // cached buffers are freed on demand
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return SIZE_MAX;   // no budget known: none applied
    return free_b + ctx->ws_bytes + pool_cached_bytes(ctx);
  };
  return f;
}

}  // namespace

extern "C" {

const char* rp_version(void) { return "ractip_b200 0.2 (sm_100a)"; }

const char* rp_strerror(int code) {
  switch (code) {
    case RP_OK: return "ok";
    case RP_ERR_ARG: return "bad argument";
    case RP_ERR_NO_DEVICE: return "no usable CUDA device (the probability stage has no CPU fallback)";
    case RP_ERR_CUDA: return "CUDA error";
    case RP_ERR_IO: return "cannot read file";
    case RP_ERR_FORMAT: return "malformed parameter data";
    case RP_ERR_NO_DEFAULTS: return "requested energy tables are not embedded; load a parameter file";
    case RP_ERR_SEQ: return "bad sequence";
    case RP_ERR_TOO_LONG: return "sequence too long";
    case RP_ERR_CAPACITY: return "output buffer too small";
    case RP_ERR_UNSUPPORTED: return "unsupported model setting";
    default: return "unknown error";
  }
}

const char* rp_last_error(const rp_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

void rp_opts_default(rp_opts* o) {
  if (!o) return;
  // defaults of src/cmdline.c:151-186 as mapped at src/ractip.cpp:1474-1498
  o->max_w = 15; o->min_w = 5; o->th_ss = 0.5f; o->th_hy = 0.1f; o->th_ac = 0.003f; o->use_pf_duplex = 0;
}

// ------------------------------------------------------------------ context
int rp_create(rp_ctx** out, const rp_model* m, int device) {
  rp_ctx* ctx = nullptr;
  if (!out || !m) return fail(nullptr, RP_ERR_ARG, "rp_create: null argument");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev < 1)
    return fail(nullptr, RP_ERR_NO_DEVICE,
                std::string("rp_create: no CUDA device (") + (e == cudaSuccess ? "count 0" : cudaGetErrorString(e)) +
                    "); the probability stage has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(nullptr, RP_ERR_ARG, "rp_create: bad device index");
  std::vector<rp::DevModel> host(1);
  int rc = rp::build_dev_model(*m, host.data());
  if (rc) return fail(nullptr, rc, "rp_create: unsupported model (temperature must be 37, dangles 2)");
  ctx = new rp_ctx;
  ctx->device = device;
  auto bail = [&](int code, const std::string& msg) {
    rp_destroy(ctx);
    return fail(nullptr, code, msg);
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  ctx->sm_count = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess)
    return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  ctx->stream = ctx->own_stream;
  if ((e = cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking)) != cudaSuccess)
    return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaEventCreateWithFlags(&ctx->ev_main, cudaEventDisableTiming)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaEventCreateWithFlags(&ctx->ev_handoff, cudaEventDisableTiming)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  for (auto& ev : ctx->ev)
    if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  for (auto& ev : ctx->ev_dom)
    if ((e = cudaEventCreate(&ev)) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaMalloc(&ctx->d_model, sizeof(rp::DevModel))) != cudaSuccess) return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  if ((e = cudaMemcpy(ctx->d_model, host.data(), sizeof(rp::DevModel), cudaMemcpyHostToDevice)) != cudaSuccess)
    return bail(RP_ERR_CUDA, cudaGetErrorString(e));
  read_settings(ctx);
  ctx->ctas_per_sm = rp::mcc_max_ctas_per_sm(2);
  ctx->ctas_per_sm1 = rp::mcc_max_ctas_per_sm(1);
  ctx->up_ctas_per_sm = rp::unstru_max_ctas_per_sm();
  ctx->mfe_ctas_per_sm = rp::mfe_max_ctas_per_sm();
  if (ctx->ctas_per_sm < 1)
    return bail(RP_ERR_CUDA, "rp_create: kernel image not loadable on this device (built for sm_100a)");
  *out = ctx;
  return RP_OK;
}

int rp_destroy(rp_ctx* ctx) {
  if (!ctx) return RP_OK;
  if (ctx->live_batches > 0) {   // batches still point into this context: the last rp_batch_destroy finishes the job
    ctx->closing = true;
    return RP_OK;
  }
  cudaSetDevice(ctx->device);
  if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
  if (ctx->ws) cudaFree(ctx->ws);
  for (auto& f : ctx->pool_free) cudaFree(f.first);
  for (auto& f : ctx->pool_live) cudaFree(f.first);
  if (ctx->d_model) cudaFree(ctx->d_model);
#ifdef RP_TUNE
  if (ctx->d_prof) cudaFree(ctx->d_prof);
#endif
  for (auto& ev : ctx->ev)
    if (ev) cudaEventDestroy(ev);
  for (auto& ev : ctx->ev_dom)
    if (ev) cudaEventDestroy(ev);
  if (ctx->side_stream) { cudaStreamSynchronize(ctx->side_stream); cudaStreamDestroy(ctx->side_stream); }
  if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
  if (ctx->ev_main) cudaEventDestroy(ctx->ev_main);
  if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
  if (ctx->ev_handoff) cudaEventDestroy(ctx->ev_handoff);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
  return RP_OK;
}

int rp_set_stream(rp_ctx* ctx, void* cuda_stream) {
  if (!ctx) return RP_ERR_ARG;
  ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
  return RP_OK;
}

int rp_get_stream(const rp_ctx* ctx, void** cuda_stream) {
  if (!ctx || !cuda_stream) return RP_ERR_ARG;
  *cuda_stream = ctx->stream;
  return RP_OK;
}

void* rp_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
  return p;
}
void rp_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

// -------------------------------------------------------------------- batch
int rp_batch_destroy(rp_batch* b) {
  if (!b) return RP_OK;
  if (b->ctx) {
    cudaSetDevice(b->ctx->device);
    if (b->last_stream && b->last_stream != b->ctx->stream) cudaStreamSynchronize(b->last_stream);
    cudaStreamSynchronize(b->ctx->stream);
  }
  if (b->ctx) {
    rp_ctx* ctx = b->ctx;
    for (void* p : {(void*)b->d_seq, (void*)b->d_perbase, (void*)b->d_probs, (void*)b->d_order, (void*)b->d_counter, (void*)b->d_dense,
                    (void*)b->d_logz, (void*)b->d_done, (void*)b->d_spairs, (void*)b->d_recs, (void*)b->d_ups, (void*)b->d_counts,
                    (void*)b->d_samples})
      pool_release(ctx, p);
    ctx->live_batches--;
    if (ctx->closing && ctx->live_batches == 0) {
      delete b;
      return rp_destroy(ctx);
    }
  }
  delete b;
  return RP_OK;
}

}  // extern "C"

namespace {
int batch_create(const char* who, rp_ctx* ctx, const rp_pair* pairs, const rp_constraint* cons,
                 const rp_stack_energy* se, int n_pairs, const rp_opts* opts, rp_batch** out,
                 const rp_sample_opts* so = nullptr, const rp_unpaired_energy* ue = nullptr) {
  if (!ctx || !out) return fail(ctx, RP_ERR_ARG, "rp_batch_create: null argument");
  *out = nullptr;
  int rc = rp::check_pairs(pairs, n_pairs, opts);
  if (rc) return fail(ctx, rc, "rp_batch_create: bad pairs/opts");
  for (int p = 0; p < n_pairs; p++)
    if ((long long)pairs[p].n1 + pairs[p].n2 > rp::RP_MAX_N)
      return fail(ctx, RP_ERR_TOO_LONG, "rp_batch_create: n1+n2 exceeds the 32-bit workspace indexing limit (12000 nt)");
  std::string msg;
  if ((rc = rp::check_constraints(pairs, cons, n_pairs, &msg)) != RP_OK) return fail(ctx, rc, std::string(who) + ": " + msg);
  if ((rc = rp::check_stack_energies(pairs, se, n_pairs, &msg)) != RP_OK) return fail(ctx, rc, std::string(who) + ": " + msg);
  if ((rc = rp::check_samples(pairs, n_pairs, opts, so, &msg)) != RP_OK) return fail(ctx, rc, std::string(who) + ": " + msg);
  if ((rc = rp::check_unpaired_energies(pairs, ue, n_pairs, opts, &msg)) != RP_OK) return fail(ctx, rc, std::string(who) + ": " + msg);
  CU(cudaSetDevice(ctx->device));
  rp_batch* b = new rp_batch;
  b->ctx = ctx;
  ctx->live_batches++;
  b->n_pairs = n_pairs;
  b->opts = *opts;
  b->slayout.resize(n_pairs);
  rp_sparse_plan(pairs, n_pairs, opts, b->slayout.data(), &b->total_recs, &b->total_upf);
  if (rp::plan_batch(pairs, n_pairs, opts, device_facts(ctx), ctx->route, &b->plan, cons, se, so, ue) != RP_OK) {
    rp_batch_destroy(b);
    return fail(ctx, RP_ERR_CUDA, "rp_batch_create: band kernel does not fit on this device");
  }
  rp::BatchPlan& p = b->plan;

  auto bail = [&](cudaError_t e, const char* what) {
    rp_batch_destroy(b);
    return fail(ctx, RP_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
  };
  cudaError_t e;
  const size_t np = p.probs.size();
  if ((e = pool_alloc(ctx, &b->d_seq, p.seq.size() + 16)) != cudaSuccess) return bail(e, "cudaMalloc seq");
  if ((e = pool_alloc(ctx, &b->d_probs, std::max<size_t>(1, np) * sizeof(Problem))) != cudaSuccess) return bail(e, "cudaMalloc probs");
  if ((e = pool_alloc(ctx, &b->d_order, std::max<size_t>(1, p.order.size()) * sizeof(int))) != cudaSuccess) return bail(e, "cudaMalloc order");
  if ((e = pool_alloc(ctx, &b->d_done, std::max<size_t>(1, np) * sizeof(int))) != cudaSuccess) return bail(e, "cudaMalloc done");
  if ((e = pool_alloc(ctx, &b->d_counter, 4 * sizeof(int))) != cudaSuccess) return bail(e, "cudaMalloc counter");
  if ((e = pool_alloc(ctx, &b->d_dense, std::max<size_t>(1, p.total_floats) * sizeof(float))) != cudaSuccess) return bail(e, "cudaMalloc dense");
  if ((e = pool_alloc(ctx, &b->d_logz, std::max<size_t>(1, (size_t)n_pairs * 3) * sizeof(double))) != cudaSuccess) return bail(e, "cudaMalloc logz");
  cudaStream_t st = ctx->stream;
  if ((e = cudaMemcpyAsync(b->d_seq, p.seq.data(), p.seq.size(), cudaMemcpyHostToDevice, st)) != cudaSuccess) return bail(e, "H2D seq");
  // per-base data only for batches with a constrained problem (keys), one whose pseudo-energies are not all 0, or a
  // sampled one (the instances that sample are the per-base ones).  One block: PerBaseHead, keys, factors, sample offsets,
  // the unpaired pseudo-energies' pair factors and log-Z terms.
  if (!p.key.empty() || !p.stack.empty() || p.sample_total || !p.unpaired.empty()) {
    const size_t kd = (p.key.size() * sizeof(uint16_t) + sizeof(double) - 1) / sizeof(double);
    b->stack_off = (unsigned)(rp::PB_HEAD + kd);
    const size_t unp_off = b->stack_off + p.stack.size() + 3 * (size_t)n_pairs;
    std::vector<double> blk(unp_off + p.unpaired.size() + p.unpaired_lz.size(), 0.);
    rp::PerBaseHead h = {};
    h.unp_off = (long long)unp_off;
    h.unp_lz_off = (long long)(unp_off + p.unpaired.size());
    std::copy(p.unpaired.begin(), p.unpaired.end(), blk.begin() + unp_off);
    std::copy(p.unpaired_lz.begin(), p.unpaired_lz.end(), blk.begin() + h.unp_lz_off);
    if (p.sample_total) {
      if ((e = pool_alloc(ctx, &b->d_samples, p.sample_total * sizeof(int16_t))) != cudaSuccess) return bail(e, "cudaMalloc samples");
      if ((e = cudaMemsetAsync(b->d_samples, 0, p.sample_total * sizeof(int16_t), st)) != cudaSuccess) return bail(e, "memset samples");
      h.samples = b->d_samples;
      h.seed = p.sample_seed;
      h.num = p.sample_num;
      h.off_doubles = (long long)(b->stack_off + p.stack.size());
      long long* off = reinterpret_cast<long long*>(blk.data() + h.off_doubles);
      for (int k = 0; k < n_pairs; k++) {
        const rp_sample_layout& L = p.sample_layout[k];
        off[3 * k] = (long long)L.s1; off[3 * k + 1] = (long long)L.s2; off[3 * k + 2] = (long long)L.co;
      }
    }
    std::memcpy(blk.data(), &h, sizeof h);
    if (!p.key.empty()) std::memcpy(blk.data() + rp::PB_HEAD, p.key.data(), p.key.size() * sizeof(uint16_t));
    std::copy(p.stack.begin(), p.stack.end(), blk.begin() + b->stack_off);
    if ((e = pool_alloc(ctx, &b->d_perbase, blk.size() * sizeof(double))) != cudaSuccess) return bail(e, "cudaMalloc per-base data");
    if ((e = cudaMemcpyAsync(b->d_perbase, blk.data(), blk.size() * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess)
      return bail(e, "H2D per-base data");
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return bail(e, "sync");   // blk is released at the end of the block
  }
  if (np) {
    if ((e = cudaMemcpyAsync(b->d_probs, p.probs.data(), np * sizeof(Problem), cudaMemcpyHostToDevice, st)) != cudaSuccess) return bail(e, "H2D probs");
    if (!p.order.empty() && (e = cudaMemcpyAsync(b->d_order, p.order.data(), p.order.size() * sizeof(int), cudaMemcpyHostToDevice, st)) != cudaSuccess) return bail(e, "H2D order");
  }
  if (p.has_single && (e = cudaMemsetAsync(b->d_dense, 0, std::max<size_t>(1, p.total_floats) * sizeof(float), st)) != cudaSuccess) return bail(e, "memset dense");
  if ((e = cudaMemsetAsync(b->d_logz, 0, std::max<size_t>(1, (size_t)n_pairs * 3) * sizeof(double), st)) != cudaSuccess) return bail(e, "memset logz");
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return bail(e, "sync");  // the host copies are complete
  std::vector<uint8_t>().swap(p.seq);   // the sequences live on the device from here
  std::vector<uint16_t>().swap(p.key);
  std::vector<double>().swap(p.stack);
  std::vector<double>().swap(p.unpaired);
  *out = b;
  return RP_OK;
}
}  // namespace

extern "C" {

int rp_batch_create(rp_ctx* ctx, const rp_pair* pairs, int n_pairs, const rp_opts* opts, rp_batch** out) {
  return batch_create("rp_batch_create", ctx, pairs, nullptr, nullptr, n_pairs, opts, out);
}

int rp_batch_create_constrained(rp_ctx* ctx, const rp_pair* pairs, const rp_constraint* cons, int n_pairs,
                                const rp_opts* opts, rp_batch** out) {
  return batch_create("rp_batch_create_constrained", ctx, pairs, cons, nullptr, n_pairs, opts, out);
}

int rp_batch_create_soft(rp_ctx* ctx, const rp_pair* pairs, const rp_constraint* cons, const rp_stack_energy* se,
                         int n_pairs, const rp_opts* opts, rp_batch** out) {
  return batch_create("rp_batch_create_soft", ctx, pairs, cons, se, n_pairs, opts, out);
}

int rp_batch_create_sampled(rp_ctx* ctx, const rp_pair* pairs, const rp_constraint* cons, const rp_stack_energy* se,
                            int n_pairs, const rp_opts* opts, const rp_sample_opts* so, rp_batch** out) {
  return batch_create("rp_batch_create_sampled", ctx, pairs, cons, se, n_pairs, opts, out, so);
}

int rp_batch_create_probed(rp_ctx* ctx, const rp_pair* pairs, const rp_constraint* cons, const rp_stack_energy* se,
                           const rp_unpaired_energy* ue, int n_pairs, const rp_opts* opts, const rp_sample_opts* so,
                           rp_batch** out) {
  return batch_create("rp_batch_create_probed", ctx, pairs, cons, se, n_pairs, opts, out, so, ue);
}

int rp_batch_run(rp_batch* b) {
  if (!b) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  const rp::BatchPlan& p = b->plan;
  CU(cudaSetDevice(ctx->device));
  ctx->timing = rp_timing{};
  ctx->timing.alg_flops = p.alg_flops;
  if (p.probs.empty()) { ctx->timing_pending = false; return RP_OK; }
  // the launches run one after the other (the band classes side by side) and share the workspace
  int rc = ensure_workspace(ctx, p.ws_doubles * sizeof(double));
  if (rc) return rc;
  const int n_bandall = p.n_band[0] + p.n_band[1];
  rp::BatchDev d;
  d.model = ctx->d_model; d.seq = b->d_seq; d.perbase = b->d_perbase; d.stack_off = b->stack_off; d.probs = b->d_probs; d.order = b->d_order + n_bandall; d.nprob = p.n_general;
  d.counter = b->d_counter; d.ws = ctx->ws; d.slot_stride = p.slot_doubles; d.nslots = std::max(p.grid, 1);
  d.dense = b->d_dense; d.logz = b->d_logz;
  d.ws_up = ctx->ws + p.ws_up; d.done = b->d_done;
  d.prof = nullptr;
  d.dbg = 0;
#ifdef RP_TUNE
  d.dbg = ctx->debug_skip;
  if (ctx->profile) {
    if (!ctx->d_prof) CU(cudaMalloc(&ctx->d_prof, 64 * sizeof(long long)));
    CU(cudaMemsetAsync(ctx->d_prof, 0, 64 * sizeof(long long), ctx->stream));
    d.prof = ctx->d_prof;
  }
#endif
  ctx->dom_timed = false;
  ctx->timing.dominant_kind = p.dom_kind;
  ctx->timing.alg_flops_dominant = p.dom_flops;
  ctx->timing.ms_dominant = 0;
  cudaStream_t st = ctx->stream;
  b->last_stream = st;
  ctx->ws_stream = st;
  CU(cudaMemsetAsync(b->d_counter, 0, 4 * sizeof(int), st));
  if (p.n_defer) CU(cudaMemsetAsync(b->d_done, 0, p.probs.size() * sizeof(int), st));
  CU(cudaEventRecord(ctx->ev[0], st));
  int launches = 0;
  if (p.n_band[0] && p.n_band[1]) CU(cudaEventRecord(ctx->ev_fork, st));   // inputs and counters are ready here
  for (int k = 0; k < 2; k++) {
    if (!p.n_band[k]) continue;
    rp::BatchDev db = d;
    db.order = b->d_order + (k ? p.n_band[0] : 0); db.nprob = p.n_band[k];
    db.counter = b->d_counter + 1 + k;
    db.ws = ctx->ws + p.ws_band[k]; db.slot_stride = p.band_slot[k]; db.nslots = p.band_grid[k];
    cudaStream_t ls = st;
    if (k == 1 && p.n_band[0]) {   // the short class runs on the side stream (forked before the first launch)
      CU(cudaStreamWaitEvent(ctx->side_stream, ctx->ev_fork, 0));
      ls = ctx->side_stream;
    }
    if (p.dom_kind == k) CU(cudaEventRecord(ctx->ev_dom[0], ls));
    CU(rp::launch_band(db, p.band_grid[k], rp::BAND_THREADS[k], p.band_smem[k], ls));
    if (p.dom_kind == k) { CU(cudaEventRecord(ctx->ev_dom[1], ls)); ctx->dom_timed = true; }
    if (k == 0 && p.split_fetch) CU(cudaEventRecord(ctx->ev_main, st));   // the long class's outputs are final here
    if (ls != st) {                 // join before anything else of the batch runs
      CU(cudaEventRecord(ctx->ev_join, ls));
      CU(cudaStreamWaitEvent(st, ctx->ev_join, 0));
    }
    launches++;
  }
  if (p.up_mode == 1) {   // the unpaired-window passes of the band classes, after both of their launches (the streams have joined)
    rp::BatchDev du = d;
    du.order = b->d_order + n_bandall + p.n_general; du.nprob = p.n_defer;
    du.counter = b->d_counter + 3;
    CU(rp::launch_unstru(du, p.up_grid, st));
    launches++;
  }
  if (p.n_mcc > 0) {
    if (p.dom_kind == 2) CU(cudaEventRecord(ctx->ev_dom[0], st));
    // a cluster shape the device (or its current partitioning) cannot schedule fails at launch, before
    // anything ran: fall back to the smaller cluster, then to one CTA per problem
    bool launched = false;
    for (int G = p.cluster; G && !launched; G = G == 16 ? 8 : 0) {
      const int ncl = std::max(1, std::min({p.n_mcc, p.grid, ctx->sm_count / G}));
      if (rp::launch_mcc_cluster(d, ncl, G, st) == cudaSuccess) launched = true;
      else cudaGetLastError();
    }
    if (!launched) CU(rp::launch_mcc(d, p.grid, p.mcc_minb, st));
    if (p.dom_kind == 2) { CU(cudaEventRecord(ctx->ev_dom[1], st)); ctx->dom_timed = true; }
    launches++;
  }
  if (p.n_duplex > 0) {
    CU(rp::launch_duplex(d, p.grid, st));
    launches++;
  }
  CU(cudaEventRecord(ctx->ev[1], st));
#ifdef RP_TUNE
  if (ctx->profile) {
    long long h[64];
    CU(cudaMemcpyAsync(h, ctx->d_prof, sizeof h, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    static const char* names[32] = {"stage", "prologue", "prologue2", "inside_A", "inside_B", "generic_in", "generic_out", "outside_A", "outside_B", "write_bp", "un_items", "un_domrows", "un_domcols", "un_windows", "write_hp", "logz", "band_A", "band_B", "collect", "sample", "", "", "", "", "finish_in.loads(t0)", "finish_in.rest(t0)", "bandA_in.head(t0)", "bandA_in.main(t0)", "bandA_in.tail(t0)", "bandA_out.PR(t0)", "bandA_out.need(t0)", "bandA_out.ML(t0)"};
    long long tot = 0;
    for (int k = 0; k < 20; k++) tot += h[k];   // the phase counters (PH_COUNT, mcc_driver.h)
    for (int k = 0; k < 32; k++)
      if (h[32 + k]) std::fprintf(stderr, "[rp_profile] %-11s %6.2f%%  calls %9lld  cycles/call %9.0f\n", names[k], 100.0 * h[k] / tot, h[32 + k], (double)h[k] / h[32 + k]);
  }
#endif
  ctx->timing.kernel_launches = launches;
  ctx->timing_pending = true;
  ctx->timed_copies = false;
  return RP_OK;
}

int rp_batch_sync(rp_batch* b) {
  if (!b) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  CU(cudaStreamSynchronize(ctx->stream));
  return RP_OK;
}

int rp_batch_fetch_dense(rp_batch* b, float* out, size_t out_floats) {
  if (!b || !out) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  const rp::BatchPlan& p = b->plan;
  if (out_floats < p.total_floats) return fail(ctx, RP_ERR_CAPACITY, "rp_batch_fetch_dense: buffer too small");
  CU(cudaSetDevice(ctx->device));
  CU(cudaEventRecord(ctx->ev[2], ctx->stream));
  if (p.total_floats && p.split_fetch) {
    // long-class sections: on the copy stream, as soon as the long class is done (ev_main), while the short class
    // still computes; short-class sections: on the main stream, which has joined the side stream
    const size_t pitch = p.pair_stride * sizeof(float);
    CU(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_main, 0));
    for (const auto& sc : p.sect_long)
      CU(cudaMemcpy2DAsync(out + sc.first, pitch, b->d_dense + sc.first, pitch, sc.second * sizeof(float), (size_t)b->n_pairs,
                           cudaMemcpyDeviceToHost, ctx->copy_stream));
    CU(cudaEventRecord(ctx->ev_copy, ctx->copy_stream));
    for (const auto& sc : p.sect_short)
      CU(cudaMemcpy2DAsync(out + sc.first, pitch, b->d_dense + sc.first, pitch, sc.second * sizeof(float), (size_t)b->n_pairs,
                           cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));
  } else if (p.total_floats) {
    CU(cudaMemcpyAsync(out, b->d_dense, p.total_floats * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  }
  CU(cudaEventRecord(ctx->ev[3], ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->timed_copies = true;
  return RP_OK;
}

}  // extern "C" (reopened below)

namespace {
int sparse_prepare(rp_batch* b) {
  rp_ctx* ctx = b->ctx;
  const int np = b->n_pairs;
  if (b->d_spairs || np == 0) return RP_OK;
  std::vector<rp::SparsePair> sp(np);
  for (int p = 0; p < np; p++) {
    const rp_dense_layout& L = b->plan.layout[p];
    const rp_sparse_layout& S = b->slayout[p];
    rp::SparsePair& q = sp[p];
    q.n1 = b->plan.probs[3 * p].n; q.n2 = b->plan.probs[3 * p + 1].n;
    q.bp1 = (long long)L.bp1; q.bp2 = (long long)L.bp2; q.hp = (long long)L.hp;
    q.x = (long long)S.x; q.y = (long long)S.y; q.z = (long long)S.z;
    q.cap_x = (int)S.cap_x; q.cap_y = (int)S.cap_y; q.cap_z = (int)S.cap_z;
    q.up1_src = (long long)L.up1; q.up2_src = (long long)L.up2;
    q.up1_dst = (long long)S.up1; q.up2_dst = (long long)S.up2;
    q.n_up1 = (int)S.n_up1; q.n_up2 = (int)S.n_up2;
    q.v = (long long)S.v; q.w = (long long)S.w;
    q.cap_v = (int)S.cap_v; q.cap_w = (int)S.cap_w;
  }
  CU(pool_alloc(ctx, &b->d_spairs, np * sizeof(rp::SparsePair)));
  CU(cudaMemcpy(b->d_spairs, sp.data(), np * sizeof(rp::SparsePair), cudaMemcpyHostToDevice));
  return RP_OK;
}

int sparse_launch(rp_batch* b, rp_rec* d_recs, float* d_ups, rp_sparse_counts* d_counts) {
  rp_ctx* ctx = b->ctx;
  rp::SparseDev s;
  s.pairs = b->d_spairs; s.dense = b->d_dense; s.recs = d_recs; s.ups = d_ups; s.counts = d_counts;
  s.th_ss = b->opts.th_ss; s.th_hy = b->opts.th_hy; s.th_ac = b->opts.th_ac;
  s.min_w = b->opts.min_w; s.max_w = b->opts.max_w;
  CU(cudaMemsetAsync(d_counts, 0, b->n_pairs * sizeof(rp_sparse_counts), ctx->stream));
  CU(rp::launch_sparse(s, b->n_pairs, d_ups != nullptr, ctx->stream));
  ctx->timing.kernel_launches += d_ups ? 2 : 1;
  return RP_OK;
}

// Work that reads the batch's outputs on the context's current stream: that stream waits (on the device) for the stream
// the batch last ran on, and becomes the one rp_batch_destroy waits for before the buffers go back to the pool.
int order_after_run(rp_batch* b) {
  rp_ctx* ctx = b->ctx;
  if (b->last_stream && b->last_stream != ctx->stream) {
    CU(cudaEventRecord(ctx->ev_handoff, b->last_stream));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_handoff, 0));
  }
  b->last_stream = ctx->stream;
  return RP_OK;
}
}  // namespace

extern "C" int rp_batch_dense_device(rp_batch* b, void* out_dev, size_t out_floats) {
  if (!b || !out_dev) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  const rp::BatchPlan& p = b->plan;
  if (out_floats < p.total_floats) return fail(ctx, RP_ERR_CAPACITY, "rp_batch_dense_device: buffer too small");
  CU(cudaSetDevice(ctx->device));
  if (b->n_pairs == 0) return RP_OK;
  int rc = order_after_run(b);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out_dev, b->d_dense, p.total_floats * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
  return RP_OK;
}

extern "C" int rp_batch_samples_device(rp_batch* b, void* out_dev, size_t n) {
  if (!b || !out_dev) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  const rp::BatchPlan& p = b->plan;
  if (n < p.sample_total) return fail(ctx, RP_ERR_CAPACITY, "rp_batch_samples_device: buffer too small");
  CU(cudaSetDevice(ctx->device));
  if (!p.sample_total) return RP_OK;
  int rc = order_after_run(b);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out_dev, b->d_samples, p.sample_total * sizeof(int16_t), cudaMemcpyDeviceToDevice, ctx->stream));
  return RP_OK;
}

extern "C" int rp_batch_fetch_samples(rp_batch* b, int16_t* out, size_t n) {
  if (!b || !out) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  const rp::BatchPlan& p = b->plan;
  if (n < p.sample_total) return fail(ctx, RP_ERR_CAPACITY, "rp_batch_fetch_samples: buffer too small");
  CU(cudaSetDevice(ctx->device));
  if (!p.sample_total) return RP_OK;
  int rc = order_after_run(b);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out, b->d_samples, p.sample_total * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RP_OK;
}

extern "C" int rp_batch_square_device(rp_batch* b, float* bp1, float* bp2, float* up1, float* up2, float* hp) {
  if (!b) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  const rp::BatchPlan& p = b->plan;
  CU(cudaSetDevice(ctx->device));
  if (b->n_pairs == 0 || !(bp1 || bp2 || up1 || up2 || hp)) return RP_OK;
  rp::SquareDev s;
  s.probs = b->d_probs; s.dense = b->d_dense;
  s.out[rp::SQ_BP1] = bp1; s.out[rp::SQ_BP2] = bp2; s.out[rp::SQ_UP1] = up1; s.out[rp::SQ_UP2] = up2; s.out[rp::SQ_HP] = hp;
  s.N1 = s.N2 = 0;
  for (int k = 0; k < b->n_pairs; k++) {   // the dimensions rp_square_plan gives the batch's pairs
    s.N1 = std::max(s.N1, p.probs[3 * k].n1);
    s.N2 = std::max(s.N2, p.probs[3 * k].n2);
  }
  s.W = std::max(b->opts.max_w, 0);
  s.tiles = (std::max(s.N1, s.N2) + 1 + 31) / 32;
  if ((long long)b->n_pairs * s.tiles > 0x7fffffffLL)
    return fail(ctx, RP_ERR_ARG, "rp_batch_square_device: batch too large for one launch");
  int rc = order_after_run(b);
  if (rc) return rc;
  CU(rp::launch_square(s, b->n_pairs, ctx->stream));
  return RP_OK;
}

extern "C" int rp_batch_sparse_device(rp_batch* b, void* recs_dev, size_t n_recs, void* ups_dev, size_t n_floats,
                                      void* counts_dev) {
  if (!b || !recs_dev || !counts_dev) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  if (n_recs < b->total_recs || (ups_dev && n_floats < b->total_upf))
    return fail(ctx, RP_ERR_CAPACITY, "rp_batch_sparse_device: buffer too small");
  CU(cudaSetDevice(ctx->device));
  if (b->n_pairs == 0) return RP_OK;
  int rc = sparse_prepare(b);
  if (rc) return rc;
  return sparse_launch(b, static_cast<rp_rec*>(recs_dev), static_cast<float*>(ups_dev),
                       static_cast<rp_sparse_counts*>(counts_dev));
}

extern "C" int rp_batch_fetch_sparse(rp_batch* b, rp_rec* recs, size_t n_recs, float* ups, size_t n_floats,
                                     rp_sparse_counts* counts) {
  if (!b || !recs || !counts) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  if (n_recs < b->total_recs || (ups && n_floats < b->total_upf))
    return fail(ctx, RP_ERR_CAPACITY, "rp_batch_fetch_sparse: buffer too small");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int np = b->n_pairs;
  if (np == 0) return RP_OK;
  int rc = sparse_prepare(b);
  if (rc) return rc;
  if (!b->d_recs) {
    CU(pool_alloc(ctx, &b->d_recs, std::max<size_t>(1, b->total_recs) * sizeof(rp_rec)));
    CU(pool_alloc(ctx, &b->d_ups, std::max<size_t>(1, b->total_upf) * sizeof(float)));
    CU(pool_alloc(ctx, &b->d_counts, np * sizeof(rp_sparse_counts)));
  }
  rc = sparse_launch(b, b->d_recs, ups ? b->d_ups : nullptr, b->d_counts);
  if (rc) return rc;
  CU(cudaEventRecord(ctx->ev[2], st));
  if (b->total_recs) CU(cudaMemcpyAsync(recs, b->d_recs, b->total_recs * sizeof(rp_rec), cudaMemcpyDeviceToHost, st));
  if (ups && b->total_upf) CU(cudaMemcpyAsync(ups, b->d_ups, b->total_upf * sizeof(float), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(counts, b->d_counts, np * sizeof(rp_sparse_counts), cudaMemcpyDeviceToHost, st));
  CU(cudaEventRecord(ctx->ev[3], st));
  CU(cudaStreamSynchronize(st));
  ctx->timed_copies = true;
  for (int p = 0; p < np; p++)
    if (counts[p].overflow) return fail(ctx, RP_ERR_CAPACITY, "rp_batch_fetch_sparse: record capacity exceeded");
  return RP_OK;
}

extern "C" {

int rp_batch_fetch_logz(rp_batch* b, double* logz, size_t n) {
  if (!b || !logz) return RP_ERR_ARG;
  rp_ctx* ctx = b->ctx;
  if (n < (size_t)b->n_pairs * 3) return fail(ctx, RP_ERR_CAPACITY, "rp_batch_fetch_logz: buffer too small");
  CU(cudaSetDevice(ctx->device));
  if (b->n_pairs)
    CU(cudaMemcpyAsync(logz, b->d_logz, (size_t)b->n_pairs * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RP_OK;
}

int rp_last_timing(const rp_ctx* cctx, rp_timing* t) {
  if (!cctx || !t) return RP_ERR_ARG;
  rp_ctx* ctx = const_cast<rp_ctx*>(cctx);
  if (ctx->timing_pending) {
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
    ctx->timing.ms_total = ms;
    if (ctx->dom_timed) {
      CU(cudaEventElapsedTime(&ms, ctx->ev_dom[0], ctx->ev_dom[1]));
      ctx->timing.ms_dominant = ms;
    }
    if (ctx->timed_copies) {
      CU(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]));
      ctx->timing.ms_d2h = ms;
    }
    ctx->timing_pending = false;
  }
  *t = ctx->timing;
  return RP_OK;
}

// ------------------------------------------------------- one-shot host calls
int rp_run_mfe(rp_ctx* ctx, const rp_pair* pairs, const rp_constraint* cons, const rp_stack_energy* se,
               const rp_unpaired_energy* ue, int n_pairs, int problems, int16_t* structures, size_t n_structures,
               int32_t* energies) {
  if (!ctx || (n_pairs > 0 && !energies)) return fail(ctx, RP_ERR_ARG, "rp_run_mfe: null argument");
  std::string msg;
  const std::string who = "rp_run_mfe: ";
  int rc = rp::check_mfe(pairs, n_pairs, cons, se, ue, problems, &msg);
  if (rc != RP_OK) return fail(ctx, rc, who + msg);
  rp::MfePlan m;
  if ((rc = rp::plan_mfe(pairs, n_pairs, cons, se, ue, problems, device_facts(ctx), &m, &msg)) != RP_OK)
    return fail(ctx, rc, who + (msg.empty() ? std::string("sizes overflow the structure buffer") : msg));
  if (n_structures < m.total || (m.total && !structures))
    return fail(ctx, RP_ERR_CAPACITY, "rp_run_mfe: the structure buffer holds fewer int16 than rp_sample_plan (num = 1) asks");
  for (int k = 0; k < 3 * n_pairs; k++) energies[k] = RP_INF;
  if (m.jobs.empty()) return RP_OK;
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  if ((rc = ensure_workspace(ctx, (size_t)m.grid * m.slot_ints * sizeof(int32_t))) != RP_OK) return rc;
  if (ctx->ws_stream && ctx->ws_stream != st) CU(cudaStreamSynchronize(ctx->ws_stream));   // its last user is done
  ctx->ws_stream = st;
  // device buffers from the pool, released at the end of the call
  std::vector<void*> bufs;
  auto release = [&]() { for (void* p : bufs) pool_release(ctx, p); };
  auto up = [&](const void* src, size_t bytes, void** dst) -> cudaError_t {
    *dst = nullptr;
    if (!bytes) return cudaSuccess;
    cudaError_t e = pool_alloc(ctx, dst, bytes);
    if (e != cudaSuccess) return e;
    bufs.push_back(*dst);
    return src ? cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, st) : cudaSuccess;
  };
  rp::MfeDev d = {};
  std::vector<int32_t> e_init((size_t)3 * n_pairs, RP_INF);
  const int zero = 0;
  void *d_seq, *d_key, *d_es, *d_eu, *d_jobs, *d_counter, *d_struct, *d_energy;
  cudaError_t e = cudaSuccess;
  if (e == cudaSuccess) e = up(m.seq.data(), m.seq.size(), &d_seq);
  if (e == cudaSuccess) e = up(m.key.data(), m.key.size() * sizeof(uint16_t), &d_key);
  if (e == cudaSuccess) e = up(m.es.data(), m.es.size() * sizeof(int32_t), &d_es);
  if (e == cudaSuccess) e = up(m.eu.data(), m.eu.size() * sizeof(int32_t), &d_eu);
  if (e == cudaSuccess) e = up(m.jobs.data(), m.jobs.size() * sizeof(rp::MfeJob), &d_jobs);
  if (e == cudaSuccess) e = up(&zero, sizeof(int), &d_counter);
  if (e == cudaSuccess) e = up(nullptr, std::max<size_t>(m.total, 1) * sizeof(int16_t), &d_struct);
  if (e == cudaSuccess) e = up(e_init.data(), e_init.size() * sizeof(int32_t), &d_energy);
  if (e == cudaSuccess) {
    d.model = ctx->d_model;
    d.seq = static_cast<const uint8_t*>(d_seq);
    d.key = static_cast<const uint16_t*>(d_key);
    d.es = static_cast<const int32_t*>(d_es);
    d.eu = static_cast<const int32_t*>(d_eu);
    d.jobs = static_cast<const rp::MfeJob*>(d_jobs);
    d.njobs = (int)m.jobs.size();
    d.counter = static_cast<int*>(d_counter);
    d.ws = reinterpret_cast<int32_t*>(ctx->ws);
    d.slot_ints = m.slot_ints;
    d.structures = static_cast<int16_t*>(d_struct);
    d.energies = static_cast<int32_t*>(d_energy);
    ctx->timing = rp_timing{};
    cudaEventRecord(ctx->ev[0], st);
    e = rp::launch_mfe(d, m.grid, st);
    cudaEventRecord(ctx->ev[1], st);
  }
  if (e == cudaSuccess && m.total) e = cudaMemcpyAsync(structures, d_struct, m.total * sizeof(int16_t), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(energies, d_energy, e_init.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    cudaStreamSynchronize(st);
    release();
    return fail(ctx, RP_ERR_CUDA, std::string("rp_run_mfe: ") + cudaGetErrorString(e));
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]);
  ctx->timing.ms_total = ms;
  ctx->timing.kernel_launches = 1;
  ctx->timing.dominant_kind = -1;
  ctx->timing_pending = false;
  ctx->dom_timed = false;
  ctx->timed_copies = false;
  release();
  return RP_OK;
}

int rp_run_dense(rp_ctx* ctx, const rp_pair* pairs, int n_pairs, const rp_opts* opts, float* out, size_t out_floats) {
  if (!ctx || !out) return fail(ctx, RP_ERR_ARG, "rp_run_dense: null argument");
  rp_batch* b = nullptr;
  int rc = rp_batch_create(ctx, pairs, n_pairs, opts, &b);
  if (rc) return rc;
  if (out_floats < b->plan.total_floats) {
    rp_batch_destroy(b);
    return fail(ctx, RP_ERR_CAPACITY, "rp_run_dense: buffer too small");
  }
  rc = rp_batch_run(b);
  if (!rc) rc = rp_batch_fetch_dense(b, out, out_floats);
  rp_timing t;
  if (!rc) rp_last_timing(ctx, &t);
  rp_batch_destroy(b);
  return rc;
}

int rp_run_sparse(rp_ctx* ctx, const rp_pair* pairs, int n_pairs, const rp_opts* opts, rp_rec* recs, size_t n_recs,
                  float* ups, size_t n_floats, rp_sparse_counts* counts) {
  if (!ctx || !recs || !counts) return fail(ctx, RP_ERR_ARG, "rp_run_sparse: null argument");
  rp_batch* b = nullptr;
  int rc = rp_batch_create(ctx, pairs, n_pairs, opts, &b);
  if (rc) return rc;
  rc = rp_batch_run(b);
  if (!rc) rc = rp_batch_fetch_sparse(b, recs, n_recs, ups, n_floats, counts);
  rp_timing t;
  if (!rc) rp_last_timing(ctx, &t);
  rp_batch_destroy(b);
  return rc;
}

// ------------------------------------------------------------------- peaks
int rp_measure_peaks(rp_ctx* ctx, double* fp64_tflops, double* smem_gbs) {
  if (!ctx) return RP_ERR_ARG;
  CU(cudaSetDevice(ctx->device));
  const int grid = ctx->sm_count * 8, threads = 256;
  double* d_out = nullptr;
  CU(cudaMalloc(&d_out, (size_t)grid * threads * sizeof(double)));
  cudaStream_t st = ctx->stream;
  float best_f = 1e30f, best_s = 1e30f;
  const int it_f = 1 << 15, it_s = 1 << 12;
  for (int rep = 0; rep < 4; rep++) {
    CU(cudaEventRecord(ctx->ev[4], st));
    CU(rp::launch_peak_fp64(d_out, grid, it_f, st));
    CU(cudaEventRecord(ctx->ev[5], st));
    CU(cudaStreamSynchronize(st));
    float ms;
    CU(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
    if (rep > 0) best_f = std::min(best_f, ms);
    CU(cudaEventRecord(ctx->ev[4], st));
    CU(rp::launch_peak_smem(d_out, grid, it_s, st));
    CU(cudaEventRecord(ctx->ev[5], st));
    CU(cudaStreamSynchronize(st));
    CU(cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]));
    if (rep > 0) best_s = std::min(best_s, ms);
  }
  CU(cudaFree(d_out));
  if (fp64_tflops) *fp64_tflops = 2.0 * 8 * (double)it_f * grid * threads / (best_f * 1e-3) / 1e12;
  if (smem_gbs) *smem_gbs = 8.0 * 16 * (double)it_s * grid * threads / (best_s * 1e-3) / 1e9;
  return RP_OK;
}

}  // extern "C"
