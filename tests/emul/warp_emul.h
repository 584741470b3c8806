// warp_emul.h -- TEST INFRASTRUCTURE.  A warp-lockstep executor for the host emulation (emul.cpp): it runs the
// 32 threads of each warp as cooperative fibers, so that the kernels' warp-shuffle forms of the split
// sums (mcc_band_shfl.cuh, mcc_wide_shfl.cuh) run on the host as they do on the device.  Never part of the product.
//
// A lane that calls a shuffle deposits its value and yields; once all 32 lanes of the warp wait at a shuffle, each
// resumes with the device's result (down: the value of lane+delta, its own if lane+delta >= 32; idx: the value of
// lane src % 32).  Warps of a phase run one after another, and a phase is a barrier, as in SerialExecT.
//
// A warp that does not meet in lockstep is a device hazard, reported as a nonzero error() instead of being smoothed
// over (the waiting lanes then resume with their own values, so the problem still runs to its end):
//   kErrExited    some lane of the warp returned while the others wait at a full-mask shuffle.  A lane that runs
//                 more shuffles than its neighbours ends up here too, at the end of the phase.
//   kErrMismatch  the lanes of a rendezvous are at different shuffles (kind, delta or source lane differ)
//   kErrThreads   the thread count is not a multiple of 32 (no phase runs)
//   kErrMask      a shuffle with a mask other than the full warp (the kernels use none)
#ifndef RP_WARP_EMUL_H
#define RP_WARP_EMUL_H

#include <setjmp.h>
#include <ucontext.h>

#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <memory>

// host stand-ins for the CUDA qualifiers and intrinsics the shuffle forms use (before mcc_driver.h)
#define RP_HOST_SHFL 1
#define __device__
#define __forceinline__ inline

namespace wemu {

enum { kErrExited = 101, kErrMismatch = 102, kErrThreads = 103, kErrMask = 104 };
enum { kDown = 0, kIdx = 1 };

// The 32 lane fibers of this host thread.  Each is created once (makecontext) and then loops: run the phase body for
// its lane, report done, wait for the next warp.  Switches between a lane and the scheduler use _setjmp/_longjmp,
// which unlike swapcontext leave the signal mask alone (no system call: a shuffle costs 64 switches).  The Makefile
// builds without _FORTIFY_SOURCE, whose longjmp check rejects a jump to another stack.
struct Warp {
  static constexpr size_t kStack = 512 * 1024;
  struct Lane {
    ucontext_t ctx;   // the fiber's entry, used once
    jmp_buf jb;       // where the lane waits
    std::unique_ptr<char[]> stack;
    bool started = false, waiting = false, done = false;
    int kind = 0, arg = 0;
    unsigned mask = 0;
    uint64_t val = 0, res = 0;
  };
  jmp_buf sched;   // where the scheduler waits
  Lane lane[32];
  void (*call)(void*, int) = nullptr;   // the phase body and its closure
  void* fn = nullptr;
  int base = 0;   // thread index of lane 0
  int cur = 0;    // the lane that runs
  int err = 0;
};

// the warp whose lanes run on this host thread
inline thread_local Warp* g_warp = nullptr;

inline Warp& thread_warp() {
  static thread_local Warp w;
  return w;
}

// lane -> scheduler, back when the scheduler resumes the lane
inline void yield_to_scheduler(Warp::Lane& L) {
  if (!_setjmp(L.jb)) _longjmp(g_warp->sched, 1);
}

inline void lane_main(int l) {
  for (;;) {
    Warp* w = g_warp;
    w->call(w->fn, w->base + l);
    w->lane[l].done = true;
    yield_to_scheduler(w->lane[l]);
  }
}

// scheduler -> lane l, back when it shuffles or returns
__attribute__((noinline)) inline void resume(Warp& w, int l) {
  Warp::Lane& L = w.lane[l];
  w.cur = l;
  L.waiting = false;
  if (_setjmp(w.sched)) return;
  if (L.started) _longjmp(L.jb, 1);
  L.started = true;
  if (!L.stack) L.stack.reset(new char[Warp::kStack]);
  getcontext(&L.ctx);
  L.ctx.uc_stack.ss_sp = L.stack.get();
  L.ctx.uc_stack.ss_size = Warp::kStack;
  L.ctx.uc_link = nullptr;   // lane_main never returns
  makecontext(&L.ctx, reinterpret_cast<void (*)()>(&lane_main), 1, l);
  setcontext(&L.ctx);
}

// lane side of a shuffle: deposit, yield to the scheduler, resume with the device's result
template <class T>
T shuffle(unsigned mask, T v, int kind, int arg) {
  static_assert(sizeof(T) <= sizeof(uint64_t), "32- or 64-bit shuffles only");
  Warp* w = g_warp;
  if (!w) std::abort();   // a shuffle outside the warp-lockstep executor
  Warp::Lane& L = w->lane[w->cur];
  L.val = 0;
  std::memcpy(&L.val, &v, sizeof v);
  L.kind = kind; L.arg = arg; L.mask = mask; L.waiting = true;
  yield_to_scheduler(L);
  T r;
  std::memcpy(&r, &L.res, sizeof r);
  return r;
}

// runs body(tid) for tid = base .. base+31 in lockstep; returns the first hazard found, or 0
template <class F>
int run_warp(Warp& w, int base, F& body) {
  w.call = [](void* fn, int tid) { (*static_cast<F*>(fn))(tid); };
  w.fn = &body;
  w.base = base;
  w.err = 0;
  g_warp = &w;
  for (auto& L : w.lane) L.waiting = L.done = false;
  for (;;) {
    // every lane that is not done runs to its next shuffle or to its end
    for (int l = 0; l < 32; l++)
      if (!w.lane[l].done) resume(w, l);
    int nwait = 0, first = -1;
    for (int l = 0; l < 32; l++)
      if (w.lane[l].waiting) { nwait++; if (first < 0) first = l; }
    if (nwait == 0) break;   // all 32 returned
    const Warp::Lane& F0 = w.lane[first];
    if (!w.err && nwait < 32) w.err = kErrExited;
    for (int l = 0; l < 32; l++) {
      Warp::Lane& L = w.lane[l];
      if (!L.waiting) continue;
      if (!w.err && L.mask != 0xffffffffu) w.err = kErrMask;
      if (!w.err && (L.kind != F0.kind || L.arg != F0.arg)) w.err = kErrMismatch;
      const int src = L.kind == kDown ? (l + L.arg < 32 ? l + L.arg : l) : (L.arg & 31);
      L.res = w.lane[src].waiting ? w.lane[src].val : L.val;
    }
  }
  g_warp = nullptr;
  return w.err;
}

// The executor (contract at the top of mcc_driver.h) of G CTAs that share one problem, warp-lockstep within each CTA:
// kShfl, so the split sums run the shuffle forms.  kBatch and kWide as in kernels.cu's CtaExecT<G, NB, W>; like
// SerialExecT it runs every rank's work in turn with one copy of shared memory.
template <int G, int NB, int W>
struct WarpExecT {
  static constexpr int kCtas = G;
  static constexpr bool kShfl = true;
  static constexpr int kBatch = NB;
  static constexpr int kWide = W;
  int T;
  int err = 0;
  Warp* warp = &thread_warp();
  explicit WarpExecT(int nthr) : T(nthr) {
    if (T % 32) err = kErrThreads;
  }
  int nthreads() const { return T; }
  template <class F>
  void phase(int, F f) {
    if (err == kErrThreads) return;
    for (int w0 = 0; w0 < T; w0 += 32) {
      const int e = run_warp(*warp, w0, f);
      if (!err) err = e;
    }
  }
  int rank_begin() const { return 0; }
  int rank_end() const { return G; }
  void sync() {}
  int error() const { return err; }
};

}  // namespace wemu

template <class T>
inline T __shfl_down_sync(unsigned mask, T v, unsigned delta, int = 32) {
  return wemu::shuffle(mask, v, wemu::kDown, (int)delta);
}
template <class T>
inline T __shfl_sync(unsigned mask, T v, int src, int = 32) {
  return wemu::shuffle(mask, v, wemu::kIdx, src);
}
inline double __ldcs(const double* p) { return *p; }
inline long long clock64() { return 0; }
inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) {
  const unsigned long long o = *p;
  *p = o + v;
  return o;
}

#endif
