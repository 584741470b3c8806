/* philox.h -- Philox4x64-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011), the counter-based
 * generator of stochastic sampling.  Plain C as well as CUDA C++: the sampling phase of the general kernel
 * (mcc_sample.h), its host emulation and the CPU oracle sampler (tests/cpp/oracle_sample.c) all call these functions,
 * so that they draw the same numbers. */
#ifndef RP_PHILOX_H
#define RP_PHILOX_H

#include <stdint.h>

#ifndef RP_HD
#ifdef __CUDACC__
#define RP_HD __host__ __device__ __forceinline__
#elif defined(__cplusplus)
#define RP_HD inline
#else
#define RP_HD static inline
#endif
#endif

/* high 64 bits of a * b */
RP_HD uint64_t rp_mulhi64(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

/* out[0..3] = Philox4x64-10(counter ctr[0..3], key key[0..1]); word 0 is the least significant of a counter or key
 * written as one integer (numpy.random.Philox's convention) */
RP_HD void rp_philox4x64(const uint64_t ctr[4], const uint64_t key[2], uint64_t out[4]) {
  uint64_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
  for (int r = 0; r < 10; r++) {
    const uint64_t m0 = 0xD2E7470EE14C6C93ull, m1 = 0xCA5A826395121157ull;
    const uint64_t hi0 = rp_mulhi64(m0, c0), lo0 = m0 * c0, hi1 = rp_mulhi64(m1, c2), lo1 = m1 * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B97F4A7C15ull;
    k1 += 0xBB67AE8584CAA73Bull;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* the uniform in [0, 1) of a 64-bit draw: its top 53 bits */
RP_HD double rp_uniform53(uint64_t x) { return (double)(x >> 11) * (1.0 / 9007199254740992.0); }

/* The block of uniform numbers 4b .. 4b+3 (one per decision of a traceback, in traceback order) of sample `sample` of
 * problem `kind` (0 s1, 1 s2, 2 s1&s2) of pair `pair`: Philox at key (seed, 3 pair + kind), counter (sample, b, 0, 0);
 * uniform number t is word t % 4 of block t / 4, through rp_uniform53.  A traceback draws a block every fourth decision. */
RP_HD void rp_sample_block(uint64_t seed, int pair, int kind, int sample, int b, uint64_t out[4]) {
  const uint64_t key[2] = {seed, 3ull * (uint64_t)pair + (uint64_t)kind};
  const uint64_t ctr[4] = {(uint64_t)sample, (uint64_t)b, 0, 0};
  rp_philox4x64(ctr, key, out);
}

#endif
