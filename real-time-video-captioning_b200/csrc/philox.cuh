// Counter-based Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the generator behind
// curand's Philox4_32_10).  Host + device, so the host can check it against the Random123 known-answer vectors.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define PHILOX_HD __host__ __device__ __forceinline__
#else
#define PHILOX_HD inline
#endif

struct Philox4 {
  uint32_t x[4];
};

PHILOX_HD void philox_mulhilo(uint32_t a, uint32_t b, uint32_t* hi, uint32_t* lo) {
  const uint64_t p = (uint64_t)a * (uint64_t)b;
  *hi = (uint32_t)(p >> 32);
  *lo = (uint32_t)p;
}

// 10 rounds over counter c0..c3 with key (k0, k1).
PHILOX_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(0xD2511F53u, c0, &hi0, &lo0);
    philox_mulhilo(0xCD9E8D57u, c2, &hi1, &lo1);
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
  }
  Philox4 r;
  r.x[0] = c0; r.x[1] = c1; r.x[2] = c2; r.x[3] = c3;
  return r;
}

// 24 random bits -> a uniform in the open interval (0, 1): ((x >> 8) + 0.5) * 2^-24, exact in double.  (Not in fp32: there
// (2^24 - 1) + 0.5 is a rounding tie that goes to 2^24, so 1 word in 2^24 would give u = 1 and an infinite race key.)
PHILOX_HD double philox_uniform(uint32_t x) { return ((double)(x >> 8) + 0.5) * 5.9604644775390625e-8; }

// The Gumbel term of the exponential race, -log(-log u), in double: finite for every u above (from -2.85 to 17.33).
PHILOX_HD float philox_gumbel(uint32_t x) { return (float)-log(-log(philox_uniform(x))); }

// Dropout mask of the student's distillation step (csrc/student_train.cu; restated in tests/student_dropout_ref.py).  Element
// idx of site `site` at dropout step `step` (mod 2^32) is kept iff philox_uniform(w) >= p in double, w = word idx % 4 of
// Philox4x32-10(counter (idx / 4, step, site, 0x44524F50 "DROP"), key = (seed low 32 bits, seed high 32 bits)); a kept element
// is scaled by 1 / (1 - p) in fp32 (inv_keep), a dropped one is 0.
constexpr uint32_t DROPOUT_TAG = 0x44524F50u;
PHILOX_HD Philox4 dropout_words(uint64_t seed, uint32_t step, uint32_t site, uint32_t idx) {
  return philox4x32_10(idx >> 2, step, site, DROPOUT_TAG, (uint32_t)seed, (uint32_t)(seed >> 32));
}
PHILOX_HD float dropout_keep(uint32_t word, float p, float inv_keep) { return philox_uniform(word) >= (double)p ? inv_keep : 0.f; }
// one element: 0 or inv_keep = 1 / (1 - p)
PHILOX_HD float dropout_scale(uint64_t seed, uint32_t step, uint32_t site, uint32_t idx, float p, float inv_keep) {
  return dropout_keep(dropout_words(seed, step, site, idx).x[idx & 3], p, inv_keep);
}
