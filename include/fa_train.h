/*
 * fa_train.h -- the seeded batch order of K9 (csrc/fa_train.cu), shared by the kernel and anything that restates it.
 *
 * Epoch e of a job with seed s visits its row list in the order row_idx[fa_perm(i, n, s, e)], i = 0 .. n - 1.
 * fa_perm is a bijection of [0, n): a 4-round balanced Feistel network on 2h bits (2^(2h) >= n, h >= 1), keyed by
 * (seed, epoch), with cycle-walking (re-encrypt until the value falls inside [0, n)).  O(1) expected work per position,
 * no sort and no table, so every thread of a CTA can compute the rows of its batch on its own.  DESIGN.md "K9".
 * Pure C99 (host) and CUDA (device).
 */
#ifndef FA_TRAIN_H_
#define FA_TRAIN_H_

#include <stdint.h>

#if defined(__CUDACC__)
#define FA_TRAIN_FN static inline __host__ __device__
#else
#define FA_TRAIN_FN static inline
#endif

#define FA_PERM_ROUNDS 4

/* splitmix64 finaliser */
FA_TRAIN_FN uint64_t fa_perm_mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

/* round key r (0 .. FA_PERM_ROUNDS - 1) of (seed, epoch) */
FA_TRAIN_FN uint32_t fa_perm_key(uint64_t seed, uint32_t epoch, int r) {
  return (uint32_t)fa_perm_mix64(fa_perm_mix64(seed) ^ ((uint64_t)epoch << 8) ^ (uint64_t)r);
}

/* bits of one Feistel half: the smallest h >= 1 with 4^h >= n */
FA_TRAIN_FN int fa_perm_half_bits(uint32_t n) {
  int h = 1;
  while (h < 16 && ((uint64_t)1 << (2 * h)) < (uint64_t)n) h++;
  return h;
}

/* round function: a 32-bit integer hash of (half, key) */
FA_TRAIN_FN uint32_t fa_perm_round(uint32_t x, uint32_t key) {
  x ^= key;
  x ^= x >> 16; x *= 0x7FEB352Du;
  x ^= x >> 15; x *= 0x846CA68Bu;
  x ^= x >> 16;
  return x;
}

/* position i (< n) of the epoch's order -> index into the job's row list */
FA_TRAIN_FN uint32_t fa_perm(uint32_t i, uint32_t n, uint64_t seed, uint32_t epoch) {
  const int h = fa_perm_half_bits(n);
  const uint32_t mask = (1u << h) - 1u;
  uint32_t k[FA_PERM_ROUNDS];
  for (int r = 0; r < FA_PERM_ROUNDS; r++) k[r] = fa_perm_key(seed, epoch, r);
  uint32_t x = i;
  do {
    uint32_t L = x >> h, R = x & mask;
    for (int r = 0; r < FA_PERM_ROUNDS; r++) {
      const uint32_t t = L ^ (fa_perm_round(R, k[r]) & mask);
      L = R;
      R = t;
    }
    x = (L << h) | R;
  } while (x >= n);
  return x;
}

#endif /* FA_TRAIN_H_ */
