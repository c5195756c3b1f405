/*
 * fa_train.h -- the seeded batch order and the launch geometry of K9 (csrc/fa_train.cu), shared by the kernel and
 * anything that restates them.
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

#include "fa_b200.h"

#if defined(__CUDACC__)
#define FA_TRAIN_FN static inline __host__ __device__
#else
#define FA_TRAIN_FN static inline
#endif

#define FA_TRAIN_THREADS 512 /* threads of the CTA that trains one job */
#define FA_TRAIN_TILE 8      /* rows per thread in the forward and delta phases; the batch is padded to a multiple */

/* Where one fa_mlp_train launch keeps what.  Dynamic shared memory starts with red ([2][FA_TRAIN_THREADS] doubles, the
 * partial min / max of the range reduction) and rng ([2][dims[0]] doubles, the ranges).  Then comes the batch area when
 * it fits under the shared-memory cap; otherwise each job has a slice of area_bytes in global scratch.  The batch area
 * holds the per-row tables (loss: double[bpad]; row, label, hit: int[bpad] each) and, from act_off, the activations.
 * Offsets in floats (parameters, activations) or bytes (the rest); every size is 64-bit. */
typedef struct fa_train_geom {
  int64_t bpad;                               /* the batch size rounded up to FA_TRAIN_TILE rows */
  int64_t w_off[FA_MLP_MAX_LAYERS];           /* floats: kernel [dims[l]][dims[l + 1]] of layer l (K7's layout) */
  int64_t b_off[FA_MLP_MAX_LAYERS];           /* floats: its bias */
  int64_t n_params;                           /* floats of parameters per job */
  int64_t a_off[FA_MLP_MAX_LAYERS + 1];       /* floats: activations (then deltas) [bpad][dims[l]] of layer l */
  int64_t n_act;                              /* floats of activations per job */
  int64_t act_off;                            /* bytes from the start of the batch area to the activations */
  int64_t area_bytes;                         /* bytes of one job's batch area, a multiple of 16 */
  int64_t area_smem_off;                      /* bytes from the start of dynamic shared memory to the batch area */
  int area_in_smem;                           /* 1: the batch area is in shared memory; 0: per-job global scratch */
  int64_t smem_bytes;                         /* dynamic shared memory of the launch */
} fa_train_geom;

/* The geometry of n_layers layers (dims[0 .. n_layers]) at batch size `batch`: the batch area goes to shared memory when
 * the whole launch then needs at most smem_cap bytes.  Returns 0, or -1 when the launch cannot be served: more than
 * smem_optin bytes of shared memory (the block's opt-in limit minus the kernel's static shared memory), or a parameter or
 * activation count past the kernel's 32-bit indexing. */
FA_TRAIN_FN int fa_train_geometry(const int* dims, int n_layers, int batch, int64_t smem_cap, int64_t smem_optin,
                                  fa_train_geom* g) {
  int64_t off = 0, act = 0;
  g->bpad = ((int64_t)batch + FA_TRAIN_TILE - 1) / FA_TRAIN_TILE * FA_TRAIN_TILE;
  for (int l = 0; l <= FA_MLP_MAX_LAYERS; l++) g->a_off[l] = 0;   /* entries past n_layers stay 0 */
  for (int l = 0; l < FA_MLP_MAX_LAYERS; l++) g->w_off[l] = g->b_off[l] = 0;
  for (int l = 0; l <= n_layers; l++) {
    g->a_off[l] = act;
    act += g->bpad * dims[l];
  }
  for (int l = 0; l < n_layers; l++) {
    g->w_off[l] = off; off += (int64_t)dims[l] * dims[l + 1];
    g->b_off[l] = off; off += dims[l + 1];
  }
  g->n_params = off;
  g->n_act = act;
  g->act_off = g->bpad * (int64_t)(sizeof(double) + 3 * sizeof(int32_t));
  g->area_bytes = (g->act_off + act * (int64_t)sizeof(float) + 15) / 16 * 16;
  g->area_smem_off = (2 * FA_TRAIN_THREADS + 2 * (int64_t)dims[0]) * (int64_t)sizeof(double);
  g->area_in_smem = g->area_smem_off + g->area_bytes <= smem_cap;
  g->smem_bytes = g->area_smem_off + (g->area_in_smem ? g->area_bytes : 0);
  return g->smem_bytes <= smem_optin && g->n_params <= INT32_MAX && g->n_act <= INT32_MAX ? 0 : -1;
}

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
