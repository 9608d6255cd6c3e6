// The keyed permutations pi_p of [0, n) that K15 (pg_enrich.cu) and K17 (pg_autocorr.cu) share; the definition is
// stated in include/pathgraph.h (K15) and restated by oracle/enrichment.py. One copy, so both kernels draw the same
// pi_p for the same seed bit for bit.
#pragma once
#include <stdint.h>

constexpr int PG_PERM_ROUNDS = 8;

// least h >= 1 with 4^h >= n: pi_p works on 2h-bit values and cycle-walks back into [0, n)
static inline int pg_perm_half_bits(int64_t n) {
  int hbits = 1;
  while (((int64_t)1 << (2 * hbits)) < n) ++hbits;
  return hbits;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// round keys k_{p,r} = splitmix64(seed ^ (64 p + r))
__device__ __forceinline__ void pg_perm_keys(uint64_t seed, uint64_t p, uint64_t (&k)[PG_PERM_ROUNDS]) {
#pragma unroll
  for (int r = 0; r < PG_PERM_ROUNDS; ++r) k[r] = splitmix64(seed ^ (64ull * p + (uint64_t)r));
}

// Calls emit(i, pi_p(i)) for i = i0, i0 + stride, ... < n. One Feistel evaluation per iteration; a lane moves to its
// next node as soon as its cycle walk lands inside [0, n), so a lane whose walk is long does not hold the other 31
// lanes back.
template <class Emit>
__device__ __forceinline__ void pg_perm_walk(int64_t i, int64_t stride, int n, int hbits,
                                             const uint64_t (&k)[PG_PERM_ROUNDS], Emit emit) {
  const uint32_t mask = (1u << hbits) - 1u;
  uint32_t x = (uint32_t)i;
  while (i < n) {
    uint32_t L = x >> hbits, R = x & mask;
#pragma unroll
    for (int r = 0; r < PG_PERM_ROUNDS; ++r) {
      const uint32_t f = (uint32_t)splitmix64((uint64_t)R ^ k[r]) & mask;
      const uint32_t nr = L ^ f;
      L = R;
      R = nr;
    }
    x = (L << hbits) | R;
    if (x < (uint32_t)n) {
      emit(i, x);
      i += stride;
      x = (uint32_t)i;
    }
  }
}
#endif
