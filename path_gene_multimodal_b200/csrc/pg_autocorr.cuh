// The prep pass K17 (pg_autocorr.cu) and K18 (pg_lisa.cu) share: column means, centred values in node-major groups of
// 4 columns (one node's group = one 32-byte sector) and m2 = sum z^2, each a fixed-order float64 sum (cta_sum_last).
// One copy, so both kernels centre a column bit for bit alike.
#pragma once
#include "pg_common.cuh"

namespace {

constexpr int TPB = 256;
constexpr int WARPS = TPB / 32;
constexpr int GX_MAX = 1184;        // CTAs of the grid-stride passes: a constant, not the SM count (fixes the sum order)

struct ac_misc {
  double mean[PG_AUTOCORR_MAX_FEAT];
  double m2[PG_AUTOCORR_MAX_FEAT];
  double s012[4];
  unsigned long long deg_sum, deg_sq, nonisolated, pad;
  // followed by the uint32 CTA tickets
};

__device__ __forceinline__ double nan_d() { return __longlong_as_double(0x7ff8000000000000ll); }

// Adds v[K] over the CTA - a thread's own share, a shuffle tree, the warps in index order - stores the CTA's sums in
// part[blockIdx.x][K] and takes a ticket. Returns true in thread 0 of the CTA that finishes last, with tot = the CTA
// partials added in index order (and the ticket re-armed for the next launch). Call once per kernel, from every thread.
template <int K>
__device__ __forceinline__ bool cta_sum_last(double (&v)[K], double* part, unsigned int* ticket, double (&tot)[K]) {
  __shared__ double s_w[WARPS][K];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], d);
    if (lane == 0) s_w[warp][k] = v[k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      double t = 0.0;
      for (int w = 0; w < WARPS; ++w) t += s_w[w][k];
      part[(int64_t)blockIdx.x * K + k] = t;
    }
    __threadfence();
    s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!s_last || threadIdx.x != 0) return false;
  __threadfence();
  const volatile double* p = part;
#pragma unroll
  for (int k = 0; k < K; ++k) tot[k] = 0.0;
  for (unsigned int g = 0; g < gridDim.x; ++g)
#pragma unroll
    for (int k = 0; k < K; ++k) tot[k] += p[(int64_t)g * K + k];
  *ticket = 0u;
  return true;
}

// blockIdx.y = group g of columns 4g..4g+3 (columns past n_feat read as 0). PASS 0: mean; PASS 1: z and m2.
template <int PASS>
__global__ void __launch_bounds__(TPB)
ac_prep_kernel(const double* __restrict__ feat, int n, int n_feat, ac_misc* misc, double4* __restrict__ zg,
               double* part, unsigned int* tickets) {
  const int g = blockIdx.y;
  double mean[4], v[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
  for (int k = 0; k < 4; ++k) mean[k] = (PASS == 1 && 4 * g + k < n_feat) ? misc->mean[4 * g + k] : 0.0;
  for (int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x; i < n; i += (int64_t)gridDim.x * TPB) {
    double z[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int f = 4 * g + k;
      const double x = f < n_feat ? feat[(int64_t)f * n + i] : 0.0;
      z[k] = f < n_feat ? x - mean[k] : 0.0;
      v[k] += PASS == 0 ? x : z[k] * z[k];
    }
    if (PASS == 1) zg[(int64_t)g * n + i] = make_double4(z[0], z[1], z[2], z[3]);
  }
  double tot[4];
  if (!cta_sum_last<4>(v, part + (int64_t)g * gridDim.x * 4, tickets + g, tot)) return;
  for (int k = 0; k < 4; ++k) {
    const int f = 4 * g + k;
    if (f >= n_feat) break;
    if (PASS == 0) misc->mean[f] = tot[k] / (double)n;  // n = 0: NaN
    else misc->m2[f] = tot[k];
  }
}

}  // namespace
