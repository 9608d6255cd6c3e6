// K17: spatial autocorrelation - Moran's I or Geary's C of per-nucleus feature columns over a symmetric CSR, against
// the same statistic under random relabelling of the nodes (squidpy.gr.spatial_autocorr's permutation test;
// definition and statistics in include/pathgraph.h).
//
// Labellings are processed in chunks of rows: row 0 is the identity (the observed statistic, computed by the same
// kernel as the permutations), row p + 1 is permutation p. One permutation moves every column at once, so pi_p is
// evaluated once per node and labelling and kept as an int32 index; a chunk holds at most PG_AUTOCORR_CHUNK_BYTES of
// indices, so the indices and one 4-column group of centred values (32 n bytes) stay in L2 together at C2 size.
//   ac_prep_kernel<0/1>   (pg_autocorr.cuh) per group of 4 columns: the column sums -> mean; then z = x - mean written
//                         node-major (one node's group = one 32-byte sector) and m2 = sum z^2.
//   ac_degree_kernel      thread / row: d_i = in-range entries, integer sums of d_i, d_i^2 and non-isolated rows.
//   ac_weights_kernel     S0 / S1 / S2 (row-standardised: thread / row over 1 / d_j of its neighbours).
//   ac_index_kernel       idx[row][i] = pi_p(i) (pg_perm.cuh, K15's permutations bit for bit).
//   ac_row_kernel         grid (CTA, labelling, group): the warp-flattened row walk of the other CSR kernels - a warp
//                         owns 32 consecutive rows and its lanes take the rows' entries 32 at a time, so a 4 200-entry
//                         row of a dense clump does not serialise a lane - with the per-entry term w_i z_i z_j (Moran)
//                         or w_i (z_i - z_j)^2 (Geary) of all 4 columns, z read through the index; the last CTA of a
//                         (labelling, group) turns the sums into the statistic.
//   ac_finish_kernel      warp / column: stat, permutation mean, ddof-0 variance (second pass), n_ge, sims.
// Every float sum is taken in a fixed order (cta_sum_last); the grid sizes depend on n only, never on the device or the
// chunk, so the result is the same bit for bit on every run, chunking and handle. Only integer atomics.
#include <algorithm>
#include <cmath>
#include "pg_autocorr.cuh"
#include "pg_perm.cuh"

namespace {

constexpr int IDX_PER_THREAD = 16;  // nodes an index thread walks (amortises its 8 round keys)
constexpr int PART_MAX = 8192;      // labellings of a chunk x CTAs: bounds the partials of one row-pass launch

__global__ void __launch_bounds__(TPB)
ac_degree_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
                 int32_t* __restrict__ deg, ac_misc* misc) {
  const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  unsigned long long d = 0;
  if (i < n) {
    for (int p = row_ptr[i], e = row_ptr[i + 1]; p < e; ++p) d += (unsigned)col[p] < (unsigned)n;
    deg[i] = (int32_t)d;
  }
  unsigned long long sq = d * d, nz = d > 0;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    d += __shfl_xor_sync(0xffffffffu, d, s);
    sq += __shfl_xor_sync(0xffffffffu, sq, s);
    nz += __shfl_xor_sync(0xffffffffu, nz, s);
  }
  if ((threadIdx.x & 31) == 0 && d) {
    atomicAdd(&misc->deg_sum, d);
    atomicAdd(&misc->deg_sq, sq);
    atomicAdd(&misc->nonisolated, nz);
  }
}

// Binary weights (one CTA): S0, S1, S2 from the integer sums. Row-standardised: thread / row, S1 and S2 as fixed-order
// float64 sums.
template <bool ROWSTD>
__global__ void __launch_bounds__(TPB)
ac_weights_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
                  const int32_t* __restrict__ deg, ac_misc* misc, double* part, unsigned int* ticket) {
  double v[2] = {0.0, 0.0};  // sum over entries (1/d_i + 1/d_j)^2, sum over rows (1 + sum_j 1/d_j)^2
  if (ROWSTD) {
    for (int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x; i < n; i += (int64_t)gridDim.x * TPB) {
      const int di = deg[i];
      if (di == 0) continue;
      const double inv_i = 1.0 / (double)di;
      double a = 0.0, t1 = 0.0;
      for (int p = row_ptr[i], e = row_ptr[i + 1]; p < e; ++p) {
        const int j = col[p];
        if ((unsigned)j >= (unsigned)n) continue;
        const double inv_j = 1.0 / (double)deg[j];
        const double t = inv_i + inv_j;
        a += inv_j;
        t1 += t * t;
      }
      v[0] += t1;
      v[1] += (1.0 + a) * (1.0 + a);
    }
  }
  double tot[2];
  if (!cta_sum_last<2>(v, part, ticket, tot)) return;
  if (ROWSTD) {
    misc->s012[0] = (double)misc->nonisolated;
    misc->s012[1] = 0.5 * tot[0];
    misc->s012[2] = tot[1];
  } else {
    misc->s012[0] = (double)misc->deg_sum;
    misc->s012[1] = (double)(2ull * misc->deg_sum);
    misc->s012[2] = (double)(4ull * misc->deg_sq);
  }
}

// idx[blockIdx.y][i] = pi_p(i) for the labelling row0 + blockIdx.y (row 0: the identity)
__global__ void __launch_bounds__(TPB)
ac_index_kernel(int n, int hbits, uint64_t seed, int row0, int32_t* __restrict__ idx) {
  const int row = row0 + blockIdx.y;
  int32_t* out = idx + (size_t)blockIdx.y * (size_t)n;
  const int64_t stride = (int64_t)gridDim.x * TPB;
  const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (row == 0) {
    for (int64_t v = i; v < n; v += stride) out[v] = (int32_t)v;
    return;
  }
  uint64_t k[PG_PERM_ROUNDS];
  pg_perm_keys(seed, (uint64_t)(row - 1), k);
  pg_perm_walk(i, stride, n, hbits, k, [&](int64_t v, uint32_t x) {
    PG_ASSERT(x < (uint32_t)n);
    out[v] = (int32_t)x;
  });
}

// blockIdx.y = labelling row0 + y of the chunk, blockIdx.z = column group. sims[row][f] = the statistic.
template <bool GEARY, bool ROWSTD>
__global__ void __launch_bounds__(TPB)
ac_row_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
              const int32_t* __restrict__ deg, const int32_t* __restrict__ idx, const double4* __restrict__ zg,
              int n_feat, int row0, const ac_misc* misc, double* part, unsigned int* tickets,
              double* __restrict__ sims) {
  const int r = blockIdx.y, g = blockIdx.z, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int32_t* pi = idx + (size_t)r * (size_t)n;
  const double4* z = zg + (size_t)g * (size_t)n;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int64_t rb = ((int64_t)blockIdx.x * WARPS + warp) * 32; rb < n; rb += (int64_t)gridDim.x * WARPS * 32) {
    // rows and entry positions in 64 bits: r0 + 32 and p0 + 31 may pass INT32_MAX at the top of the int32 range
    const int64_t r0 = rb, own = r0 + lane;
    const int rp = row_ptr[min(own, (int64_t)n)];
    const int begin = __shfl_sync(0xffffffffu, rp, 0);
    const int end = row_ptr[min(r0 + 32, (int64_t)n)];
    // this lane's row: a = w_i z_i (Moran) or z_i (Geary), w = w_i
    double4 a = make_double4(0.0, 0.0, 0.0, 0.0);
    double w = 1.0;
    if (own < n) {
      a = z[pi[own]];
      if (ROWSTD) {
        const int d = deg[own];
        w = d > 0 ? 1.0 / (double)d : 0.0;
      }
      if (!GEARY && ROWSTD) { a.x *= w; a.y *= w; a.z *= w; a.w *= w; }
    }
    for (int64_t p0 = begin; p0 < end; p0 += 32) {
      const int64_t p = p0 + lane;
      int kk = 0;  // the last of the 32 rows whose range starts at or before p
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const int v = __shfl_sync(0xffffffffu, rp, kk + step);
        if (v <= p) kk += step;
      }
      const double a0 = __shfl_sync(0xffffffffu, a.x, kk), a1 = __shfl_sync(0xffffffffu, a.y, kk);
      const double a2 = __shfl_sync(0xffffffffu, a.z, kk), a3 = __shfl_sync(0xffffffffu, a.w, kk);
      const double wk = (GEARY && ROWSTD) ? __shfl_sync(0xffffffffu, w, kk) : 1.0;
      if (p >= end) continue;
      const int j = col[p];
      if ((unsigned)j >= (unsigned)n) continue;
      PG_ASSERT((unsigned)pi[j] < (unsigned)n);
      const double4 b = z[pi[j]];
      if (GEARY) {
        const double d0 = a0 - b.x, d1 = a1 - b.y, d2 = a2 - b.z, d3 = a3 - b.w;
        if (ROWSTD) {
          acc[0] += wk * (d0 * d0); acc[1] += wk * (d1 * d1); acc[2] += wk * (d2 * d2); acc[3] += wk * (d3 * d3);
        } else {
          acc[0] += d0 * d0; acc[1] += d1 * d1; acc[2] += d2 * d2; acc[3] += d3 * d3;
        }
      } else {
        acc[0] += a0 * b.x; acc[1] += a1 * b.y; acc[2] += a2 * b.z; acc[3] += a3 * b.w;
      }
    }
  }
  const int slot = r * gridDim.z + g;
  double tot[4];
  if (!cta_sum_last<4>(acc, part + (int64_t)slot * gridDim.x * 4, tickets + slot, tot)) return;
  const double s0 = misc->s012[0];
  for (int k = 0; k < 4; ++k) {
    const int f = 4 * g + k;
    if (f >= n_feat) break;
    const double m2 = misc->m2[f];
    double stat = nan_d();
    if (s0 != 0.0 && m2 != 0.0)
      stat = GEARY ? ((double)(n - 1) * tot[k]) / (2.0 * s0 * m2) : ((double)n * tot[k]) / (s0 * m2);
    sims[(int64_t)(row0 + r) * n_feat + f] = stat;
  }
}

// warp / column f: sims_ws [P + 1][n_feat] (row 0 observed) -> the outputs
__global__ void __launch_bounds__(TPB)
ac_finish_kernel(const double* __restrict__ sims_ws, int n_feat, int n_perms, const ac_misc* misc,
                 pg_autocorr_out o) {
  const int f = (blockIdx.x * TPB + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (f >= n_feat) return;  // warp-uniform
  const double stat = sims_ws[f];
  double s = 0.0;
  unsigned long long ge = 0;
  for (int p = lane; p < n_perms; p += 32) {
    const double v = sims_ws[(int64_t)(p + 1) * n_feat + f];
    s += v;
    ge += v >= stat;
    if (o.sims) o.sims[(int64_t)p * n_feat + f] = v;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, d);
    ge += __shfl_xor_sync(0xffffffffu, ge, d);
  }
  const double mean = s / (double)n_perms;  // n_perms = 0: NaN
  double q = 0.0;
  for (int p = lane; p < n_perms; p += 32) {
    const double dv = sims_ws[(int64_t)(p + 1) * n_feat + f] - mean;
    q += dv * dv;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) q += __shfl_xor_sync(0xffffffffu, q, d);
  if (lane != 0) return;
  if (o.stat) o.stat[f] = stat;
  if (o.perm_mean) o.perm_mean[f] = mean;
  if (o.perm_var) o.perm_var[f] = q / (double)n_perms;
  if (o.n_ge) o.n_ge[f] = (int64_t)ge;
  if (f == 0 && o.s012)
    for (int k = 0; k < 3; ++k) o.s012[k] = misc->s012[k];
}

}  // namespace

extern "C" {

int pg_spatial_autocorr(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t n_feat,
                        const double* feat, int32_t flags, int32_t n_perms, uint64_t seed, const pg_autocorr_out* out,
                        pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0, "pg_spatial_autocorr: negative n");
  PG_REQUIRE(h, n_feat >= 1 && n_feat <= PG_AUTOCORR_MAX_FEAT, "pg_spatial_autocorr: n_feat must be in 1..%d",
             PG_AUTOCORR_MAX_FEAT);
  PG_REQUIRE(h, n_perms >= 0 && n_perms <= PG_ENRICH_MAX_PERMS, "pg_spatial_autocorr: n_perms must be in 0..%d",
             PG_ENRICH_MAX_PERMS);
  PG_REQUIRE(h, (flags & ~(PG_AUTOCORR_GEARY | PG_AUTOCORR_ROW_STD)) == 0, "pg_spatial_autocorr: unknown flags %d",
             flags);
  PG_REQUIRE(h, row_ptr, "pg_spatial_autocorr: row_ptr is NULL");
  PG_REQUIRE(h, n == 0 || (col && feat), "pg_spatial_autocorr: col / feat is NULL");
  pg_autocorr_out o{};
  if (out) o = *out;
  const bool geary = flags & PG_AUTOCORR_GEARY, rowstd = flags & PG_AUTOCORR_ROW_STD;
  const int G = (n_feat + 3) / 4;
  const int64_t rows_total = (int64_t)n_perms + 1;
  const int gx = std::max(1, std::min(pg_div_up(n, TPB), GX_MAX));
  const int64_t chunk = std::min<int64_t>({rows_total, std::max<int64_t>(1, (int64_t)PG_AUTOCORR_CHUNK_BYTES / (4 * std::max(n, 1))),
                                           std::max(1, PART_MAX / gx)});
  const int n_tickets = (int)std::max<int64_t>(chunk * G, G);
  const size_t misc_bytes = sizeof(ac_misc) + 4 * (size_t)n_tickets;
  int rc;
  if ((rc = pg_reserve(h, h->ac_z, std::max<size_t>(32, (size_t)G * n * sizeof(double4))))) return rc;
  if ((rc = pg_reserve(h, h->ac_idx, std::max<size_t>(4, (size_t)chunk * n * 4)))) return rc;
  if ((rc = pg_reserve(h, h->ac_deg, std::max<size_t>(4, (size_t)n * 4)))) return rc;
  if ((rc = pg_reserve(h, h->ac_sims, (size_t)rows_total * n_feat * 8))) return rc;
  if ((rc = pg_reserve(h, h->ac_part, (size_t)chunk * G * gx * 4 * 8))) return rc;
  if ((rc = pg_reserve(h, h->ac_misc, misc_bytes))) return rc;
  ac_misc* misc = (ac_misc*)h->ac_misc.p;
  unsigned int* tickets = (unsigned int*)((char*)h->ac_misc.p + sizeof(ac_misc));
  double* part = (double*)h->ac_part.p;
  double4* zg = (double4*)h->ac_z.p;
  int32_t* deg = (int32_t*)h->ac_deg.p;
  int32_t* idx = (int32_t*)h->ac_idx.p;
  double* sims = (double*)h->ac_sims.p;
  PG_CUDA(h, cudaMemsetAsync(misc, 0, misc_bytes, s));

  PG_LAUNCH(h, s, "ac_prep_kernel<0>",
            ac_prep_kernel<0><<<dim3(gx, G), TPB, 0, s>>>(feat, n, n_feat, misc, zg, part, tickets));
  PG_LAUNCH(h, s, "ac_prep_kernel<1>",
            ac_prep_kernel<1><<<dim3(gx, G), TPB, 0, s>>>(feat, n, n_feat, misc, zg, part, tickets));
  PG_LAUNCH(h, s, "ac_degree_kernel",
            ac_degree_kernel<<<std::max(1, pg_div_up(n, TPB)), TPB, 0, s>>>(row_ptr, col, n, deg, misc));
  if (rowstd)
    PG_LAUNCH(h, s, "ac_weights_kernel<1>",
              ac_weights_kernel<true><<<gx, TPB, 0, s>>>(row_ptr, col, n, deg, misc, part, tickets));
  else
    PG_LAUNCH(h, s, "ac_weights_kernel<0>",
              ac_weights_kernel<false><<<1, TPB, 0, s>>>(row_ptr, col, n, deg, misc, part, tickets));

  const int hbits = pg_perm_half_bits(n);
  const int gx_idx = std::max(1, (int)std::min<int64_t>(pg_div_up(n, (int64_t)TPB * IDX_PER_THREAD), 1 << 20));
  auto row_kernel = geary ? (rowstd ? ac_row_kernel<true, true> : ac_row_kernel<true, false>)
                          : (rowstd ? ac_row_kernel<false, true> : ac_row_kernel<false, false>);
  for (int64_t r0 = 0; r0 < rows_total; r0 += chunk) {
    const int rows = (int)std::min(chunk, rows_total - r0);
    PG_LAUNCH(h, s, "ac_index_kernel",
              ac_index_kernel<<<dim3(gx_idx, rows), TPB, 0, s>>>(n, hbits, seed, (int)r0, idx));
    PG_ASSERT(r0 + rows <= rows_total && (int64_t)rows * G <= n_tickets);
    PG_LAUNCH(h, s, "ac_row_kernel",
              row_kernel<<<dim3(gx, rows, G), TPB, 0, s>>>(row_ptr, col, n, deg, idx, zg, n_feat, (int)r0, misc, part,
                                                          tickets, sims));
  }
  PG_LAUNCH(h, s, "ac_finish_kernel",
            ac_finish_kernel<<<pg_div_up((int64_t)n_feat * 32, TPB), TPB, 0, s>>>(sims, n_feat, n_perms, misc, o));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
