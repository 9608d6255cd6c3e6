// K18: local indicators of spatial association - local Moran's I_i or Getis-Ord Gi / Gi* of every node and feature
// column over a symmetric CSR, against conditional permutations (esda's Moran_Local / G_Local crand; definitions in
// include/pathgraph.h).
//
// esda draws ONE index set per permutation and shares it across the nodes, so in permutation p every node reads the same
// <= 2K values z[r_p[j]], z[r_p[j] + 1] (node i takes the second when r_p[j] >= i, to skip itself). A CTA stages those
// values in shared memory once and its lanes read them as broadcasts: the hot loop is select + add on data already on
// chip, with no random DRAM traffic per node.
//   ac_prep_kernel<0/1>   (pg_autocorr.cuh) K17's centring: mean, z node-major in groups of 4 columns, m2.
//   lk_degree_kernel      thread / row: d_i = entries in [0, n) other than i; nodes per degree (CTA histogram of the
//                         small degrees in shared memory, one global add per CTA and degree).
//   pg_scan_i32           offsets of the degrees (clears the counts, which become the scatter cursor).
//   lk_order_kernel       counting-sort scatter: ord = the nodes in ascending degree, so a warp's lanes, and a CTA's
//                         tile, share their loop bounds. The order inside a degree is not fixed and does not matter:
//                         every node's arithmetic is its own.
//   lk_node_kernel        grid (tile of TPB nodes in degree order, column group): thread / node.
//                         1. S_i over its CSR row in entry order -> lag, stat_i (lk_coef / lk_stat).
//                         2. Permutations in steps: the CTA evaluates the draws r_p[j] (pg_perm.cuh, on [0, n - 1)) for
//                            up to PSTEP permutations x the tile's largest degree, and stages them with z[r], z[r + 1]
//                            (SLOTS slots); each lane selects by r >= i, adds in ascending j, forms stat_ip through
//                            lk_stat and updates its delta / delta^2 / n_ge accumulators in ascending p. Rows longer
//                            than SLOTS (a dense clump, up to d = n - 1) take one permutation per step and walk j in
//                            tiles of SLOTS with the sum carried in registers.
//                         3. perm_mean / perm_var / n_ge from the carried sums.
// A node's sums are sequential in one thread, so the outputs do not depend on the tiling, the order inside a degree, the
// run or the handle, and need no cross-thread reduction. The draws are recomputed per CTA and column group instead of
// being staged in global memory: the host never learns K (that would cost a synchronisation), and a draw (an 8-round
// Feistel evaluation) costs less than the tile's 4 x TPB adds that consume it.
#include <algorithm>
#include <cmath>
#include "pg_autocorr.cuh"
#include "pg_perm.cuh"

namespace {

constexpr int SLOTS = 512;   // (permutation, draw) slots of one step: int32 id + z[r], z[r + 1] (68 B each)
constexpr int PSTEP = 32;    // permutations of one step at most (their round keys are staged too)
constexpr int SMALL_DEG = 256;  // degrees counted / scattered through a CTA's shared-memory histogram

enum { LK_MORAN = 0, LK_GI = 1, LK_GI_STAR = 2 };

// stat = a S + b for node i's column: the one arithmetic path from a neighbour sum S (observed or permuted) to the
// statistic. a and b depend on i only: Moran a = c z_i w; Gi* a = w / D, b = w_ii z_i / D; Gi a = w / D,
// b = W_i z_i / ((n - 1) D), D the denominator of include/pathgraph.h.
__device__ __forceinline__ double lk_stat(double s, double a, double b) { return fma(s, a, b); }

template <int MODE>
__device__ __forceinline__ void lk_coef(int n, int d, bool rowstd, double zi, double m2, double& a, double& b) {
  const double nn = (double)n;
  a = nan_d();
  b = nan_d();
  if (MODE == LK_MORAN) {
    if (m2 != 0.0) {
      a = ((nn - 1.0) / m2) * zi * (rowstd ? (d > 0 ? 1.0 / (double)d : 0.0) : 1.0);
      b = 0.0;
    }
  } else if (MODE == LK_GI_STAR) {
    const double w = rowstd ? 1.0 / (double)(d + 1) : 1.0;
    const double W = rowstd ? 1.0 : (double)(d + 1), S1 = rowstd ? w : (double)(d + 1);
    const double q = (nn * S1 - W * W) / (nn - 1.0);
    if (n >= 2 && m2 > 0.0 && q > 0.0) {
      const double den = sqrt(m2 / nn) * sqrt(q);
      a = w / den;
      b = w * zi / den;
    }
  } else {
    if (n >= 3 && d > 0) {
      const double w = rowstd ? 1.0 / (double)d : 1.0;
      const double W = rowstd ? 1.0 : (double)d, S1 = rowstd ? w : (double)d;
      const double s2 = (m2 - zi * zi * nn / (nn - 1.0)) / (nn - 1.0);
      const double q = ((nn - 1.0) * S1 - W * W) / (nn - 2.0);
      if (s2 > 0.0 && q > 0.0) {
        const double den = sqrt(s2) * sqrt(q);
        a = w / den;
        b = W * zi / ((nn - 1.0) * den);
      }
    }
  }
}

__device__ __forceinline__ double4 d4_add(double4 s, double4 v) {
  return make_double4(s.x + v.x, s.y + v.y, s.z + v.z, s.w + v.w);
}
__device__ __forceinline__ double d4_get(const double4& v, int k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }

// thread / row: deg[i] = entries in [0, n) other than i; cnt[d] += 1
__global__ void __launch_bounds__(TPB)
lk_degree_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
                 int32_t* __restrict__ deg, int32_t* __restrict__ cnt) {
  __shared__ int s_cnt[SMALL_DEG];
  for (int t = threadIdx.x; t < SMALL_DEG; t += TPB) s_cnt[t] = 0;
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (i < n) {
    int d = 0;
    for (int p = row_ptr[i], e = row_ptr[i + 1]; p < e; ++p) {
      const int j = col[p];
      d += (unsigned)j < (unsigned)n && j != (int)i;
    }
    deg[i] = d;
    if (d < SMALL_DEG) atomicAdd(&s_cnt[d], 1);
    else atomicAdd(&cnt[d], 1);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < SMALL_DEG; t += TPB)
    if (s_cnt[t]) atomicAdd(&cnt[t], s_cnt[t]);
}

// ord[off[d_i] + rank] = i, rank taken from the cursor cur (zero on entry)
__global__ void __launch_bounds__(TPB)
lk_order_kernel(int n, const int32_t* __restrict__ deg, const int32_t* __restrict__ off, int32_t* __restrict__ cur,
                int32_t* __restrict__ ord) {
  __shared__ int s_cnt[SMALL_DEG];
  __shared__ int s_base[SMALL_DEG];
  for (int t = threadIdx.x; t < SMALL_DEG; t += TPB) s_cnt[t] = 0;
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  const int d = i < n ? deg[i] : -1;
  int rank = 0;
  if (d >= 0 && d < SMALL_DEG) rank = atomicAdd(&s_cnt[d], 1);
  else if (d >= SMALL_DEG) rank = atomicAdd(&cur[d], 1);
  __syncthreads();
  for (int t = threadIdx.x; t < SMALL_DEG; t += TPB)
    if (s_cnt[t]) s_base[t] = atomicAdd(&cur[t], s_cnt[t]);
  __syncthreads();
  if (d < 0) return;
  const int pos = off[d] + (d < SMALL_DEG ? s_base[d] : 0) + rank;
  PG_ASSERT(pos >= 0 && pos < n);
  ord[pos] = (int32_t)i;
}

// grid (tile, group g): thread / node ord[tile * TPB + t], columns 4g..4g+3
template <int MODE>
__global__ void __launch_bounds__(TPB, 2)
lk_node_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
               const int32_t* __restrict__ deg, const int32_t* __restrict__ ord, const double4* __restrict__ zg,
               int n_feat, bool rowstd, int n_perms, int hbits, uint64_t seed, const ac_misc* misc, pg_local_out o) {
  __shared__ int32_t s_r[SLOTS];
  __shared__ double4 s_v[SLOTS][2];
  __shared__ uint64_t s_key[PSTEP][PG_PERM_ROUNDS];
  const int g = blockIdx.y, nf = min(4, n_feat - 4 * g);
  const double4* z = zg + (size_t)g * (size_t)n;
  const int64_t t0 = (int64_t)blockIdx.x * TPB, slot = t0 + threadIdx.x;
  if (blockIdx.x == 0 && threadIdx.x < nf) {
    if (o.mean) o.mean[4 * g + threadIdx.x] = misc->mean[4 * g + threadIdx.x];
    if (o.m2) o.m2[4 * g + threadIdx.x] = misc->m2[4 * g + threadIdx.x];
  }
  const bool active = slot < n;
  const int i = active ? ord[slot] : 0;
  const int d = active ? deg[i] : 0;

  // observed: S_i in CSR entry order, then lag and stat through lk_stat
  double a[4], b[4], stat0[4];
  {
    double4 s = make_double4(0.0, 0.0, 0.0, 0.0);
    double4 zi = make_double4(0.0, 0.0, 0.0, 0.0);
    if (active) {
      zi = z[i];
      for (int p = row_ptr[i], e = row_ptr[i + 1]; p < e; ++p) {
        const int j = col[p];
        if ((unsigned)j >= (unsigned)n || j == i) continue;
        s = d4_add(s, z[j]);
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      lk_coef<MODE>(n, d, rowstd, d4_get(zi, k), k < nf ? misc->m2[4 * g + k] : 0.0, a[k], b[k]);
      const double sk = d4_get(s, k);
      stat0[k] = lk_stat(sk, a[k], b[k]);
      if (active && k < nf) {
        const size_t at = (size_t)(4 * g + k) * (size_t)n + (size_t)i;
        if (o.stat) o.stat[at] = stat0[k];
        if (o.lag) o.lag[at] = rowstd ? (d > 0 ? sk / (double)d : 0.0) : sk;
      }
    }
  }

  // permutations
  double s1[4] = {0.0, 0.0, 0.0, 0.0}, s2[4] = {0.0, 0.0, 0.0, 0.0};
  int ge[4] = {0, 0, 0, 0};
  double4 acc = make_double4(0.0, 0.0, 0.0, 0.0);
  const int dmax = t0 < n ? deg[ord[min(t0 + TPB, (int64_t)n) - 1]] : 0;  // the tile's largest degree (ord ascends)
  const int m = n - 1;                                          // draws come from [0, n - 1)
  if (dmax > 0 && n_perms > 0) {
    const int pc = min(PSTEP, max(1, SLOTS / dmax)), jt = min(dmax, SLOTS);
    for (int p0 = 0; p0 < n_perms; p0 += pc) {
      const int np = min(pc, n_perms - p0);
      __syncthreads();  // the previous step's readers are done with s_key / s_r / s_v
      for (int t = threadIdx.x; t < np; t += TPB) {
        uint64_t k[PG_PERM_ROUNDS];
        pg_perm_keys(seed, (uint64_t)(p0 + t), k);
#pragma unroll
        for (int r = 0; r < PG_PERM_ROUNDS; ++r) s_key[t][r] = k[r];
      }
      __syncthreads();
      for (int j0 = 0; j0 < dmax; j0 += jt) {
        const int nj = min(jt, dmax - j0);
        if (j0 > 0) __syncthreads();
        for (int t = threadIdx.x; t < np * nj; t += TPB) {
          const int pp = t / nj, j = j0 + t - pp * nj;
          uint64_t k[PG_PERM_ROUNDS];
#pragma unroll
          for (int r = 0; r < PG_PERM_ROUNDS; ++r) k[r] = s_key[pp][r];
          int32_t rj = 0;
          pg_perm_walk(j, m, m, hbits, k, [&](int64_t, uint32_t x) { rj = (int32_t)x; });
          PG_ASSERT(rj >= 0 && rj < m);
          s_r[t] = rj;
          s_v[t][0] = z[rj];
          s_v[t][1] = z[rj + 1];
        }
        __syncthreads();
        if (d <= j0) continue;
        const int je = min(d - j0, nj);
        for (int pp = 0; pp < np; ++pp) {
          if (j0 == 0) acc = make_double4(0.0, 0.0, 0.0, 0.0);
          const int base = pp * nj;
          for (int jj = 0; jj < je; ++jj) {
            const int r = s_r[base + jj];
            acc = d4_add(acc, s_v[base + jj][r >= i ? 1 : 0]);
          }
          if (d > j0 + nj) continue;  // the row goes on in the next j tile (one permutation per step)
          const int p = p0 + pp;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const double st = lk_stat(d4_get(acc, k), a[k], b[k]);
            const double dl = st - stat0[k];
            s1[k] += dl;
            s2[k] += dl * dl;
            ge[k] += st >= stat0[k];
            if (o.sims && k < nf) o.sims[((size_t)p * n_feat + 4 * g + k) * (size_t)n + (size_t)i] = st;
          }
        }
      }
    }
  }
  if (!active) return;
  const bool perm = d > 0 && n_perms > 0;
  for (int k = 0; k < nf; ++k) {
    const size_t at = (size_t)(4 * g + k) * (size_t)n + (size_t)i;
    const double e1 = s1[k] / (double)n_perms, e2 = s2[k] / (double)n_perms, v = e2 - e1 * e1;
    if (o.perm_mean) o.perm_mean[at] = perm ? stat0[k] + e1 : nan_d();
    if (o.perm_var) o.perm_var[at] = perm ? (v < 0.0 ? 0.0 : v) : nan_d();  // rounding can dip below 0; NaN stays
    if (o.n_ge) o.n_ge[at] = perm ? ge[k] : 0;
    if (o.sims && d == 0)
      for (int p = 0; p < n_perms; ++p) o.sims[((size_t)p * n_feat + 4 * g + k) * (size_t)n + (size_t)i] = nan_d();
  }
}

}  // namespace

extern "C" {

int pg_local_autocorr(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t n_feat,
                      const double* feat, int32_t flags, int32_t n_perms, uint64_t seed, const pg_local_out* out,
                      pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0, "pg_local_autocorr: negative n");
  PG_REQUIRE(h, n_feat >= 1 && n_feat <= PG_AUTOCORR_MAX_FEAT, "pg_local_autocorr: n_feat must be in 1..%d",
             PG_AUTOCORR_MAX_FEAT);
  PG_REQUIRE(h, n_perms >= 0 && n_perms <= PG_ENRICH_MAX_PERMS, "pg_local_autocorr: n_perms must be in 0..%d",
             PG_ENRICH_MAX_PERMS);
  PG_REQUIRE(h, (flags & ~(PG_AUTOCORR_ROW_STD | PG_LOCAL_GETIS_ORD | PG_LOCAL_STAR)) == 0,
             "pg_local_autocorr: unknown flags %d", flags);
  PG_REQUIRE(h, !(flags & PG_LOCAL_STAR) || (flags & PG_LOCAL_GETIS_ORD),
             "pg_local_autocorr: PG_LOCAL_STAR needs PG_LOCAL_GETIS_ORD");
  PG_REQUIRE(h, row_ptr, "pg_local_autocorr: row_ptr is NULL");
  PG_REQUIRE(h, n == 0 || (col && feat), "pg_local_autocorr: col / feat is NULL");
  pg_local_out o{};
  if (out) o = *out;
  const bool rowstd = flags & PG_AUTOCORR_ROW_STD;
  const int mode = !(flags & PG_LOCAL_GETIS_ORD) ? LK_MORAN : (flags & PG_LOCAL_STAR) ? LK_GI_STAR : LK_GI;
  const int G = (n_feat + 3) / 4;
  const int gx = std::max(1, std::min(pg_div_up(n, TPB), GX_MAX));
  const size_t misc_bytes = sizeof(ac_misc) + 4 * (size_t)G;
  int rc;
  if ((rc = pg_reserve(h, h->ac_z, std::max<size_t>(32, (size_t)G * n * sizeof(double4))))) return rc;
  if ((rc = pg_reserve(h, h->ac_deg, std::max<size_t>(4, (size_t)n * 4)))) return rc;
  if ((rc = pg_reserve(h, h->ac_part, (size_t)G * gx * 4 * 8))) return rc;
  if ((rc = pg_reserve(h, h->ac_misc, misc_bytes))) return rc;
  if ((rc = pg_reserve(h, h->lk_cnt, ((size_t)n + 1) * 4))) return rc;
  if ((rc = pg_reserve(h, h->lk_off, ((size_t)n + 1) * 4))) return rc;
  if ((rc = pg_reserve(h, h->lk_ord, std::max<size_t>(4, (size_t)n * 4)))) return rc;
  ac_misc* misc = (ac_misc*)h->ac_misc.p;
  unsigned int* tickets = (unsigned int*)((char*)h->ac_misc.p + sizeof(ac_misc));
  double* part = (double*)h->ac_part.p;
  double4* zg = (double4*)h->ac_z.p;
  int32_t* deg = (int32_t*)h->ac_deg.p;
  int32_t* cnt = (int32_t*)h->lk_cnt.p;
  int32_t* off = (int32_t*)h->lk_off.p;
  int32_t* ord = (int32_t*)h->lk_ord.p;
  PG_CUDA(h, cudaMemsetAsync(misc, 0, misc_bytes, s));
  PG_CUDA(h, cudaMemsetAsync(cnt, 0, ((size_t)n + 1) * 4, s));

  PG_LAUNCH(h, s, "ac_prep_kernel<0>",
            ac_prep_kernel<0><<<dim3(gx, G), TPB, 0, s>>>(feat, n, n_feat, misc, zg, part, tickets));
  PG_LAUNCH(h, s, "ac_prep_kernel<1>",
            ac_prep_kernel<1><<<dim3(gx, G), TPB, 0, s>>>(feat, n, n_feat, misc, zg, part, tickets));
  const int gn = std::max(1, pg_div_up(n, TPB));
  if (n > 0) {
    PG_LAUNCH(h, s, "lk_degree_kernel", lk_degree_kernel<<<gn, TPB, 0, s>>>(row_ptr, col, n, deg, cnt));
    if ((rc = pg_scan_i32(h, cnt, off, n, s, nullptr, /*clear_in=*/true))) return rc;
    PG_LAUNCH(h, s, "lk_order_kernel", lk_order_kernel<<<gn, TPB, 0, s>>>(n, deg, off, cnt, ord));
  }
  const int hbits = pg_perm_half_bits(n - 1);
  auto node_kernel = mode == LK_MORAN ? lk_node_kernel<LK_MORAN> : mode == LK_GI ? lk_node_kernel<LK_GI>
                                                                                   : lk_node_kernel<LK_GI_STAR>;
  PG_LAUNCH(h, s, "lk_node_kernel",
            node_kernel<<<dim3(gn, G), TPB, 0, s>>>(row_ptr, col, n, deg, ord, zg, n_feat, rowstd, n_perms, hbits, seed,
                                                     misc, o));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
