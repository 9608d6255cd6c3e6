// K15: neighbourhood enrichment - the type-interaction matrix of an undirected edge list against the same counts under
// random relabelling of the nodes (squidpy.gr.nhood_enrichment's label-permutation z-score; definition and statistics
// in include/pathgraph.h).
//
// The labellings are processed in chunks of rows: row 0 is the identity (the observed matrix, counted by the same
// kernel as the permutations), row p + 1 is permutation p. A chunk holds at most PG_ENRICH_CHUNK_BYTES of uint8
// labels, so its rows stay in L2 between the two kernels of the chunk and a 20 M-nucleus slide needs a bounded
// workspace.
//   perm_labels_kernel  lab[row][i] = type[pi_p(i)] as uint8 (0 = outside 1..T). One keyed Feistel evaluation per node
//                       and permutation (x cycle-walks; pg_perm.cuh, shared with K17); each lane walks its own queue
//                       of nodes, so a lane whose walk is long does not hold the other 31 lanes back.
//   perm_count_kernel   grid-stride over the edge rows of one labelling; every (t_i, t_j) pair is counted once in a
//                       lane-private shared-memory column ([T*T][32] uint32: a warp's 32 increments always hit 32
//                       different banks, so the dominant pair - type 1 x type 1 is a quarter of all entries on C2 -
//                       does not serialise), then flushed with one warp reduction and one int64 atomic per pair.
//   enrich_finish_kernel  one warp per (a, b): c_p = u_p[a][b] + u_p[b][a] of the ordered-pair counts u, S1 and the
//                       128-bit S2 over p, and the four outputs, each exact integer converted to float64 once.
// Only integer atomics: the outputs do not depend on the order in which they arrive.
#include <algorithm>
#include "pg_common.cuh"
#include "pg_perm.cuh"

namespace {

constexpr int TPB = 256;
constexpr int LAB_PER_THREAD = 16;     // nodes a labels thread walks (amortises its 8 round keys)
constexpr int EDGES_PER_THREAD = 16;   // edge rows a count thread takes per labelling (amortises the counter flush)

__device__ __forceinline__ uint8_t label_of(int t, int n_types) {
  return (t >= 1 && t <= n_types) ? (uint8_t)t : (uint8_t)0;
}

// lab[blockIdx.y][i] for the labelling row0 + blockIdx.y
__global__ void __launch_bounds__(TPB)
perm_labels_kernel(const int32_t* __restrict__ type, int n, int n_types, int hbits, uint64_t seed, int row0,
                   uint8_t* __restrict__ lab) {
  const int row = row0 + blockIdx.y;
  uint8_t* out = lab + (size_t)blockIdx.y * (size_t)n;
  const int64_t stride = (int64_t)gridDim.x * TPB;
  int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (row == 0) {
    for (; i < n; i += stride) out[i] = label_of(__ldg(&type[i]), n_types);
    return;
  }
  uint64_t k[PG_PERM_ROUNDS];
  pg_perm_keys(seed, (uint64_t)(row - 1), k);
  pg_perm_walk(i, stride, n, hbits, k, [&](int64_t v, uint32_t x) { out[v] = label_of(__ldg(&type[x]), n_types); });
}

// cnt[blockIdx.y][(a-1) T + (b-1)] += number of edge rows (i, j) with labels (a, b) in labelling blockIdx.y
__global__ void __launch_bounds__(TPB)
perm_count_kernel(const int32_t* __restrict__ edges, int64_t n_edges, int n, int n_types,
                  const uint8_t* __restrict__ lab, unsigned long long* __restrict__ cnt) {
  extern __shared__ uint32_t s_c[];  // [T*T][32]
  const int nk = n_types * n_types, lane = threadIdx.x & 31;
  for (int q = threadIdx.x; q < nk * 32; q += TPB) s_c[q] = 0u;
  __syncthreads();
  const uint8_t* t = lab + (size_t)blockIdx.y * (size_t)n;
  const int64_t stride = (int64_t)gridDim.x * TPB;
  for (int64_t e = (int64_t)blockIdx.x * TPB + threadIdx.x; e < n_edges; e += stride) {
    const int i = __ldg(&edges[2 * e]), j = __ldg(&edges[2 * e + 1]);
    if ((unsigned)i >= (unsigned)n || (unsigned)j >= (unsigned)n) continue;
    const int a = __ldg(&t[i]), b = __ldg(&t[j]);
    if (a == 0 || b == 0) continue;
    atomicAdd(&s_c[((a - 1) * n_types + (b - 1)) * 32 + lane], 1u);
  }
  __syncthreads();
  unsigned long long* out = cnt + (size_t)blockIdx.y * (size_t)nk;
  for (int q = threadIdx.x >> 5; q < nk; q += TPB / 32) {
    const uint32_t v = __reduce_add_sync(0xffffffffu, s_c[q * 32 + lane]);
    if (lane == 0 && v) atomicAdd(&out[q], (unsigned long long)v);
  }
}

__global__ void __launch_bounds__(TPB)
enrich_finish_kernel(const unsigned long long* __restrict__ cnt, int n_types, int n_perms, pg_enrich_out o) {
  const int nk = n_types * n_types;
  const int w = (blockIdx.x * TPB + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= nk) return;  // warp-uniform
  const int ab = w, ba = (w % n_types) * n_types + w / n_types;
  unsigned long long s1 = 0ull;
  unsigned __int128 s2 = 0;
  for (int p = lane; p < n_perms; p += 32) {
    const unsigned long long* row = cnt + (size_t)(p + 1) * (size_t)nk;
    const unsigned long long c = row[ab] + row[ba];
    s1 += c;
    s2 += (unsigned __int128)c * c;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, d);
    const unsigned long long lo = __shfl_xor_sync(0xffffffffu, (unsigned long long)s2, d);
    const unsigned long long hi = __shfl_xor_sync(0xffffffffu, (unsigned long long)(s2 >> 64), d);
    s2 += ((unsigned __int128)hi << 64) | lo;
  }
  if (lane != 0) return;
  const long long c0 = (long long)(cnt[ab] + cnt[ba]);
  const long long S1 = (long long)s1, P = n_perms;
  const __int128 var = (__int128)P * (__int128)s2 - (__int128)S1 * S1;  // P^2 x the ddof-0 variance, exact
  const double sd = __dsqrt_rn((double)var);
  if (o.count) o.count[w] = c0;
  if (o.perm_mean) o.perm_mean[w] = __ddiv_rn((double)S1, (double)P);
  if (o.perm_std) o.perm_std[w] = __ddiv_rn(sd, (double)P);
  if (o.zscore) o.zscore[w] = __ddiv_rn((double)(P * c0 - S1), sd);
}

}  // namespace

extern "C" {

int pg_nhood_enrichment(pg_handle* h, int32_t n, const int32_t* type, int32_t n_types, int64_t n_edges,
                        const int32_t* edges, int32_t n_perms, uint64_t seed, const pg_enrich_out* out,
                        pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && n_edges >= 0, "pg_nhood_enrichment: negative size");
  PG_REQUIRE(h, n_types >= 1 && n_types <= PG_MAX_TYPES, "pg_nhood_enrichment: n_types must be in 1..%d", PG_MAX_TYPES);
  PG_REQUIRE(h, n_perms >= 1 && n_perms <= PG_ENRICH_MAX_PERMS, "pg_nhood_enrichment: n_perms must be in 1..%d",
             PG_ENRICH_MAX_PERMS);
  PG_REQUIRE(h, n == 0 || type, "pg_nhood_enrichment: type is NULL");
  PG_REQUIRE(h, n_edges == 0 || edges, "pg_nhood_enrichment: edges is NULL");
  PG_REQUIRE(h, ((uintptr_t)edges & 3) == 0, "pg_nhood_enrichment: edges must be 4-byte aligned");
  pg_enrich_out o{};
  if (out) o = *out;
  const int nk = n_types * n_types;
  const int64_t rows_total = (int64_t)n_perms + 1;
  int rc;
  if ((rc = pg_reserve(h, h->enrich_cnt, (size_t)rows_total * nk * sizeof(int64_t)))) return rc;
  unsigned long long* cnt = (unsigned long long*)h->enrich_cnt.p;
  PG_CUDA(h, cudaMemsetAsync(cnt, 0, (size_t)rows_total * nk * sizeof(int64_t), s));
  if (n > 0 && n_edges > 0) {
    const int hbits = pg_perm_half_bits(n);
    const int64_t chunk = std::min<int64_t>({std::max<int64_t>(1, (int64_t)PG_ENRICH_CHUNK_BYTES / n), rows_total, 65535});
    if ((rc = pg_reserve(h, h->enrich_lab, (size_t)chunk * (size_t)n))) return rc;
    uint8_t* lab = (uint8_t*)h->enrich_lab.p;
    const int gx_lab = (int)std::min<int64_t>(pg_div_up(n, (int64_t)TPB * LAB_PER_THREAD), 1 << 20);
    const int gx_cnt = (int)std::min<int64_t>(pg_div_up(n_edges, (int64_t)TPB * EDGES_PER_THREAD), 1 << 20);
    const size_t smem = (size_t)nk * 32 * sizeof(uint32_t);
    for (int64_t r0 = 0; r0 < rows_total; r0 += chunk) {
      const int rows = (int)std::min(chunk, rows_total - r0);
      PG_LAUNCH(h, s, "perm_labels_kernel",
                perm_labels_kernel<<<dim3(gx_lab, rows), TPB, 0, s>>>(type, n, n_types, hbits, seed, (int)r0, lab));
      PG_LAUNCH(h, s, "perm_count_kernel",
                perm_count_kernel<<<dim3(gx_cnt, rows), TPB, smem, s>>>(edges, n_edges, n, n_types, lab,
                                                                        cnt + (size_t)r0 * nk));
    }
  }
  PG_LAUNCH(h, s, "enrich_finish_kernel",
            enrich_finish_kernel<<<pg_div_up((int64_t)nk * 32, TPB), TPB, 0, s>>>(cnt, n_types, n_perms, o));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
