// K19: cell clusters - connected components and DBSCAN over a CSR, and a per-cluster table (definitions in
// include/pathgraph.h).
//
// Components are found by union-find in the style of ECL-CC (Jaiganesh & Burtscher 2018), which needs no round per unit
// of graph diameter (a slide-wide chain of nuclei has a diameter in the thousands; label propagation would need as many
// rounds):
//   cl_core_kernel      DBSCAN only, thread / row: core_i = (in-range non-self entries + 1 >= min_samples); the row walk
//                       stops at min_samples - 1 entries, so a clump's long rows cost no more than a short one.
//   cl_init_kernel      parent[v] = v.
//   cl_hook_kernel      the warp-flattened row walk of K11 / K17 / K18 (a warp owns 32 consecutive rows and its lanes
//                       take the rows' entries 32 at a time): every joining entry (i, j) finds both roots with path
//                       halving and links the larger root under the smaller one with atomicCAS. parent[v] <= v always,
//                       and a link only ever hangs a root under a smaller root, so every tree's root is its smallest
//                       member whatever order the atomics arrive in.
//   cl_compress_kernel  parent[v] = root(v); is_root[v] = (root == v), and core for DBSCAN.
//   pg_scan_i32         rank = exclusive scan of is_root; the total is the label count.
//   cl_label_kernel     label[v] = rank[parent[v]] (components; DBSCAN core nodes), -1 for the others.
//   cl_border_kernel    DBSCAN only, thread / row: a non-core node takes the smallest label among its core neighbours.
// So the labels number the components in the order of their smallest (core) member, which is scipy's and sklearn's
// numbering, and they do not depend on the run.
//
// The table groups the members by label with a stable LSD counting sort - no atomic decides an output position:
//   cl_hist_kernel      members per cluster (integer atomics: the counts do not depend on the order) -> scan = offsets.
//   per 8-bit digit of the label, least significant first:
//     cl_digit_count_kernel  tile / CTA: members per digit in the tile, stored digit-major -> scan = each (digit, tile)'s
//                            first output slot;
//     cl_digit_place_kernel  tile / CTA, in node order within the tile: a member's slot = its (digit, tile) start + the
//                            tile's earlier members of the digit, from warp __match_any_sync ranks and per-warp digit
//                            counts in shared memory (K9's stable in-CTA ranking).
//   The first pass reads the nodes 0..n-1 in order and drops the non-members; later passes read the previous order.
//   cl_props_kernel     warp / cluster over its members in ascending node index: counts, per-type counts, fixed-order
//                       coordinate sums, bounding box and the grouped member coordinates.
#include <algorithm>
#include <cmath>
#include "pg_common.cuh"

namespace {

constexpr int TPB = 256;
constexpr int WARPS = TPB / 32;
constexpr int DIGIT_BITS = 8;
constexpr int DIGITS = 1 << DIGIT_BITS;
constexpr int PLACE_ROUNDS = 8;                  // rounds of TPB members a placing CTA walks
constexpr int TILE = TPB * PLACE_ROUNDS;         // members per tile of the LSD passes
constexpr unsigned FULL = 0xffffffffu;

// root of v: ECL-CC's path halving. parent[] only ever moves towards smaller ancestors of the same tree, so a stale read
// makes a path longer, never wrong; the reads bypass L1 so that another SM's links are seen.
__device__ __forceinline__ int uf_find(int32_t* parent, int v) {
  int cur = __ldcg(parent + v);
  if (cur != v) {
    int prev = v, next;
    while (cur > (next = __ldcg(parent + cur))) {
      parent[prev] = next;
      prev = cur;
      cur = next;
    }
  }
  return cur;
}

__device__ __forceinline__ void uf_union(int32_t* parent, int a, int b) {
  a = uf_find(parent, a);
  b = uf_find(parent, b);
  while (a != b) {
    const int hi = max(a, b), lo = min(a, b);
    const int old = atomicCAS(parent + hi, hi, lo);
    if (old == hi) return;
    // hi was linked meanwhile: continue from its new root
    if (hi == a) a = uf_find(parent, old); else b = uf_find(parent, old);
  }
}

__global__ void __launch_bounds__(TPB)
cl_core_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n, int need,
               uint8_t* __restrict__ core) {
  const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (i >= n) return;
  int d = 0;
  for (int p = row_ptr[i], e = row_ptr[i + 1]; p < e && d < need; ++p) {
    const int j = col[p];
    d += (unsigned)j < (unsigned)n && j != i;
  }
  core[i] = d >= need;
}

__global__ void __launch_bounds__(TPB) cl_init_kernel(int n, int32_t* __restrict__ parent) {
  const int64_t v = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (v < n) parent[v] = (int32_t)v;
}

// DBSCAN: only core-core entries join (core != NULL)
__global__ void __launch_bounds__(TPB)
cl_hook_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
               const uint8_t* __restrict__ core, int32_t* parent) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t rb = ((int64_t)blockIdx.x * WARPS + warp) * 32; rb < n; rb += (int64_t)gridDim.x * WARPS * 32) {
    const int64_t own = rb + lane;
    const int rp = row_ptr[min(own, (int64_t)n)];
    const int begin = __shfl_sync(FULL, rp, 0);
    const int end = row_ptr[min(rb + 32, (int64_t)n)];
    const int act = own < n && (!core || core[own]);
    if (!__any_sync(FULL, act)) continue;
    for (int64_t p0 = begin; p0 < end; p0 += 32) {
      const int64_t p = p0 + lane;
      int kk = 0;  // the last of the 32 rows whose range starts at or before p
#pragma unroll
      for (int step = 16; step > 0; step >>= 1) {
        const int v = __shfl_sync(FULL, rp, kk + step);
        if (v <= p) kk += step;
      }
      const int ok = __shfl_sync(FULL, act, kk);
      if (p >= end || !ok) continue;
      const int i = (int)(rb + kk), j = col[p];
      if ((unsigned)j >= (unsigned)n || j == i || (core && !core[j])) continue;
      uf_union(parent, i, j);
    }
  }
}

__global__ void __launch_bounds__(TPB)
cl_compress_kernel(int n, const uint8_t* __restrict__ core, int32_t* parent, int32_t* __restrict__ is_root) {
  const int64_t v = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (v >= n) return;
  int r = parent[v];
  for (int q; r != (q = parent[r]);) r = q;
  parent[v] = r;
  is_root[v] = r == v && (!core || core[v]);
}

__global__ void __launch_bounds__(TPB)
cl_label_kernel(int n, const uint8_t* __restrict__ core, const int32_t* __restrict__ parent,
                const int32_t* __restrict__ rank, int32_t* __restrict__ label) {
  const int64_t v = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (v >= n) return;
  label[v] = (!core || core[v]) ? rank[parent[v]] : -1;
}

// sklearn's dbscan_inner grows clusters one at a time in label order, and a border point joins the first cluster that
// reaches it, i.e. the smallest label among its core neighbours
__global__ void __launch_bounds__(TPB)
cl_border_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
                 const uint8_t* __restrict__ core, int32_t* __restrict__ label) {
  const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (i >= n || core[i]) return;
  int best = INT32_MAX;
  for (int p = row_ptr[i], e = row_ptr[i + 1]; p < e; ++p) {
    const int j = col[p];
    if ((unsigned)j >= (unsigned)n || j == i || !core[j]) continue;
    best = min(best, label[j]);
  }
  label[i] = best == INT32_MAX ? -1 : best;
}

__global__ void __launch_bounds__(TPB)
cl_hist_kernel(int n, const int32_t* __restrict__ label, int k, int32_t* __restrict__ count) {
  const int64_t v = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (v >= n) return;
  const int c = label[v];
  if ((unsigned)c < (unsigned)k) atomicAdd(count + c, 1);
}

// element e of an LSD pass: (node, digit), digit DIGITS when e holds no member. FIRST: e is node e itself and a label
// outside [0, k) is not a member; later passes: the members, in the previous pass's order, m_dev[0] of them.
template <bool FIRST>
__device__ __forceinline__ int lsd_digit(int64_t e, int m, const int32_t* __restrict__ in,
                                         const int32_t* __restrict__ label, int k, int shift, int* node) {
  *node = -1;
  if (e >= m) return DIGITS;
  const int v = FIRST ? (int)e : in[e];
  const int c = label[v];
  if (FIRST && (unsigned)c >= (unsigned)k) return DIGITS;
  *node = v;
  return (c >> shift) & (DIGITS - 1);
}

template <bool FIRST>
__global__ void __launch_bounds__(TPB)
cl_digit_count_kernel(const int32_t* __restrict__ in, int n, const int32_t* __restrict__ m_dev,
                      const int32_t* __restrict__ label, int k, int shift, int n_tiles, int32_t* __restrict__ cnt) {
  __shared__ int h[DIGITS];
  for (int d = threadIdx.x; d < DIGITS; d += TPB) h[d] = 0;
  __syncthreads();
  const int m = FIRST ? n : *m_dev;
  const int64_t t0 = (int64_t)blockIdx.x * TILE;
  for (int r = 0; r < PLACE_ROUNDS; ++r) {
    int node;
    const int d = lsd_digit<FIRST>(t0 + (int64_t)r * TPB + threadIdx.x, m, in, label, k, shift, &node);
    if (d < DIGITS) atomicAdd(h + d, 1);
  }
  __syncthreads();
  for (int d = threadIdx.x; d < DIGITS; d += TPB) cnt[(int64_t)d * n_tiles + blockIdx.x] = h[d];
}

template <bool FIRST>
__global__ void __launch_bounds__(TPB)
cl_digit_place_kernel(const int32_t* __restrict__ in, int n, const int32_t* __restrict__ m_dev,
                      const int32_t* __restrict__ label, int k, int shift, int n_tiles,
                      const int32_t* __restrict__ start, int32_t* __restrict__ out) {
  __shared__ int wcnt[WARPS][DIGITS];
  __shared__ int base[DIGITS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int m = FIRST ? n : *m_dev;
  const int64_t t0 = (int64_t)blockIdx.x * TILE;
  if (t0 >= m) return;  // CTA-uniform
  for (int d = tid; d < DIGITS; d += TPB) {
    base[d] = start[(int64_t)d * n_tiles + blockIdx.x];
    for (int w = 0; w < WARPS; ++w) wcnt[w][d] = 0;
  }
  __syncthreads();
  const unsigned lt = (1u << lane) - 1u;
  for (int r = 0; r < PLACE_ROUNDS; ++r) {
    int node;
    const int d = lsd_digit<FIRST>(t0 + (int64_t)r * TPB + tid, m, in, label, k, shift, &node);
    const unsigned peers = __match_any_sync(FULL, d);
    const int rank = __popc(peers & lt);
    if (d < DIGITS && rank == 0) wcnt[warp][d] = __popc(peers);
    __syncthreads();
    if (d < DIGITS) {
      int slot = base[d] + rank;
      for (int w = 0; w < warp; ++w) slot += wcnt[w][d];
      PG_ASSERT(slot >= 0 && slot < m);
      out[slot] = node;
    }
    __syncthreads();
    for (int dd = tid; dd < DIGITS; dd += TPB) {
      int s = 0;
      for (int w = 0; w < WARPS; ++w) { s += wcnt[w][dd]; wcnt[w][dd] = 0; }
      base[dd] += s;
    }
    __syncthreads();
  }
}

// warp / cluster c: members order[off[c] .. off[c + 1]) in ascending node index
__global__ void __launch_bounds__(TPB)
cl_props_kernel(const int32_t* __restrict__ order, const int32_t* __restrict__ off, int k,
                const double2* __restrict__ xy, const int32_t* __restrict__ type, int n_types,
                const uint8_t* __restrict__ core, pg_cluster_out o) {
  __shared__ int tc[WARPS][PG_MAX_TYPES];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * WARPS + warp;
  if (c >= k) return;  // warp-uniform
  if (lane < PG_MAX_TYPES) tc[warp][lane] = 0;
  __syncwarp();
  const int b = off[c], e = off[c + 1];
  double sx = 0.0, sy = 0.0;
  double x0 = INFINITY, y0 = INFINITY, x1 = -INFINITY, y1 = -INFINITY;
  int n_core = 0;
  for (int p = b + lane; p < e; p += 32) {
    const int v = order[p];
    const double2 q = xy[v];
    sx += q.x;
    sy += q.y;
    x0 = fmin(x0, q.x); y0 = fmin(y0, q.y); x1 = fmax(x1, q.x); y1 = fmax(y1, q.y);
    if (core) n_core += core[v] != 0;
    if (type) {
      const int t = type[v];
      if (t >= 1 && t <= n_types) atomicAdd(&tc[warp][t - 1], 1);
    }
    if (o.member_xy) reinterpret_cast<double2*>(o.member_xy)[p] = q;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    sx += __shfl_down_sync(FULL, sx, s);
    sy += __shfl_down_sync(FULL, sy, s);
    x0 = fmin(x0, __shfl_down_sync(FULL, x0, s));
    y0 = fmin(y0, __shfl_down_sync(FULL, y0, s));
    x1 = fmax(x1, __shfl_down_sync(FULL, x1, s));
    y1 = fmax(y1, __shfl_down_sync(FULL, y1, s));
    n_core += __shfl_down_sync(FULL, n_core, s);
  }
  __syncwarp();
  if (o.type_count && lane < n_types) o.type_count[c * n_types + lane] = tc[warp][lane];
  if (lane != 0) return;
  const int m = e - b;
  if (o.n_members) o.n_members[c] = m;
  if (o.n_core) o.n_core[c] = n_core;
  if (o.member_off) {
    o.member_off[c] = b;
    if (c == k - 1) o.member_off[k] = e;
  }
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  if (o.centroid) {
    o.centroid[2 * c] = m ? sx / (double)m : nan;
    o.centroid[2 * c + 1] = m ? sy / (double)m : nan;
  }
  if (o.bbox) {
    o.bbox[4 * c] = m ? x0 : nan;
    o.bbox[4 * c + 1] = m ? y0 : nan;
    o.bbox[4 * c + 2] = m ? x1 : nan;
    o.bbox[4 * c + 3] = m ? y1 : nan;
  }
}

int blocks_for(int64_t n) { return std::max(1, pg_div_up(n, TPB)); }

// shared by pg_connected_components (core == NULL) and pg_dbscan
int components(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, const uint8_t* core,
               int32_t* label, int32_t* n_labels, cudaStream_t s) {
  int rc;
  if ((rc = pg_reserve(h, h->cl_parent, std::max<size_t>(16, (size_t)n * 4)))) return rc;
  if ((rc = pg_reserve(h, h->cl_count, std::max<size_t>(16, (size_t)n * 4)))) return rc;
  if ((rc = pg_reserve(h, h->cl_scan, (size_t)n * 4 + 16))) return rc;
  int32_t* parent = (int32_t*)h->cl_parent.p;
  int32_t* is_root = (int32_t*)h->cl_count.p;
  int32_t* rank = (int32_t*)h->cl_scan.p;
  if (n > 0) {
    PG_LAUNCH(h, s, "cl_init_kernel", cl_init_kernel<<<blocks_for(n), TPB, 0, s>>>(n, parent));
    PG_LAUNCH(h, s, "cl_hook_kernel", cl_hook_kernel<<<blocks_for(n), TPB, 0, s>>>(row_ptr, col, n, core, parent));
    PG_LAUNCH(h, s, "cl_compress_kernel",
              cl_compress_kernel<<<blocks_for(n), TPB, 0, s>>>(n, core, parent, is_root));
  }
  if ((rc = pg_scan_i32(h, is_root, rank, n, s, n_labels))) return rc;
  if (n > 0) {
    PG_LAUNCH(h, s, "cl_label_kernel", cl_label_kernel<<<blocks_for(n), TPB, 0, s>>>(n, core, parent, rank, label));
    if (core)
      PG_LAUNCH(h, s, "cl_border_kernel", cl_border_kernel<<<blocks_for(n), TPB, 0, s>>>(row_ptr, col, n, core, label));
  }
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // namespace

extern "C" {

int pg_connected_components(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t* label,
                            int32_t* n_labels, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0, "pg_connected_components: negative n");
  PG_REQUIRE(h, row_ptr && n_labels, "pg_connected_components: row_ptr / n_labels is NULL");
  PG_REQUIRE(h, n == 0 || (col && label), "pg_connected_components: col / label is NULL");
  return components(h, n, row_ptr, col, nullptr, label, n_labels, s);
}

int pg_dbscan(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t min_samples,
              int32_t* label, uint8_t* core, int32_t* n_labels, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0, "pg_dbscan: negative n");
  PG_REQUIRE(h, min_samples >= 1, "pg_dbscan: min_samples must be >= 1");
  PG_REQUIRE(h, row_ptr && n_labels, "pg_dbscan: row_ptr / n_labels is NULL");
  PG_REQUIRE(h, n == 0 || (col && label && core), "pg_dbscan: col / label / core is NULL");
  if (n > 0)
    PG_LAUNCH(h, s, "cl_core_kernel",
              cl_core_kernel<<<blocks_for(n), TPB, 0, s>>>(row_ptr, col, n, min_samples - 1, core));
  return components(h, n, row_ptr, col, core, label, n_labels, s);
}

int pg_cluster_props(pg_handle* h, int32_t n, const int32_t* label, int32_t n_clusters, const double* xy,
                     const int32_t* type, int32_t n_types, const uint8_t* core, const pg_cluster_out* out,
                     pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && n_clusters >= 0, "pg_cluster_props: negative n / n_clusters");
  PG_REQUIRE(h, n_types >= 1 && n_types <= PG_MAX_TYPES, "pg_cluster_props: n_types must be in 1..%d", PG_MAX_TYPES);
  PG_REQUIRE(h, out, "pg_cluster_props: out is NULL");
  pg_cluster_out o = *out;
  PG_REQUIRE(h, n == 0 || (label && xy), "pg_cluster_props: label / xy is NULL");
  PG_REQUIRE(h, n == 0 || !o.type_count || type, "pg_cluster_props: type_count needs type");
  PG_REQUIRE(h, n == 0 || !o.n_core || core, "pg_cluster_props: n_core needs core");
  PG_REQUIRE(h, ((uintptr_t)xy & 15) == 0 && ((uintptr_t)o.member_xy & 15) == 0,
             "pg_cluster_props: xy / member_xy must be 16-byte aligned");
  if (o.member_off && n_clusters == 0) PG_CUDA(h, cudaMemsetAsync(o.member_off, 0, 4, s));
  if (n_clusters == 0) return PG_OK;
  const int n_tiles = std::max(1, pg_div_up(n, TILE));
  const size_t scan_len = std::max<size_t>((size_t)n_clusters, (size_t)DIGITS * n_tiles);
  if ((size_t)DIGITS * n_tiles > INT32_MAX) return pg_set_error(h, PG_ERR_INVALID, "pg_cluster_props: n too large");
  int rc;
  if ((rc = pg_reserve(h, h->cl_parent, std::max<size_t>(16, (size_t)n * 4)))) return rc;
  if ((rc = pg_reserve(h, h->cl_order, std::max<size_t>(16, (size_t)n * 4)))) return rc;
  if ((rc = pg_reserve(h, h->cl_count, scan_len * 4))) return rc;
  if ((rc = pg_reserve(h, h->cl_scan, scan_len * 4 + 16))) return rc;
  if ((rc = pg_reserve(h, h->cl_off, (size_t)n_clusters * 4 + 16))) return rc;
  int32_t* cnt = (int32_t*)h->cl_count.p;
  int32_t* start = (int32_t*)h->cl_scan.p;
  int32_t* off = (int32_t*)h->cl_off.p;  // [k + 1]; off[k] = the members, the element count of the later passes
  int32_t* buf[2] = {(int32_t*)h->cl_parent.p, (int32_t*)h->cl_order.p};

  PG_CUDA(h, cudaMemsetAsync(cnt, 0, (size_t)n_clusters * 4, s));
  if (n > 0) PG_LAUNCH(h, s, "cl_hist_kernel", cl_hist_kernel<<<blocks_for(n), TPB, 0, s>>>(n, label, n_clusters, cnt));
  if ((rc = pg_scan_i32(h, cnt, off, n_clusters, s))) return rc;

  int passes = 1;
  while (passes * DIGIT_BITS < 31 && ((int64_t)(n_clusters - 1) >> (passes * DIGIT_BITS)) != 0) ++passes;
  const int32_t* in = nullptr;
  for (int p = 0; p < passes && n > 0; ++p) {
    const int shift = p * DIGIT_BITS;
    int32_t* dst = buf[p & 1];
    if (p == 0) {
      PG_LAUNCH(h, s, "cl_digit_count_kernel",
                cl_digit_count_kernel<true><<<n_tiles, TPB, 0, s>>>(in, n, off + n_clusters, label, n_clusters, shift,
                                                                   n_tiles, cnt));
    } else {
      PG_LAUNCH(h, s, "cl_digit_count_kernel",
                cl_digit_count_kernel<false><<<n_tiles, TPB, 0, s>>>(in, n, off + n_clusters, label, n_clusters, shift,
                                                                    n_tiles, cnt));
    }
    if ((rc = pg_scan_i32(h, cnt, start, DIGITS * n_tiles, s))) return rc;
    if (p == 0) {
      PG_LAUNCH(h, s, "cl_digit_place_kernel",
                cl_digit_place_kernel<true><<<n_tiles, TPB, 0, s>>>(in, n, off + n_clusters, label, n_clusters, shift,
                                                                   n_tiles, start, dst));
    } else {
      PG_LAUNCH(h, s, "cl_digit_place_kernel",
                cl_digit_place_kernel<false><<<n_tiles, TPB, 0, s>>>(in, n, off + n_clusters, label, n_clusters, shift,
                                                                    n_tiles, start, dst));
    }
    in = dst;
  }
  PG_LAUNCH(h, s, "cl_props_kernel",
            cl_props_kernel<<<pg_div_up(n_clusters, WARPS), TPB, 0, s>>>(in, off, n_clusters, (const double2*)xy, type,
                                                                         n_types, core, o));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
