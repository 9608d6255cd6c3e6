// K5: k-nearest-neighbour query on the uniform grid.
// Reference: /root/reference/hovernet_tile_inference.ipynb:1815-1850 - KNN.from_array(coords, k)
// (libpysal -> scipy cKDTree.query(k+1) minus self) and the per-neighbour sqrt(dx*dx+dy*dy).
// Order is the canonical (d^2, id) of north_star; self is removed by id, so duplicates at
// distance 0 are ordinary neighbours.
//
// Two passes, both one thread per point in cell order:
//   select pass (k <= 16): searches only the 3x3 block of cells around the point - three contiguous runs of the
//       strip-ordered record array, walked as one merged loop with four 256-bit loads in flight, exactly like the
//       radius walk - and picks the k nearest by histogram + rank (see knn_select_kernel); a point is final when
//       its k-th distance does not reach past the block; the others are appended to a retry list.
//   ring pass: the general search (thread per point, ring expansion until the k-th distance is inside the searched
//       block, k best kept sorted in registers) over the retry list - or over every point when k > 16.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include "pg_query.cuh"

namespace {

constexpr int TPB = 128;

// The k best so far, ascending by (d2, id), RIGHT-aligned in KMAX register slots: the k-th best always sits in the
// last slot (so the bar is a fixed register, whatever k is) and the KMAX - k slots in front hold -infinity, which
// nothing ever sorts before. Every index below is a compile-time constant, so the list stays in registers.
template <int KMAX>
struct topk {
  double d2[KMAX];
  int id[KMAX];
  __device__ __forceinline__ void init(int k) {
#pragma unroll
    for (int s = 0; s < KMAX; ++s) {
      const bool used = s >= KMAX - k;
      d2[s] = __longlong_as_double(used ? 0x7ff0000000000000ll : 0xfff0000000000000ll);
      id[s] = used ? 0x7fffffff : -1;
    }
  }
  // insert (cd2, cid), known to sort before the last slot: the last slot drops out. The place r of the newcomer
  // is counted with KMAX - 1 independent comparisons (no serial "already placed" chain), then every slot picks
  // its new content with two integer tests.
  __device__ __forceinline__ void insert(double cd2, int cid) {
    int r = 0;
#pragma unroll
    for (int s = 0; s < KMAX - 1; ++s) r += (d2[s] < cd2 || (d2[s] == cd2 && id[s] < cid)) ? 1 : 0;
#pragma unroll
    for (int s = KMAX - 1; s > 0; --s) {
      const bool shift = s > r, here = s == r;
      d2[s] = shift ? d2[s - 1] : (here ? cd2 : d2[s]);
      id[s] = shift ? id[s - 1] : (here ? cid : id[s]);
    }
    if (r == 0) { d2[0] = cd2; id[0] = cid; }
  }
  __device__ __forceinline__ double worst_d2() const { return d2[KMAX - 1]; }
  __device__ __forceinline__ int worst_id() const { return id[KMAX - 1]; }
};

// the same list for large k, in local memory (dynamic indexing, loops kept rolled): 64 slots do not fit registers
template <int KMAX>
struct topk_local {
  double d2[KMAX];
  int id[KMAX];
  __device__ __forceinline__ void init(int k) {
#pragma unroll 1
    for (int s = 0; s < KMAX; ++s) {
      const bool used = s >= KMAX - k;
      d2[s] = __longlong_as_double(used ? 0x7ff0000000000000ll : 0xfff0000000000000ll);
      id[s] = used ? 0x7fffffff : -1;
    }
  }
  __device__ __forceinline__ void insert(double cd2, int cid) {
    int s = KMAX - 1;
#pragma unroll 1
    while (s > 0 && (cd2 < d2[s - 1] || (cd2 == d2[s - 1] && cid < id[s - 1]))) { d2[s] = d2[s - 1]; id[s] = id[s - 1]; --s; }
    d2[s] = cd2; id[s] = cid;
  }
  __device__ __forceinline__ double worst_d2() const { return d2[KMAX - 1]; }
  __device__ __forceinline__ int worst_id() const { return id[KMAX - 1]; }
};

struct knn_out {
  int32_t* knn_idx;
  double* dist64;
  float* dist32;
  double x_lo, x_hi;
  int32_t* halo_ok;
};

template <int KMAX, class TOP>
__device__ __forceinline__ void write_row(const knn_out& o, const TOP& top, int k, int row, double qx) {
  const int64_t base = (int64_t)row * k - (KMAX - k);
#pragma unroll (KMAX <= 32 ? KMAX : 1)
  for (int s = 0; s < KMAX; ++s) {
    if (s >= KMAX - k) {
      o.knn_idx[base + s] = top.id[s];
      const double d = sqrt(top.d2[s]);
      if (o.dist64) o.dist64[base + s] = d;
      if (o.dist32) o.dist32[base + s] = (float)d;
    }
  }
  if (o.halo_ok) {
    // every point with x in [x_lo, x_hi) is present; the answer is complete iff the k-th
    // neighbour is strictly closer than both faces (slack keeps the test conservative)
    const double dk = sqrt(top.worst_d2()) * (1.0 + 1e-9);
    if (!(dk < qx - o.x_lo && dk < o.x_hi - qx)) atomicExch(o.halo_ok, 0);
  }
}

// distance from (qx, qy) in cell (cx, cy) to the nearest face of the (2R+1)^2 block that still has cells behind it
// (infinity when the block covers the grid), minus a safety margin
__device__ __forceinline__ double block_bound(const pg_grid_view& g, double qx, double qy, int cx, int cy, int R) {
  double bound = __longlong_as_double(0x7ff0000000000000ll);
  if (cx - R > 0) bound = fmin(bound, qx - (g.x0 + (double)(cx - R) * g.cell));
  if (cx + R < g.nx - 1) bound = fmin(bound, (g.x0 + (double)(cx + R + 1) * g.cell) - qx);
  if (cy - R > 0) bound = fmin(bound, qy - (g.y0 + (double)(cy - R) * g.cell));
  if (cy + R < g.ny - 1) bound = fmin(bound, (g.y0 + (double)(cy + R + 1) * g.cell) - qy);
  return bound - 1e-6 * g.cell;
}

// ---- select pass (k <= 16): the same 3x3 block, but no list is kept sorted while candidates stream by.
//   pass 1  histogram of the candidates' squared distances below bound^2 (bound = distance to the nearest block
//           face with cells behind it: nothing beyond it can be trusted) in 16 equal bins of d^2 - uniform points
//           fill them evenly - packed as 16-bit counters in four registers;
//   pick    the first bin b* where the running count reaches k: every point of bins 0..b* is a survivor, the k
//           nearest are among them and (bins being monotone in d^2) nothing outside them can be nearer;
//   pass 2  walk the runs again (L1 hits) and park the <= KMAX + KMAX/2 survivors in shared memory;
//   rank    each survivor counts the survivors that sort before it by (d^2, id) and, if fewer than k do, writes
//           itself straight to that slot of the output row.
// Every lane does the same amount of work (no insertion that runs whenever ANY lane has a hit). A point whose
// block cannot answer (fewer than k candidates inside bound, too many survivors, counters would overflow, the
// block covers the whole grid) goes to the retry list of the ring pass.
template <class F>
__device__ __forceinline__ void walk3x3(const pg_grid_view& g, int cx, int cy, F&& f) {
  const int pad = g.n;  // the sentinel record
  const int sy = cy >> PG_STRIP_LOG, ly = cy & (PG_STRIP - 1);
  const bool has_l = cx > 0, has_r = cx + 1 < g.nx;
  int edge = -1;  // strip-edge points: the row across the edge lives in the adjacent strip
  if (ly == 0 && sy > 0) edge = (((sy - 1) * g.nx + cx) << PG_STRIP_LOG) + PG_STRIP - 1;
  else if (ly == PG_STRIP - 1 && sy + 1 < g.nys) edge = ((sy + 1) * g.nx + cx) << PG_STRIP_LOG;
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    const int32_t* c;
    int lo, hi;
    if (pass == 0) {
      c = g.cell_start + ((sy * g.nx + cx) << PG_STRIP_LOG);
      lo = max(ly - 1, 0); hi = min(ly + 1, PG_STRIP - 1) + 1;
    } else {
      if (edge < 0) break;
      c = g.cell_start + edge;
      lo = 0; hi = 1;
    }
    const int b1 = c[lo], e1 = c[hi];
    int b0 = 0, e0 = 0, b2 = 0, e2 = 0;
    if (has_l) { b0 = c[lo - PG_STRIP]; e0 = c[hi - PG_STRIP]; }
    if (has_r) { b2 = c[lo + PG_STRIP]; e2 = c[hi + PG_STRIP]; }
    const int n0 = e0 - b0, n01 = n0 + (e1 - b1), tot = n01 + (e2 - b2);
    const int off1 = b1 - n0, off2 = b2 - n01;
    auto pos = [&](int t) { return t < tot ? t + (t < n0 ? b0 : (t < n01 ? off1 : off2)) : pad; };
    for (int t = 0; t < tot; t += 4) {
      const int j0 = pos(t), j1 = pos(t + 1), j2 = pos(t + 2), j3 = pos(t + 3);
      PG_ASSERT(j0 >= 0 && j0 <= pad && j1 >= 0 && j1 <= pad && j2 >= 0 && j2 <= pad && j3 >= 0 && j3 <= pad);
      const pg_rec r0 = pg_ld_rec(g.rec + j0), r1 = pg_ld_rec(g.rec + j1);
      const pg_rec r2 = pg_ld_rec(g.rec + j2), r3 = pg_ld_rec(g.rec + j3);
      f(r0); f(r1); f(r2); f(r3);
    }
  }
}

constexpr int SEL_BINS = 16;

template <int KMAX>
__global__ void __launch_bounds__(TPB)
knn_select_kernel(pg_grid_view g, int k, knn_out o, int32_t* retry, int32_t* retry_count) {
  constexpr int S = KMAX + KMAX / 2;  // survivors a thread can park
  __shared__ double s_d2[S][TPB];
  __shared__ int s_id[S][TPB];
  const int tid = threadIdx.x;
  pg_pdl_launch();
  pg_pdl_wait();
  const int p = blockIdx.x * TPB + tid;
  if (p >= g.n) return;
  const pg_rec me = pg_ld_rec_ordered(g.rec + p);
  if (me.row >= g.n_query) return;  // halo points own no row
  const int cx = pg_cell_coord(me.x, g.x0, g.inv_cell, g.nx);
  const int cy = pg_cell_coord(me.y, g.y0, g.inv_cell, g.ny);
  const double bound = block_bound(g, me.x, me.y, cx, cy, 1);
  auto walk = [&](auto&& f) __attribute__((always_inline)) { walk3x3(g, cx, cy, f); };
  bool ok = bound > 0.0 && bound < 1e300;  // infinite: the block covers the grid (tiny inputs) - ring pass
  const double bound2 = ok ? bound * bound : 0.0;  // the histogram spans [0, bound^2)
  const double inv_binw = ok ? (double)SEL_BINS / bound2 : 0.0;
  ok = ok && inv_binw < 1e300;

  // ---- pass 1: histogram of d^2 below bound^2
  unsigned long long pk0 = 0, pk1 = 0, pk2 = 0, pk3 = 0;
  int seen = 0;
  auto bin_of = [&](double d2) { return min(SEL_BINS - 1, __double2int_rd(__dmul_rn(d2, inv_binw))); };
  if (ok) {
    walk([&](const pg_rec& c) {
      const double d2 = pg_dist2(me.x, me.y, c.x, c.y);
      ++seen;
      if (d2 < bound2 && c.id != me.id) {
        const int b = bin_of(d2);
        const unsigned long long inc = 1ull << ((b & 3) * 16);
        const int w = b >> 2;
        pk0 += w == 0 ? inc : 0ull; pk1 += w == 1 ? inc : 0ull;
        pk2 += w == 2 ? inc : 0ull; pk3 += w == 3 ? inc : 0ull;
      }
    });
    ok = seen < 65536;  // 16-bit counters
  }
  // ---- pick the bin that holds the k-th nearest
  int bstar = -1, m = 0;
  if (ok) {
    int cum = 0;
#pragma unroll
    for (int b = 0; b < SEL_BINS; ++b) {
      const unsigned long long w = b < 4 ? pk0 : (b < 8 ? pk1 : (b < 12 ? pk2 : pk3));
      cum += (int)((w >> ((b & 3) * 16)) & 0xffffu);
      if (bstar < 0 && cum >= k) { bstar = b; m = cum; }
    }
    ok = bstar >= 0 && m <= S;
  }
  if (!ok) {
    const int slot = atomicAdd(retry_count, 1);
    PG_ASSERT(slot >= 0 && slot < g.n);
    retry[slot] = p;
    return;
  }
  // ---- pass 2: park the survivors
  int cnt = 0;
  walk([&](const pg_rec& c) {
    const double d2 = pg_dist2(me.x, me.y, c.x, c.y);
    if (d2 < bound2 && c.id != me.id && bin_of(d2) <= bstar && cnt < S) {
      s_d2[cnt][tid] = d2; s_id[cnt][tid] = c.id;
      ++cnt;
    }
  });
  // ---- rank: place = number of survivors that sort before (ids are distinct)
  const int64_t base = (int64_t)me.row * k;
  for (int a = 0; a < cnt; ++a) {
    const double da = s_d2[a][tid];
    const int ia = s_id[a][tid];
    int rank = 0;
    for (int b = 0; b < cnt; ++b) {
      const double db = s_d2[b][tid];
      const int ib = s_id[b][tid];
      rank += (db < da || (db == da && ib < ia)) ? 1 : 0;
    }
    if (rank < k) {
      PG_ASSERT(me.row >= 0 && me.row < g.n_query && ia >= 0);
      o.knn_idx[base + rank] = ia;
      const double d = sqrt(da);
      if (o.dist64) o.dist64[base + rank] = d;
      if (o.dist32) o.dist32[base + rank] = (float)d;
      if (rank == k - 1 && o.halo_ok) {  // see write_row
        const double dk = d * (1.0 + 1e-9);
        if (!(dk < me.x - o.x_lo && dk < o.x_hi - me.x)) atomicExch(o.halo_ok, 0);
      }
    }
  }
}

// ---- ring pass: over `list[0 .. *list_count)` (positions in the cell-ordered array), or over every point
template <int KMAX, class TOP>
__global__ void __launch_bounds__(TPB)
knn_ring_kernel(pg_grid_view g, int k, knn_out o, const int32_t* list, const int32_t* list_count) {
  pg_pdl_launch();
  pg_pdl_wait();
  const int limit = list ? *list_count : g.n;
  for (int t = blockIdx.x * TPB + threadIdx.x; t < limit; t += gridDim.x * TPB) {
    const int p = list ? list[t] : t;
    const pg_rec me = pg_ld_rec_ordered(g.rec + p);
    if (me.row >= g.n_query) continue;
    const double2 q = make_double2(me.x, me.y);
    const int cx = pg_cell_coord(q.x, g.x0, g.inv_cell, g.nx);
    const int cy = pg_cell_coord(q.y, g.y0, g.inv_cell, g.ny);
    TOP top;
    top.init(k);
    double wd2 = top.worst_d2();
    int wid = top.worst_id();
    auto consider = [&](const pg_rec& c) __attribute__((always_inline)) {
      const double d2 = pg_dist2(q.x, q.y, c.x, c.y);
      if (d2 <= wd2 && c.id != me.id) {
        const int cid = c.id;
        if (d2 < wd2 || cid < wid) {
          top.insert(d2, cid);
          wd2 = top.worst_d2();
          wid = top.worst_id();
        }
      }
    };
    const int pad = g.n;  // the sentinel record (infinitely far: never inserted)
    auto scan = [&](int b, int e) __attribute__((always_inline)) {
      if (KMAX > 16) {  // every point takes this path: one candidate at a time keeps the long list in registers
        for (int j = b; j < e; ++j) consider(pg_ld_rec(g.rec + j));
        return;
      }
      for (int j = b; j < e; j += 4) {  // four loads in flight: the retried points are few, their latency is what costs
        const int p1 = j + 1 < e ? j + 1 : pad, p2 = j + 2 < e ? j + 2 : pad, p3 = j + 3 < e ? j + 3 : pad;
        const pg_rec r0 = pg_ld_rec(g.rec + j), r1 = pg_ld_rec(g.rec + p1);
        const pg_rec r2 = pg_ld_rec(g.rec + p2), r3 = pg_ld_rec(g.rec + p3);
        consider(r0); consider(r1); consider(r2); consider(r3);
      }
    };
    int R = 1;
    pg_visit_block(g, cx, cy, 1, scan);
    while (true) {
      const bool covers = cx - R <= 0 && cx + R >= g.nx - 1 && cy - R <= 0 && cy + R >= g.ny - 1;
      if (covers) break;
      const double bound = block_bound(g, q.x, q.y, cx, cy, R);
      if (bound > 0.0 && wd2 <= bound * bound) break;
      ++R;
      pg_visit_ring(g, cx, cy, R, scan);
    }
    write_row<KMAX>(o, top, k, me.row, q.x);
  }
}

// knn_neighbor_coords of cell 11 (ipynb:1838-1840): out[i][s] = xy[knn_idx[i][s]], one thread per list entry
__global__ void __launch_bounds__(256)
knn_coords_kernel(const int32_t* __restrict__ idx, const double2* __restrict__ xy, int64_t entries, int32_t n_points, double2* __restrict__ out) {
  const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (e >= entries) return;
  const int j = idx[e];
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  out[e] = (j >= 0 && j < n_points) ? xy[j] : make_double2(nan, nan);
}

__global__ void knn_prepare_kernel(int32_t* halo_ok, int32_t* retry_count) {
  if (halo_ok) *halo_ok = 1;
  *retry_count = 0;
}

}  // namespace

extern "C" int pg_knn(pg_handle* h, int32_t k, int32_t* knn_idx, double* dist64, float* dist32,
                      double x_lo, double x_hi, int32_t* halo_ok, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  if (!h->grid.built) return pg_set_error(h, PG_ERR_STATE, "pg_knn: call pg_grid_build first");
  const pg_grid& gr = h->grid;
  PG_REQUIRE(h, k >= 1 && k <= PG_MAX_K, "pg_knn: k must be in 1..%d (got %d)", PG_MAX_K, k);
  PG_REQUIRE(h, k < gr.n, "pg_knn: k (%d) must be smaller than the number of points (%d)", k, gr.n);
  // no query rows (a strip that holds only halo points): the [0, k] outputs may be empty allocations
  PG_REQUIRE(h, knn_idx != nullptr || gr.n_query == 0, "pg_knn: knn_idx is NULL");
  int32_t* retry_count = (int32_t*)((char*)h->misc.p + PG_MISC_KNN_RETRY);
  PG_LAUNCH(h, s, "knn_prepare_kernel", knn_prepare_kernel<<<1, 1, 0, s>>>(halo_ok, retry_count));
  PG_LAUNCH_CHECK(h);
  if (gr.n_query == 0) return PG_OK;
  pg_grid_view v = pg_make_view(h);
  knn_out o{knn_idx, dist64, dist32, x_lo, x_hi, halo_ok};
  const int blocks = pg_div_up(gr.n, TPB);
  if (k <= 16) {
    int rc = pg_reserve(h, h->knn_retry, ((size_t)gr.n + 8) * sizeof(int32_t));
    if (rc) return rc;
    int32_t* retry = (int32_t*)h->knn_retry.p;
    // 3x3 select over every point -> retry list -> ring pass over the list. (Tried and measured slower at the ~6 %
    // retry rate of a 1.15 d_k cell: a 5x5 select pass over the list, and one warp per retried point - see DESIGN.md.)
    const int ring_blocks = std::min(blocks, h->sm_count * 8);
    if (k <= 8) {
      PG_LAUNCH(h, s, "knn_select_kernel<8>", pg_launch_pdl(6, knn_select_kernel<8>, blocks, TPB, s, v, (int)k, o, retry, retry_count));
      PG_LAUNCH(h, s, "knn_ring_kernel<8>", pg_launch_pdl(7, knn_ring_kernel<8, topk<8>>, ring_blocks, TPB, s, v, (int)k, o, (const int32_t*)retry, (const int32_t*)retry_count));
    } else {
      PG_LAUNCH(h, s, "knn_select_kernel<16>", pg_launch_pdl(6, knn_select_kernel<16>, blocks, TPB, s, v, (int)k, o, retry, retry_count));
      PG_LAUNCH(h, s, "knn_ring_kernel<16>", pg_launch_pdl(7, knn_ring_kernel<16, topk<16>>, ring_blocks, TPB, s, v, (int)k, o, (const int32_t*)retry, (const int32_t*)retry_count));
    }
  } else if (k <= 32) {
    PG_LAUNCH(h, s, "knn_ring_kernel<32>", pg_launch_pdl(7, knn_ring_kernel<32, topk<32>>, blocks, TPB, s, v, (int)k, o, (const int32_t*)nullptr, (const int32_t*)nullptr));
  } else {
    PG_LAUNCH(h, s, "knn_ring_kernel<64>", pg_launch_pdl(7, knn_ring_kernel<64, topk_local<64>>, blocks, TPB, s, v, (int)k, o, (const int32_t*)nullptr, (const int32_t*)nullptr));
  }
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

extern "C" int pg_knn_neighbor_coords(pg_handle* h, int32_t n_rows, int32_t k, const int32_t* knn_idx, const double* xy,
                                      int32_t n_points, double* out_xy, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n_rows >= 0 && k >= 1 && n_points >= 0, "pg_knn_neighbor_coords: bad sizes");
  PG_REQUIRE(h, n_rows == 0 || (knn_idx && xy && out_xy), "pg_knn_neighbor_coords: NULL array");
  PG_REQUIRE(h, (((uintptr_t)xy | (uintptr_t)out_xy) & 15) == 0, "pg_knn_neighbor_coords: xy / out must be 16-byte aligned");
  const int64_t entries = (int64_t)n_rows * k;
  if (entries == 0) return PG_OK;
  PG_LAUNCH(h, s, "knn_coords_kernel", knn_coords_kernel<<<pg_div_up(entries, 256), 256, 0, s>>>(knn_idx, (const double2*)xy, entries, n_points, (double2*)out_xy));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}
