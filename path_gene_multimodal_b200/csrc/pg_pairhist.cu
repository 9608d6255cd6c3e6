// K16: type-pair distance histogram over the built grid (squidpy.gr.co_occurrence's counts, Ripley's K; definition in
// include/pathgraph.h).
//
// pair_hist_kernel: one warp per query point, points taken in cell order (8 neighbours per CTA step share most of their
// candidate records in L1). The (2R+1)^2 block of the point is enumerated as runs of the cell-ordered array (one per
// column and strip, pg_visit_column's split); the warp holds up to 32 runs at a time, one per lane, scans their lengths
// and strides its 32 lanes over the flattened candidate range, finding each lane's run with a 5-step shuffle search. So
// every loop of the walk has a warp-uniform trip count, the lanes stay busy however short the runs are, and the full-warp
// __match_any_sync below is legal.
//
// Counters: per CTA [n_thr][T][T] uint32 in shared memory (64 KB at T = 16 and 64 thresholds), flushed to the int64
// histogram with one global atomic per non-zero counter. A pair's bin is a binary search over the squared thresholds
// in shared memory. All lanes of a warp share the query point's type, so on C2 (half the nuclei of type 1) many lanes
// hit the same (bin, 1, 1) counter: lanes with the same counter are aggregated (__match_any_sync) and one of them adds
// the group's size.
//
// Overflow bound: a counter grows by at most one per candidate a warp of the CTA walks, so between two flushes it holds
// at most the sum of the CTA's walked candidates since the last flush. Before every step each warp publishes its point's
// candidate count c_w (<= n - 1 < 2^31) and every thread replays the same running sum: a flush is placed before warp w
// walks whenever acc + c_w would pass 2^32 - 1. One step thus splits into phases only in the quadratic regime (t_max
// spanning a slide of about 2^32 / 8 points per CTA step); otherwise the CTA flushes once, at its end.
// Only integer atomics: the histogram does not depend on the run, the schedule or the handle.
#include <algorithm>
#include <cmath>
#include "pg_query.cuh"

namespace {

constexpr int TPB = 256;
constexpr int WARPS = TPB / 32;
constexpr int STEPS_PER_TICKET = 16;             // CTA steps (of WARPS points) per ticket taken from the global cursor
constexpr int TICKET = WARPS * STEPS_PER_TICKET;
// The flush bound. A -DPG_CHECK build may lower it (PG_PAIRHIST_COUNTER_MAX=...) so that ordinary test inputs take the
// flush phases; the histogram does not depend on it.
#ifndef PG_PAIRHIST_COUNTER_MAX
#define PG_PAIRHIST_COUNTER_MAX 0xffffffffull
#endif
constexpr unsigned long long COUNTER_MAX = PG_PAIRHIST_COUNTER_MAX;

struct thr_t {
  double t2[PG_PAIRHIST_MAX_THR];  // squared thresholds, ascending
};

struct hist_out {
  unsigned long long* hist;        // [n_thr][T][T]
  unsigned long long* type_count;  // [T] or NULL
  unsigned long long* ticket;      // zeroed before the launch
};

// The runs of the block around (cx, cy): run r = (column xa + r % ncols, strip sa + r / ncols).
struct block_runs {
  int xa, ya, yb, sa, ncols, nruns;
};

__device__ __forceinline__ block_runs make_runs(const pg_grid_view& g, int cx, int cy, int R) {
  block_runs b;
  b.xa = max(cx - R, 0);
  const int xb = min(cx + R, g.nx - 1);
  b.ya = max(cy - R, 0);
  b.yb = min(cy + R, g.ny - 1);
  b.sa = b.ya >> PG_STRIP_LOG;
  b.ncols = xb - b.xa + 1;
  b.nruns = b.ncols * ((b.yb >> PG_STRIP_LOG) - b.sa + 1);
  return b;
}

// [begin, end) of run r in the cell-ordered array (empty for r >= nruns)
__device__ __forceinline__ int2 run_at(const pg_grid_view& g, const block_runs& b, int r) {
  if (r >= b.nruns) return make_int2(0, 0);
  const int s = b.sa + r / b.ncols, x = b.xa + r % b.ncols;
  const int s0 = s << PG_STRIP_LOG;
  const int la = max(b.ya, s0) - s0, lb = min(b.yb, s0 + PG_STRIP - 1) - s0;
  const int32_t* c = g.cell_start + (((int64_t)s * g.nx + x) << PG_STRIP_LOG);
  return make_int2(c[la], c[lb + 1]);
}

__device__ __forceinline__ void flush_counters(uint32_t* s_cnt, int nk, unsigned long long* hist) {
  for (int k = threadIdx.x; k < nk; k += TPB) {
    const uint32_t v = s_cnt[k];
    if (v) {
      atomicAdd(&hist[k], (unsigned long long)v);
      s_cnt[k] = 0u;
    }
  }
}

__global__ void __launch_bounds__(TPB)
pair_hist_kernel(pg_grid_view g, int R, int n_types, int n_thr, thr_t thr, hist_out o) {
  extern __shared__ uint32_t s_cnt[];  // [n_thr][T][T]
  __shared__ double s_t2[PG_PAIRHIST_MAX_THR];
  __shared__ unsigned long long s_cand[2][WARPS];
  __shared__ unsigned long long s_tc[PG_MAX_TYPES];
  __shared__ long long s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tt = n_types * n_types, nk = n_thr * tt;
  for (int k = tid; k < nk; k += TPB) s_cnt[k] = 0u;
  if (tid < PG_PAIRHIST_MAX_THR) s_t2[tid] = thr.t2[tid];
  if (tid < PG_MAX_TYPES) s_tc[tid] = 0ull;
  unsigned long long acc = 0;  // candidates walked by the CTA since the last flush (identical in every thread)
  int parity = 0;

  for (;;) {
    __syncthreads();  // (first pass: the zeroed counters; later: every thread has read s_base)
    if (tid == 0) s_base = (long long)atomicAdd(o.ticket, (unsigned long long)TICKET);
    __syncthreads();
    const long long base = s_base;
    if (base >= g.n) break;  // CTA-uniform
    const double t2max = s_t2[n_thr - 1];
    for (int step = 0; step < STEPS_PER_TICKET; ++step) {
      // ---- this warp's point and its candidate count
      const long long q = base + (long long)step * WARPS + warp;
      bool walk = false;
      pg_rec me;
      block_runs b;
      unsigned long long cand = 0;
      if (q < g.n) {
        me = pg_ld_rec(g.rec + q);
        if (me.row < g.n_query && me.type >= 1 && me.type <= n_types) {
          walk = true;
          const int cx = pg_cell_coord(me.x, g.x0, g.inv_cell, g.nx);
          const int cy = pg_cell_coord(me.y, g.y0, g.inv_cell, g.ny);
          b = make_runs(g, cx, cy, R);
          for (int r0 = 0; r0 < b.nruns; r0 += 32) {
            const int2 be = run_at(g, b, r0 + lane);
            cand += (unsigned long long)__reduce_add_sync(0xffffffffu, (unsigned)(be.y - be.x));
          }
        }
        if (walk && lane == 0) atomicAdd(&s_tc[me.type - 1], 1ull);
      }
      if (lane == 0) s_cand[parity][warp] = cand;
      __syncthreads();
      // ---- phases: a flush goes before warp w whenever the CTA's counters could otherwise pass 2^32 - 1
      unsigned flush_before = 0;
#pragma unroll
      for (int w = 0; w < WARPS; ++w) {
        const unsigned long long c = s_cand[parity][w];
        if (acc + c > COUNTER_MAX) { flush_before |= 1u << w; acc = 0; }
        acc += c;
      }
      parity ^= 1;
      for (int w0 = 0; w0 < WARPS;) {
        int w1 = w0 + 1;
        while (w1 < WARPS && !((flush_before >> w1) & 1u)) ++w1;
        if ((flush_before >> w0) & 1u) {  // CTA-uniform
          __syncthreads();
          flush_counters(s_cnt, nk, o.hist);
          __syncthreads();
        }
        if (walk && warp >= w0 && warp < w1) {
          const int arow = (me.type - 1) * n_types;
          for (int r0 = 0; r0 < b.nruns; r0 += 32) {
            const int2 be = run_at(g, b, r0 + lane);
            const int len = be.y - be.x;
            int incl = len;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
              const int y = __shfl_up_sync(0xffffffffu, incl, d);
              if (lane >= d) incl += y;
            }
            const int excl = incl - len;
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            for (int p0 = 0; p0 < total; p0 += 32) {
              const int p = p0 + lane;
              int k = 0;  // the last run that starts at or before p (empty runs share their start with the next)
#pragma unroll
              for (int st = 16; st > 0; st >>= 1) {
                const int v = __shfl_sync(0xffffffffu, excl, k + st);
                if (v <= p) k += st;
              }
              const int rb = __shfl_sync(0xffffffffu, be.x, k), rx = __shfl_sync(0xffffffffu, excl, k);
              int key = -1;
              if (p < total) {
                const int j = rb + (p - rx);
                PG_ASSERT(j >= 0 && j < g.n);
                const pg_rec c = pg_ld_rec(g.rec + j);
                const double d2 = pg_dist2(me.x, me.y, c.x, c.y);
                if (c.id != me.id && c.type >= 1 && c.type <= n_types && d2 <= t2max) {
                  int lo = 0, hi = n_thr - 1;  // the first bin whose squared threshold is >= d2
                  while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (d2 <= s_t2[mid]) hi = mid; else lo = mid + 1;
                  }
                  key = lo * tt + arow + (c.type - 1);
                }
              }
              const unsigned peers = __match_any_sync(0xffffffffu, key);
              if (key >= 0 && lane == __ffs(peers) - 1) {
                PG_ASSERT(key < nk);
                atomicAdd(&s_cnt[key], (uint32_t)__popc(peers));
              }
            }
          }
        }
        w0 = w1;
      }
    }
  }
  flush_counters(s_cnt, nk, o.hist);  // the loop ended on a barrier: every warp's counts are in
  if (o.type_count && tid < n_types && s_tc[tid]) atomicAdd(&o.type_count[tid], s_tc[tid]);
}

}  // namespace

extern "C" {

int pg_pair_dist_hist(pg_handle* h, int32_t n_types, int32_t n_thr, const double* thresholds, int64_t* hist,
                      int64_t* type_count, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  if (!h->grid.built) return pg_set_error(h, PG_ERR_STATE, "pg_pair_dist_hist: call pg_grid_build first");
  PG_REQUIRE(h, n_types >= 1 && n_types <= PG_MAX_TYPES, "pg_pair_dist_hist: n_types must be in 1..%d", PG_MAX_TYPES);
  PG_REQUIRE(h, n_thr >= 1 && n_thr <= PG_PAIRHIST_MAX_THR, "pg_pair_dist_hist: n_thr must be in 1..%d",
             PG_PAIRHIST_MAX_THR);
  PG_REQUIRE(h, thresholds != nullptr && hist != nullptr, "pg_pair_dist_hist: thresholds / hist is NULL");
  PG_REQUIRE(h, (((uintptr_t)hist | (uintptr_t)type_count) & 7) == 0, "pg_pair_dist_hist: hist / type_count must be 8-byte aligned");
  thr_t thr;
  for (int b = 0; b < PG_PAIRHIST_MAX_THR; ++b) thr.t2[b] = INFINITY;
  for (int b = 0; b < n_thr; ++b) {
    const double t = thresholds[b];
    PG_REQUIRE(h, std::isfinite(t) && t >= 0, "pg_pair_dist_hist: thresholds must be finite and >= 0");
    PG_REQUIRE(h, b == 0 || t > thresholds[b - 1], "pg_pair_dist_hist: thresholds must be strictly ascending");
    thr.t2[b] = t * t;  // rounded once, as the radius rule's r * r
  }
  const pg_grid& gr = h->grid;
  const int tt = n_types * n_types, nk = n_thr * tt;
  PG_CUDA(h, cudaMemsetAsync(hist, 0, (size_t)nk * sizeof(int64_t), s));
  if (type_count) PG_CUDA(h, cudaMemsetAsync(type_count, 0, (size_t)n_types * sizeof(int64_t), s));
  if (gr.n == 0 || gr.n_query == 0) return PG_OK;
  unsigned long long* ticket = (unsigned long long*)((char*)h->misc.p + PG_MISC_PAIRHIST_TICKET);
  PG_CUDA(h, cudaMemsetAsync(ticket, 0, sizeof(unsigned long long), s));

  const int R = pg_ring_radius(thresholds[n_thr - 1], gr);
  const size_t smem = (size_t)nk * sizeof(uint32_t);
  PG_CUDA(h, cudaFuncSetAttribute(pair_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  PG_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pair_hist_kernel, TPB, smem));
  const int blocks = std::max(1, std::min(std::max(per_sm, 1) * h->sm_count, pg_div_up(gr.n, TICKET)));
  hist_out o{(unsigned long long*)hist, (unsigned long long*)type_count, ticket};
  PG_LAUNCH(h, s, "pair_hist_kernel",
            pair_hist_kernel<<<blocks, TPB, smem, s>>>(pg_make_view(h), R, n_types, n_thr, thr, o));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
