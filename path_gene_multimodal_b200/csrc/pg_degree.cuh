// Degree statistics of the graph producers: the K6 row pass (pg_radius.cu), the K7 rank pass and K8
// pg_compose_degree (pg_graph.cu). Min, max, sum, sum of squares and node count of the degrees, and a histogram whose
// last bin takes every degree >= hist_len - 1.
// Every CTA reduces its nodes thread -> warp -> CTA in shared memory and adds its share to accumulators kept in the
// handle (PG_MISC_ACC / PG_MISC_ACC_HIST); the CTA that finishes last copies them to the caller's pg_degree_stats /
// hist and puts them back into their reset state, so the reduction needs no init / finish launches of its own. A
// histogram longer than PG_ACC_HIST_MAX bins skips the shared bins and the accumulators: its nodes add straight into
// the caller's hist, which pg_degree_prepare zeroes first.
#pragma once
#include "pg_common.cuh"

// All zero between launches - the state pg_create's clear of the misc buffer leaves - like the histogram accumulators.
struct pg_stats_acc {
  unsigned int not_min;  // ~(min degree): for d >= 0, ~d as unsigned falls as d rises, and every ~d is above 0
  unsigned int max1;     // max degree + 1
  unsigned long long sum, sumsq;
  unsigned int done;     // CTAs finished
};

// the kernels' view of the caller's outputs
struct pg_degree_out {
  pg_degree_stats* stats;  // NULL: not wanted
  int32_t* hist;           // NULL: not wanted
  int hist_len;
  pg_stats_acc* acc;
  int32_t* acc_hist;
};

// Builds the view for a graph of n nodes. Zeroes a histogram too long for the shared bins; for n == 0 writes the
// empty graph's result (statistics and histogram all zero), and no kernel has to run.
static inline int pg_degree_prepare(pg_handle* h, pg_degree_stats* stats, int32_t* hist, int32_t hist_len, int64_t n,
                                    cudaStream_t s, pg_degree_out* o) {
  o->stats = stats;
  o->hist = hist;
  o->hist_len = hist ? hist_len : 0;
  o->acc = (pg_stats_acc*)((char*)h->misc.p + PG_MISC_ACC);
  o->acc_hist = (int32_t*)((char*)h->misc.p + PG_MISC_ACC_HIST);
  if (stats && n == 0) PG_CUDA(h, cudaMemsetAsync(stats, 0, sizeof(*stats), s));
  if (hist && (n == 0 || hist_len > PG_ACC_HIST_MAX))
    PG_CUDA(h, cudaMemsetAsync(hist, 0, (size_t)hist_len * sizeof(int32_t), s));
  return PG_OK;
}

#ifdef __CUDACC__
// One CTA of THREADS threads. Every thread calls arm, and a CTA barrier follows before the first add; add and commit
// are warp-collective; finish is for all threads, after a CTA barrier that follows every commit.
template <int THREADS>
struct pg_degree_cta {
  struct smem_t {
    unsigned long long sum, sq;
    int hist[PG_ACC_HIST_MAX];
    int mn, mx, last;
  };
  smem_t& sm;
  const pg_degree_out& o;  // a kernel parameter
  int mn = 0x7fffffff, mx = -1;  // this thread's nodes
  long long sum = 0, sq = 0;

  __device__ __forceinline__ pg_degree_cta(smem_t& s, const pg_degree_out& out) : sm(s), o(out) {}

  static __device__ __forceinline__ bool on(const pg_degree_out& o) { return o.stats != nullptr || o.hist != nullptr; }
  static __device__ __forceinline__ bool shared_bins(const pg_degree_out& o) {
    return o.hist != nullptr && o.hist_len <= PG_ACC_HIST_MAX;
  }

  // the CTA's shared state: zero bins, empty min / max / sums
  static __device__ __forceinline__ void arm(smem_t& sm, const pg_degree_out& o) {
    if (shared_bins(o))
      for (int i = threadIdx.x; i < o.hist_len; i += THREADS) sm.hist[i] = 0;
    if (threadIdx.x == 0) { sm.mn = 0x7fffffff; sm.mx = -1; sm.sum = 0; sm.sq = 0; }
  }

  // every lane calls, with or without a node. Degrees cluster on a few bins: one atomic per distinct bin of the warp
  // instead of one per lane.
  __device__ __forceinline__ void add(int deg, bool valid) {
    if (o.hist) {
      const int bin = valid ? min(deg, o.hist_len - 1) : -1;
      const unsigned int peers = __match_any_sync(0xffffffffu, bin);
      if (valid && (threadIdx.x & 31) == __ffs(peers) - 1) {  // two calls: a shared-memory atomic, not a generic one
        if (shared_bins(o)) atomicAdd(&sm.hist[bin], __popc(peers));
        else atomicAdd(&o.hist[bin], __popc(peers));
      }
    }
    if (o.stats && valid) { mn = min(mn, deg); mx = max(mx, deg); sum += deg; sq += (long long)deg * deg; }
  }

  // warp -> CTA
  __device__ __forceinline__ void commit() {
    if (!o.stats) return;
    const int wmn = __reduce_min_sync(0xffffffffu, mn), wmx = __reduce_max_sync(0xffffffffu, mx);
    long long wsum = sum, wsq = sq;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { wsum += __shfl_xor_sync(0xffffffffu, wsum, d); wsq += __shfl_xor_sync(0xffffffffu, wsq, d); }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(&sm.mn, wmn); atomicMax(&sm.mx, wmx);
      atomicAdd(&sm.sum, (unsigned long long)wsum); atomicAdd(&sm.sq, (unsigned long long)wsq);
    }
  }

  // CTA -> accumulators; the last CTA of the grid publishes the statistics of the graph's n_nodes nodes and re-arms
  // the accumulators. Returns (in every thread) whether this CTA was the last.
  __device__ __forceinline__ bool finish(long long n_nodes) {
    if (o.stats && threadIdx.x == 0) {
      atomicMax(&o.acc->not_min, ~(unsigned int)sm.mn); atomicMax(&o.acc->max1, (unsigned int)(sm.mx + 1));
      atomicAdd(&o.acc->sum, sm.sum); atomicAdd(&o.acc->sumsq, sm.sq);
    }
    if (shared_bins(o))
      for (int i = threadIdx.x; i < o.hist_len; i += THREADS)
        if (sm.hist[i]) atomicAdd(&o.acc_hist[i], sm.hist[i]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) sm.last = atomicAdd(&o.acc->done, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!sm.last) return false;
    __threadfence();
    if (shared_bins(o))
      for (int i = threadIdx.x; i < o.hist_len; i += THREADS) {
        o.hist[i] = *(volatile int32_t*)&o.acc_hist[i];
        o.acc_hist[i] = 0;
      }
    if (threadIdx.x == 0) {
      volatile pg_stats_acc* a = o.acc;
      if (o.stats) {
        o.stats->min_degree = n_nodes ? (int32_t)~a->not_min : 0;
        o.stats->max_degree = n_nodes ? (int32_t)a->max1 - 1 : 0;
        o.stats->sum_degree = (long long)a->sum; o.stats->sumsq_degree = (long long)a->sumsq;
        o.stats->n_nodes = n_nodes;
      }
      a->not_min = 0; a->max1 = 0; a->sum = 0; a->sumsq = 0; a->done = 0;
    }
    return true;
  }
};
#endif
