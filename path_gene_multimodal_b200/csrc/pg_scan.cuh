// Device-side core of the single-pass exclusive scan (K3), shared by the plain scan kernel (pg_scan.cu)
// and the fused row scan + un-permute kernel of the radius graph (pg_radius.cu).
// Decoupled look-back organised for short chains: tiles are handed out by an atomic ticket (so a tile only
// ever waits on tiles that are already running); every tile publishes its aggregate at once, then sums the
// aggregates of the earlier tiles of its GROUP (THREADS tiles) directly, one descriptor per thread - a
// single L2 round trip - and adds the inclusive prefix published by the last tile of the previous group.
// Descriptor words carry an epoch tag, so nothing has to be cleared between scans.
#pragma once
#include "pg_common.cuh"

struct pg_scan_state {
  uint64_t* agg;         // [num_tiles] aggregate of one tile
  uint64_t* gpre;        // [num_groups] inclusive prefix up to the end of a group
  unsigned int* ticket;  // tile dispenser, re-armed by the tile that takes the last ticket
  uint32_t epoch;
  int num_tiles;
};

// reserves / versions the descriptor storage for a scan of num_tiles tiles with groups of `group` tiles
int pg_scan_prepare(pg_handle* h, int num_tiles, int group, cudaStream_t s, pg_scan_state* st);

#ifdef __CUDACC__
__device__ __forceinline__ uint64_t pg_pack_desc(uint32_t epoch, int32_t value) {
  return ((uint64_t)epoch << 32) | (uint32_t)value;
}
__device__ __forceinline__ uint64_t pg_ld_relaxed_u64(const uint64_t* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void pg_st_relaxed_u64(uint64_t* p, uint64_t v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

template <int THREADS>
struct pg_tile_scan {
  struct smem_t {
    int tile;
    int warp_sum[THREADS / PG_WARP];
    int red[THREADS / PG_WARP];
  };

  // all threads call; returns the tile this CTA works on
  static __device__ __forceinline__ int take_tile(smem_t& sm, const pg_scan_state& st) {
    if (threadIdx.x == 0) {
      int t = (int)atomicAdd(st.ticket, 1u);
      if (t == st.num_tiles - 1) atomicExch(st.ticket, 0u);  // every ticket is out: re-arm for the next scan
      sm.tile = t;
    }
    __syncthreads();
    return sm.tile;
  }

  // all threads call with the sum of their own items; returns the exclusive prefix of the thread's first
  // item over the whole array. total (if the tile is the last one) receives the grand total.
  static __device__ __forceinline__ int thread_prefix(smem_t& sm, const pg_scan_state& st, int tile, int tsum,
                                                      bool* is_last_tile, int* grand_total) {
    int tile_sum;
    const int thread_off = local_scan(sm, st, tile, tsum, &tile_sum);
    return thread_off + look_back(sm, st, tile, tile_sum, is_last_tile, grand_total);
  }

  // first half: scan inside the tile and publish the tile's aggregate at once; returns the exclusive prefix of
  // the thread's first item inside the tile. Work placed between the two halves overlaps the look-back wait.
  static __device__ __forceinline__ int local_scan(smem_t& sm, const pg_scan_state& st, int tile, int tsum, int* tile_sum_out) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int incl = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += y;
    }
    if (lane == 31) sm.warp_sum[warp] = incl;
    __syncthreads();
    int warp_off = 0, tile_sum = 0;
#pragma unroll
    for (int w = 0; w < THREADS / PG_WARP; ++w) {
      int s = sm.warp_sum[w];
      if (w < warp) warp_off += s;
      tile_sum += s;
    }
    if (tid == 0) pg_st_relaxed_u64(&st.agg[tile], pg_pack_desc(st.epoch, tile_sum));
    *tile_sum_out = tile_sum;
    return warp_off + incl - tsum;
  }

  // second half: prefix of this tile = prefix of the previous group + aggregates of the earlier tiles of my group
  static __device__ __forceinline__ int look_back(smem_t& sm, const pg_scan_state& st, int tile, int tile_sum,
                                                  bool* is_last_tile, int* grand_total) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int group = tile / THREADS, first = group * THREADS;
    int contrib = 0;
    const int pred = first + tid;
    if (pred < tile) {
      uint64_t w;
      do { w = pg_ld_relaxed_u64(&st.agg[pred]); } while ((uint32_t)(w >> 32) != st.epoch);
      contrib = (int32_t)(uint32_t)w;
    }
    if (tid == THREADS - 1 && group > 0) {  // this lane never has a predecessor (pred >= first + THREADS - 1 >= tile)
      uint64_t w;
      do { w = pg_ld_relaxed_u64(&st.gpre[group - 1]); } while ((uint32_t)(w >> 32) != st.epoch);
      contrib = (int32_t)(uint32_t)w;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, d);
    if (lane == 0) sm.red[warp] = contrib;
    __syncthreads();
    int prefix = 0;
#pragma unroll
    for (int w = 0; w < THREADS / PG_WARP; ++w) prefix += sm.red[w];
    if (tid == 0 && tile == first + THREADS - 1) pg_st_relaxed_u64(&st.gpre[group], pg_pack_desc(st.epoch, prefix + tile_sum));
    *is_last_tile = tile == st.num_tiles - 1;
    *grand_total = prefix + tile_sum;
    return prefix;
  }
};
#endif
