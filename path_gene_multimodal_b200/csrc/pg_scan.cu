// K3: single-pass exclusive scan (int32) used for cell_start and CSR row pointers.
// The look-back machinery lives in pg_scan.cuh; this file is the plain array scan: tiles of 4096 items
// (256 threads x 16), 1M items = 245 tiles = one look-back group, i.e. no serial chain at all.
#include <algorithm>
#include <climits>
#include <cstring>
#include "pg_scan.cuh"

namespace {

#ifndef PG_SCAN_ITEMS
#define PG_SCAN_ITEMS 16
#endif
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = PG_SCAN_ITEMS;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// CLEAR: the input is zeroed as it is read (the cell histogram is handed back clean for the next build,
// which saves a memset node per build).
// pub.acc != NULL: the first CTA also publishes the degree statistics accumulated by the kernel before
// this one on the stream and resets the accumulators.
template <bool CLEAR>
__global__ void __launch_bounds__(SCAN_THREADS)
scan_kernel(int32_t* in, int32_t* out, int32_t n, pg_scan_state st, int32_t* total_copy, pg_scan_publish pub) {
  using TS = pg_tile_scan<SCAN_THREADS>;
  __shared__ typename TS::smem_t sm;
  pg_pdl_launch();
  pg_pdl_wait();
  if (pub.acc && blockIdx.x == 0) pg_publish_stats(pub, SCAN_THREADS);
  const int tile = TS::take_tile(sm, st);
  const int64_t base = (int64_t)tile * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;

  int v[SCAN_ITEMS];
  if (base + SCAN_ITEMS <= n) {
    int4* p = reinterpret_cast<int4*>(in + base);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS / 4; ++i) {
      int4 q = p[i];
      v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
    }
    if (CLEAR) {
#pragma unroll
      for (int i = 0; i < SCAN_ITEMS / 4; ++i) p[i] = make_int4(0, 0, 0, 0);
    }
  } else {
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
      v[i] = (base + i < n) ? in[base + i] : 0;
      if (CLEAR && base + i < n) in[base + i] = 0;
    }
  }
  int tsum = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) { int x = v[i]; v[i] = tsum; tsum += x; }
  bool last;
  int total;
  const int off = TS::thread_prefix(sm, st, tile, tsum, &last, &total);
  if (threadIdx.x == 0 && last) {
    out[n] = total;
    if (total_copy) *total_copy = total;
  }
  if (base + SCAN_ITEMS <= n) {
    int4* p = reinterpret_cast<int4*>(out + base);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS / 4; ++i)
      p[i] = make_int4(v[4 * i] + off, v[4 * i + 1] + off, v[4 * i + 2] + off, v[4 * i + 3] + off);
  } else {
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i)
      if (base + i < n) out[base + i] = v[i] + off;
  }
}

__global__ void scan_empty_kernel(int32_t* out, int32_t* total_copy) {
  out[0] = 0;
  if (total_copy) *total_copy = 0;
}

// 64-bit sum of the scan's input (two's complement, so the unsigned atomics add signed values correctly)
__global__ void __launch_bounds__(SCAN_THREADS)
sum_i64_kernel(const int32_t* __restrict__ in, int32_t n, unsigned long long* __restrict__ sum) {
  long long v = 0;
  for (int64_t i = (int64_t)blockIdx.x * SCAN_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * SCAN_THREADS) v += in[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0 && v != 0) atomicAdd(sum, (unsigned long long)v);
}

}  // namespace

int pg_scan_prepare(pg_handle* h, int num_tiles, int group, cudaStream_t s, pg_scan_state* st) {
  const int num_groups = pg_div_up(num_tiles, group);
  const size_t need = 256 + (size_t)(num_tiles + num_groups + 2) * sizeof(uint64_t);
  if (need > h->scan_state.cap) {
    int rc = pg_reserve(h, h->scan_state, need);
    if (rc) return rc;
    PG_CUDA(h, cudaMemsetAsync(h->scan_state.p, 0, h->scan_state.cap, s));
  }
  h->scan_epoch += 1;
  if (h->scan_epoch == 0xffffffffu) {  // epoch 0 means "never written": start over on a clean slate
    PG_CUDA(h, cudaMemsetAsync(h->scan_state.p, 0, h->scan_state.cap, s));
    h->scan_epoch = 1;
  }
  st->ticket = (unsigned int*)h->scan_state.p;
  st->agg = (uint64_t*)((char*)h->scan_state.p + 256);
  st->gpre = st->agg + num_tiles;
  st->epoch = h->scan_epoch;
  st->num_tiles = num_tiles;
  return PG_OK;
}

int pg_scan_i32(pg_handle* h, const int32_t* in, int32_t* out, int32_t n, cudaStream_t s, int32_t* total_copy,
                bool clear_in, const pg_scan_publish* publish) {
  pg_scan_publish pub{};
  if (publish) pub = *publish;
  if (n < 0) return pg_set_error(h, PG_ERR_INVALID, "scan: n < 0");
  if (n == 0) {
    PG_LAUNCH(h, s, "scan_empty_kernel", scan_empty_kernel<<<1, 1, 0, s>>>(out, total_copy));
    PG_LAUNCH_CHECK(h);
    return PG_OK;
  }
  if (((uintptr_t)in & 15) || ((uintptr_t)out & 15))
    return pg_set_error(h, PG_ERR_INVALID, "scan: in/out must be 16-byte aligned");
  const int num_tiles = pg_div_up(n, SCAN_TILE);
  pg_scan_state st;
  int rc = pg_scan_prepare(h, num_tiles, SCAN_THREADS, s, &st);
  if (rc) return rc;
  if (clear_in)
    PG_LAUNCH(h, s, "scan_kernel", pg_launch_pdl(1, scan_kernel<true>, num_tiles, SCAN_THREADS, s, const_cast<int32_t*>(in), out, n, st, total_copy, pub));
  else
    PG_LAUNCH(h, s, "scan_kernel", pg_launch_pdl(1, scan_kernel<false>, num_tiles, SCAN_THREADS, s, const_cast<int32_t*>(in), out, n, st, total_copy, pub));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_scan_i32_total(pg_handle* h, const int32_t* in, int32_t* out, int32_t n, cudaStream_t s, int32_t* total_copy,
                      const char* what, int64_t* total) {
  unsigned long long* sum = (unsigned long long*)((char*)h->misc.p + PG_MISC_SUM64);
  PG_CUDA(h, cudaMemsetAsync(sum, 0, sizeof(*sum), s));
  if (n > 0) {
    const int blocks = (int)std::min<int64_t>(pg_div_up(n, SCAN_THREADS), 1024);
    PG_LAUNCH(h, s, "sum_i64_kernel", sum_i64_kernel<<<blocks, SCAN_THREADS, 0, s>>>(in, n, sum));
    PG_LAUNCH_CHECK(h);
  }
  int rc = pg_scan_i32(h, in, out, n, s, total_copy);
  if (rc) return rc;
  PG_CUDA(h, cudaMemcpyAsync(&h->pinned[12], sum, sizeof(*sum), cudaMemcpyDeviceToHost, s));
  PG_CUDA(h, cudaStreamSynchronize(s));
  int64_t t;
  memcpy(&t, &h->pinned[12], sizeof(t));
  if (t < 0 || t > INT32_MAX)
    return pg_set_error(h, PG_ERR_INVALID, "%s: %lld scratch entries needed, more than int32 offsets address (%d)", what,
                        (long long)t, INT32_MAX);
  *total = t;
  return PG_OK;
}

extern "C" int pg_exclusive_scan_i32(pg_handle* h, const int32_t* in, int32_t* out, int32_t n, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = (cudaStream_t)stream;
  return pg_scan_i32(h, in, out, n, (cudaStream_t)stream, nullptr, false);
}
