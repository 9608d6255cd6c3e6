// Strip sharding of one giant slide (SURVEY 8e, BASELINE config 5): the device-side pieces of the exchange steps
// (K9), most of which the first version left to eager torch ops (bucketize / argsort / index_put):
//   pg_strip_partition   points -> 24-byte records grouped by owning strip (the send buffer of the all-to-all),
//                        stable and deterministic: count per (strip, CTA) -> one look-back scan -> placement by
//                        warp match + in-CTA prefix. No atomics, no sort.
//   pg_halo_pack / _push the points near the strip edges -> 24-byte records, into a local buffer (then all-gathered)
//                        or straight into every peer's receive slab.
//   pg_halo_unpack_multi several x-ranges of the gathered (or, _slab, the received) halo records appended behind the
//                        owned points in one enqueue (each range starts where the previous one ended, read on the
//                        device), so the host reads all counts with ONE synchronisation.
//   pg_gid_maps          dense maps global id -> local row and global id -> type for the undirected union of a
//                        strip + halo (rows address their neighbours by global id).
// No reference counterpart: the reference runs one slide per LSF job (/root/reference/main.py:322-335).
#include <algorithm>
#include "pg_common.cuh"

namespace {

constexpr int TPB = 256;
constexpr int MAX_STRIPS = 64;

struct strip_edges {
  int n_inner;                    // world - 1
  double inner[MAX_STRIPS - 1];   // ascending
};

// torch.bucketize(x, inner, right=True): the number of inner edges <= x
__device__ __forceinline__ int owner_of(double x, const strip_edges& e) {
  int o = 0;
  for (int q = 0; q < e.n_inner; ++q) o += x >= e.inner[q] ? 1 : 0;
  return o;
}

__global__ void __launch_bounds__(TPB)
partition_count_kernel(const double2* __restrict__ xy, int n, strip_edges e, int n_cta, int32_t* __restrict__ counts) {
  __shared__ int s_cnt[MAX_STRIPS];
  const int world = e.n_inner + 1;
  if (threadIdx.x < world) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  const int i = blockIdx.x * TPB + threadIdx.x;
  const int o = i < n ? owner_of(xy[i].x, e) : -1;
  const unsigned peers = __match_any_sync(0xffffffffu, o);
  if (o >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_cnt[o], __popc(peers));
  __syncthreads();
  if (threadIdx.x < world) counts[(int64_t)threadIdx.x * n_cta + blockIdx.x] = s_cnt[threadIdx.x];  // strip-major
}

__global__ void __launch_bounds__(TPB)
partition_place_kernel(const double2* __restrict__ xy, const int32_t* __restrict__ type, const int32_t* __restrict__ gid,
                       int n, strip_edges e, int n_cta, const int32_t* __restrict__ base, pg_halo_rec* __restrict__ out,
                       int32_t* __restrict__ totals) {
  __shared__ int s_warp[TPB / 32][MAX_STRIPS];
  const int world = e.n_inner + 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int q = threadIdx.x; q < (TPB / 32) * MAX_STRIPS; q += TPB) (&s_warp[0][0])[q] = 0;
  __syncthreads();
  const int i = blockIdx.x * TPB + threadIdx.x;
  double2 p = make_double2(0, 0);
  int o = -1;
  if (i < n) { p = xy[i]; o = owner_of(p.x, e); }
  const unsigned peers = __match_any_sync(0xffffffffu, o);
  const int rank_in_warp = __popc(peers & ((1u << lane) - 1u));
  if (o >= 0 && lane == __ffs(peers) - 1) s_warp[warp][o] = __popc(peers);
  __syncthreads();
  if (o >= 0) {
    int before = 0;
    for (int w = 0; w < warp; ++w) before += s_warp[w][o];
    pg_halo_rec r;
    r.x = p.x; r.y = p.y; r.gid = gid ? gid[i] : i; r.type = type ? type[i] : 0;
    out[base[(int64_t)o * n_cta + blockIdx.x] + before + rank_in_warp] = r;   // input order kept inside every strip
  }
  if (blockIdx.x == 0 && threadIdx.x < world)
    totals[threadIdx.x] = base[(int64_t)(threadIdx.x + 1) * n_cta] - base[(int64_t)threadIdx.x * n_cta];
}

// ---- compact staging format of contour vertices: int16 half-pixels -> float32 pixels.
// skimage.measure.find_contours(mask, 0.5) (aggregated_hovernet_run.py:185) puts every vertex on the half-pixel
// lattice of its tile, so 2 * coordinate is a small integer: a table staged as int16 pairs carries the polygons in 4
// bytes per vertex instead of 8 (float32) or 16 (float64) over the host link, and widening is exact (x = 0.5 * q).
__global__ void __launch_bounds__(TPB)
widen_halfpx_kernel(const int16_t* __restrict__ in, float* __restrict__ out, int64_t n_values) {
  const int64_t i8 = ((int64_t)blockIdx.x * TPB + threadIdx.x) * 8;
  if (i8 + 8 <= n_values) {
    const int4 q = *reinterpret_cast<const int4*>(in + i8);
    const int w[4] = {q.x, q.y, q.z, q.w};
    float f[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      f[2 * k] = 0.5f * (float)(int16_t)(w[k] & 0xffff);
      f[2 * k + 1] = 0.5f * (float)(int16_t)((unsigned)w[k] >> 16);
    }
    float4* o = reinterpret_cast<float4*>(out + i8);
    o[0] = make_float4(f[0], f[1], f[2], f[3]);
    o[1] = make_float4(f[4], f[5], f[6], f[7]);
  } else {
    for (int64_t i = i8; i < n_values; ++i) out[i] = 0.5f * (float)in[i];
  }
}

// ---- K9: the halo exchange ---------------------------------------------------------------------------------------
// A rank selects its points near the strip edges into 24-byte records; the receiver appends the records of each x-range
// behind its owned points. Two transports share the select and the append:
//   NCCL:        pack into a local buffer -> all-gather (sharding.py) -> unpack the flat gathered array, skipping this
//                rank's own window.
//   peer memory: every rank owns a receive slab [world][cap] of records followed by [world] int32 counts, mapped into
//                all ranks (symmetric memory). The select kernel of rank r stores each record straight into slot [r][o]
//                of every peer's slab (P2P stores through NVSwitch); a one-warp kernel then publishes the count. No
//                staging buffer, no padded payload, no collective library call, and no host read to size anything -
//                the receiver's unpack walks world x cap slots and takes the first count[src] of every source.

// Warp-aggregated append, one atomic per warp: the lanes with `take` get consecutive slots of the list counted by
// *count. Returns the lane's slot, -1 without `take`. Every lane of the warp calls it.
__device__ __forceinline__ int warp_append(bool take, int32_t* count) {
  const unsigned m = __ballot_sync(0xffffffffu, take);
  if (m == 0) return -1;
  const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(count, __popc(m));
  base = __shfl_sync(0xffffffffu, base, leader);
  return take ? base + __popc(m & ((1u << lane) - 1u)) : -1;
}

// where a selected record goes (slot o < cap)
struct local_dst {     // pg_halo_pack: a buffer of cap records
  pg_halo_rec* out;
  int cap;
  __device__ void store(int o, const pg_halo_rec& r) const { out[o] = r; }
};
struct peer_dst {      // pg_halo_push: slot [rank][o] of every peer's slab
  const unsigned long long* peer_ptrs;   // read through __ldg: nvcc ignores __restrict__ on a struct member, and without
  int world, rank, cap;                  // it every peer store would be assumed to alias the table
  __device__ void store(int o, const pg_halo_rec& r) const {
    PG_ASSERT(o >= 0 && o < cap && rank >= 0 && rank < world);
    for (int q = 0; q < world; ++q)
      if (q != rank) reinterpret_cast<pg_halo_rec*>(__ldg(&peer_ptrs[q]))[(size_t)rank * cap + o] = r;
  }
};

// the points with x < lo_edge or x >= hi_edge (never a NaN x); *count counts all of them, slots past dst.cap raise the
// overflow flag. Profiled as halo_pack_kernel / halo_push_kernel.
template <class Dst>
__global__ void __launch_bounds__(TPB)
halo_select_kernel(const double2* __restrict__ xy, const int32_t* __restrict__ type, const int32_t* __restrict__ gid,
                   int n, double lo_edge, double hi_edge, Dst dst, int32_t* count, int32_t* overflow) {
  const int i = blockIdx.x * TPB + threadIdx.x;
  bool take = false;
  double2 p = make_double2(0, 0);
  if (i < n) { p = xy[i]; take = p.x < lo_edge || p.x >= hi_edge; }
  const int o = warp_append(take, count);
  if (o < 0) return;
  if (o >= dst.cap) { atomicExch(overflow, 1); return; }
  pg_halo_rec r;
  r.x = p.x; r.y = p.y; r.gid = gid ? gid[i] : i; r.type = type ? type[i] : 0;
  dst.store(o, r);
}

__global__ void halo_push_counts_kernel(const unsigned long long* __restrict__ peer_ptrs, int world, int rank, int cap,
                                        const int32_t* __restrict__ count) {
  const int q = threadIdx.x;
  if (q >= world || q == rank) return;
  int32_t* counts = reinterpret_cast<int32_t*>(reinterpret_cast<char*>(peer_ptrs[q]) + (size_t)world * cap * sizeof(pg_halo_rec));
  counts[rank] = *count;                  // unclamped: a receiver that sees more than cap raises its overflow flag too
  __threadfence_system();
}

// has(s): whether slot s of an unpack's record array holds a record. slab_src::has also raises the overflow flag
// (once per source) when a source's published count exceeds cap.
struct gathered_src {  // pg_halo_unpack_multi: the flat gathered records; [skip_begin, skip_end) are this rank's own
  using index = int;
  int n_recs, skip_begin, skip_end;
  __device__ bool has(int s, int32_t*) const { return s < n_recs && !(s >= skip_begin && s < skip_end); }
};
struct slab_src {      // pg_halo_unpack_slab: slot s = entry s % cap of source s / cap, valid below that source's count
  using index = int64_t;       // world x cap may pass 2^31
  const int32_t* src_counts;   // [world], behind the world x cap records
  int world, rank, cap;
  __device__ bool has(int64_t s, int32_t* overflow) const {
    if (s >= (int64_t)world * cap) return false;
    const int src = (int)(s / cap), idx = (int)(s - (int64_t)src * cap);
    const int cnt = src != rank ? __ldg(&src_counts[src]) : 0;
    if (idx == 0 && cnt > cap) atomicExch(overflow, 1);
    return idx < min(cnt, cap);
  }
};

// appends the records with x in [x_lo, x_hi) (never a NaN x); the first free slot is n_base + the counts of the
// ranges before this one. Profiled as halo_unpack_range_kernel / halo_unpack_slab_kernel.
template <class Src>
__global__ void __launch_bounds__(TPB)
halo_unpack_kernel(const pg_halo_rec* __restrict__ recs, Src src, double x_lo, double x_hi, double2* __restrict__ xy,
                   int32_t* __restrict__ type, int32_t* __restrict__ gid, int n_base, int capacity, int32_t* counts,
                   int range, int32_t* overflow) {
  const typename Src::index s = (typename Src::index)blockIdx.x * TPB + threadIdx.x;
  int first = n_base;
  for (int q = 0; q < range; ++q) first += counts[q];
  bool take = false;
  pg_halo_rec r;
  r.x = r.y = 0; r.gid = r.type = 0;
  if (src.has(s, overflow)) {
    r = recs[s];
    take = r.x >= x_lo && r.x < x_hi;
  }
  const int at = warp_append(take, &counts[range]);
  if (at < 0) return;
  const int o = first + at;
  PG_ASSERT(o >= n_base);
  if (o < capacity) {
    xy[o] = make_double2(r.x, r.y);
    if (type) type[o] = r.type;
    if (gid) gid[o] = r.gid;
  } else {
    atomicExch(overflow, 1);
  }
}

// clears counts_out [n_ranges], then one launch per non-empty range over the `slots` records of recs
template <class Src>
int unpack_ranges(pg_handle* h, cudaStream_t s, const char* name, const pg_halo_rec* recs, Src src, int64_t slots,
                  int32_t n_ranges, const double* ranges, double* xy, int32_t* type, int32_t* gid, int32_t n_base,
                  int32_t capacity, int32_t* counts_out) {
  PG_CUDA(h, cudaMemsetAsync(counts_out, 0, (size_t)n_ranges * sizeof(int32_t), s));
  if (slots == 0) return PG_OK;
  int32_t* ovf = (int32_t*)((char*)h->misc.p + PG_MISC_OVERFLOW);
  for (int r = 0; r < n_ranges; ++r) {
    if (!(ranges[2 * r + 1] > ranges[2 * r])) continue;  // empty range
    PG_LAUNCH(h, s, name, halo_unpack_kernel<<<pg_div_up(slots, TPB), TPB, 0, s>>>(
        recs, src, ranges[2 * r], ranges[2 * r + 1], (double2*)xy, type, gid, n_base, capacity, counts_out, r, ovf));
    PG_LAUNCH_CHECK(h);
  }
  return PG_OK;
}

__global__ void __launch_bounds__(TPB)
gid_maps_kernel(const int32_t* __restrict__ gid, const int32_t* __restrict__ type, int n, int n_rows, int n_ids,
                int32_t* __restrict__ id_map, int32_t* __restrict__ type_by_gid) {
  const int i = blockIdx.x * TPB + threadIdx.x;
  if (i >= n) return;
  const int g = gid[i];
  if (g < 0 || g >= n_ids) return;
  if (i < n_rows && id_map) id_map[g] = i;
  if (type_by_gid) type_by_gid[g] = type ? type[i] : 0;
}

// int32 counts -> uint8 / uint16 (what crosses PCIe when the caller asks for narrow counts); values that do not fit
// raise the handle's overflow flag (pg_check_overflow) and are stored saturated
template <typename T>
__global__ void __launch_bounds__(TPB)
narrow_counts_kernel(const int4* __restrict__ src, int64_t n4, int64_t n, T* __restrict__ dst, int32_t* overflow) {
  const int64_t i = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (i >= n4) return;
  constexpr int LIM = sizeof(T) == 1 ? 255 : 65535;
  int v[4];
  if (4 * i + 4 <= n) { const int4 q = src[i]; v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
  else { const int32_t* s1 = reinterpret_cast<const int32_t*>(src); for (int t = 0; t < 4; ++t) v[t] = 4 * i + t < n ? s1[4 * i + t] : 0; }
  bool bad = false;
#pragma unroll
  for (int t = 0; t < 4; ++t) { bad |= v[t] < 0 || v[t] > LIM; v[t] = min(max(v[t], 0), LIM); }
  if (bad) atomicExch(overflow, 1);
  if (4 * i + 4 <= n) {
    if (sizeof(T) == 1) reinterpret_cast<uint32_t*>(dst)[i] = (uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) | ((uint32_t)v[3] << 24);
    else reinterpret_cast<uint2*>(dst)[i] = make_uint2((uint32_t)v[0] | ((uint32_t)v[1] << 16), (uint32_t)v[2] | ((uint32_t)v[3] << 16));
  } else {
    for (int t = 0; t < 4; ++t) if (4 * i + t < n) dst[4 * i + t] = (T)v[t];
  }
}

}  // namespace

extern "C" {

int pg_narrow_counts(pg_handle* h, const int32_t* src, int64_t n, void* dst, int32_t bits, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && (bits == 8 || bits == 16) && (n == 0 || (src && dst)), "pg_narrow_counts: bits must be 8 or 16");
  PG_REQUIRE(h, ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 7) == 0, "pg_narrow_counts: src must be 16-byte, dst 8-byte aligned");
  if (n == 0) return PG_OK;
  const int64_t n4 = (n + 3) / 4;
  int32_t* ovf = (int32_t*)((char*)h->misc.p + PG_MISC_OVERFLOW);
  if (bits == 8) PG_LAUNCH(h, s, "narrow_counts_kernel", narrow_counts_kernel<uint8_t><<<pg_div_up(n4, TPB), TPB, 0, s>>>((const int4*)src, n4, n, (uint8_t*)dst, ovf));
  else PG_LAUNCH(h, s, "narrow_counts_kernel", narrow_counts_kernel<uint16_t><<<pg_div_up(n4, TPB), TPB, 0, s>>>((const int4*)src, n4, n, (uint16_t*)dst, ovf));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_strip_partition(pg_handle* h, int32_t n, const double* xy, const int32_t* type, const int32_t* gid,
                       int32_t n_strips, const double* inner_edges, pg_halo_rec* out, int32_t* totals, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && n_strips >= 1 && n_strips <= MAX_STRIPS && totals, "pg_strip_partition: need 1 <= n_strips <= %d", MAX_STRIPS);
  PG_REQUIRE(h, n == 0 || (xy && out), "pg_strip_partition: xy / out is NULL");
  PG_REQUIRE(h, n_strips == 1 || inner_edges, "pg_strip_partition: inner_edges is NULL");
  PG_REQUIRE(h, ((uintptr_t)xy & 15) == 0 && ((uintptr_t)out & 7) == 0, "pg_strip_partition: xy must be 16-byte aligned");
  strip_edges e;
  e.n_inner = n_strips - 1;
  for (int q = 0; q < e.n_inner; ++q) {
    e.inner[q] = inner_edges[q];
    PG_REQUIRE(h, q == 0 || e.inner[q] >= e.inner[q - 1], "pg_strip_partition: inner_edges must ascend");
  }
  if (n == 0) {
    PG_CUDA(h, cudaMemsetAsync(totals, 0, (size_t)n_strips * sizeof(int32_t), s));
    return PG_OK;
  }
  const int n_cta = pg_div_up(n, TPB);
  const int64_t cells = (int64_t)n_strips * n_cta;
  int rc;
  // counts [n_strips][n_cta] (16-byte aligned) and their exclusive scan [cells + 1], both in one scratch buffer
  const size_t cnt_bytes = ((size_t)cells * sizeof(int32_t) + 15) & ~(size_t)15;
  if ((rc = pg_reserve(h, h->cell_of, cnt_bytes + ((size_t)cells + 8) * sizeof(int32_t)))) return rc;
  int32_t* counts = (int32_t*)h->cell_of.p;
  int32_t* base = (int32_t*)((char*)h->cell_of.p + cnt_bytes);
  PG_LAUNCH(h, s, "partition_count_kernel", partition_count_kernel<<<n_cta, TPB, 0, s>>>((const double2*)xy, n, e, n_cta, counts));
  PG_LAUNCH_CHECK(h);
  if ((rc = pg_scan_i32(h, counts, base, (int32_t)cells, s))) return rc;
  PG_LAUNCH(h, s, "partition_place_kernel", partition_place_kernel<<<n_cta, TPB, 0, s>>>((const double2*)xy, type, gid, n, e, n_cta, base, out, totals));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_halo_pack(pg_handle* h, int32_t n, const double* xy, const int32_t* type, const int32_t* gid,
                 double lo_edge, double hi_edge, pg_halo_rec* out, int32_t capacity, int32_t* count_out,
                 pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && capacity >= 0 && count_out && (capacity == 0 || out), "pg_halo_pack: bad argument");
  PG_CUDA(h, cudaMemsetAsync(count_out, 0, sizeof(int32_t), s));
  if (n > 0) {
    PG_LAUNCH(h, s, "halo_pack_kernel", halo_select_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>(
        (const double2*)xy, type, gid, n, lo_edge, hi_edge, local_dst{out, capacity}, count_out,
        (int32_t*)((char*)h->misc.p + PG_MISC_OVERFLOW)));
    PG_LAUNCH_CHECK(h);
  }
  return PG_OK;
}

int pg_halo_unpack_multi(pg_handle* h, const pg_halo_rec* recs, int32_t n_recs, int32_t skip_begin, int32_t skip_end,
                         int32_t n_ranges, const double* ranges, double* xy, int32_t* type, int32_t* gid, int32_t n_base,
                         int32_t capacity, int32_t* counts_out, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n_recs >= 0 && n_base >= 0 && capacity >= n_base && n_ranges >= 1 && n_ranges <= 8 && ranges && counts_out && xy,
             "pg_halo_unpack_multi: bad argument");
  return unpack_ranges(h, s, "halo_unpack_range_kernel", recs, gathered_src{n_recs, skip_begin, skip_end}, n_recs, n_ranges,
                       ranges, xy, type, gid, n_base, capacity, counts_out);
}

int pg_widen_halfpx(pg_handle* h, int64_t n_values, const int16_t* in, float* out, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n_values >= 0 && (n_values == 0 || (in && out)), "pg_widen_halfpx: bad argument");
  PG_REQUIRE(h, (((uintptr_t)in | (uintptr_t)out) & 15) == 0, "pg_widen_halfpx: in / out must be 16-byte aligned");
  if (n_values == 0) return PG_OK;
  PG_LAUNCH(h, s, "widen_halfpx_kernel", widen_halfpx_kernel<<<pg_div_up(pg_div_up(n_values, 8), TPB), TPB, 0, s>>>(in, out, n_values));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_halo_push(pg_handle* h, int32_t n, const double* xy, const int32_t* type, const int32_t* gid, double lo_edge,
                 double hi_edge, const uint64_t* peer_ptrs_dev, int32_t world, int32_t rank, int32_t cap, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && world >= 1 && world <= 1024 && rank >= 0 && rank < world && cap >= 1 && peer_ptrs_dev,
             "pg_halo_push: bad argument");
  PG_REQUIRE(h, (int64_t)world * cap < 0x7fffffff, "pg_halo_push: world x cap must stay below 2^31 slots");
  int32_t* count = (int32_t*)((char*)h->misc.p + PG_MISC_HALOCNT);
  PG_CUDA(h, cudaMemsetAsync(count, 0, sizeof(int32_t), s));
  if (n > 0) {
    PG_LAUNCH(h, s, "halo_push_kernel", halo_select_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>(
        (const double2*)xy, type, gid, n, lo_edge, hi_edge, peer_dst{(const unsigned long long*)peer_ptrs_dev, world, rank, cap},
        count, (int32_t*)((char*)h->misc.p + PG_MISC_OVERFLOW)));
    PG_LAUNCH_CHECK(h);
  }
  PG_LAUNCH(h, s, "halo_push_counts_kernel", halo_push_counts_kernel<<<1, 1024, 0, s>>>((const unsigned long long*)peer_ptrs_dev, world, rank, cap, count));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_halo_unpack_slab(pg_handle* h, const void* slab, int32_t world, int32_t rank, int32_t cap, int32_t n_ranges,
                        const double* ranges, double* xy, int32_t* type, int32_t* gid, int32_t n_base, int32_t capacity,
                        int32_t* counts_out, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, slab && world >= 1 && rank >= 0 && rank < world && cap >= 1 && n_base >= 0 && capacity >= n_base &&
                    n_ranges >= 1 && n_ranges <= 8 && ranges && counts_out && xy, "pg_halo_unpack_slab: bad argument");
  const pg_halo_rec* recs = (const pg_halo_rec*)slab;
  const int64_t slots = (int64_t)world * cap;
  return unpack_ranges(h, s, "halo_unpack_slab_kernel", recs, slab_src{(const int32_t*)(recs + slots), world, rank, cap}, slots,
                       n_ranges, ranges, xy, type, gid, n_base, capacity, counts_out);
}

int pg_gid_maps(pg_handle* h, int32_t n, int32_t n_rows, const int32_t* gid, const int32_t* type, int32_t n_ids,
                int32_t* id_map, int32_t* type_by_gid, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && n_rows >= 0 && n_rows <= n && n_ids >= 0 && (n == 0 || gid), "pg_gid_maps: bad argument");
  if (id_map) PG_CUDA(h, cudaMemsetAsync(id_map, 0xff, (size_t)n_ids * sizeof(int32_t), s));   // -1: the id has no row here
  if (type_by_gid) PG_CUDA(h, cudaMemsetAsync(type_by_gid, 0, (size_t)n_ids * sizeof(int32_t), s));
  if (n == 0) return PG_OK;
  PG_LAUNCH(h, s, "gid_maps_kernel", gid_maps_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>(gid, type, n, n_rows, n_ids, id_map, type_by_gid));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
