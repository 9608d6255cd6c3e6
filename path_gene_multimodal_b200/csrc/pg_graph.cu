// K7 undirected union of directed kNN lists, `edges` (i<j) extraction from a symmetric CSR, and the
// stand-alone K8 (neighbour-type composition + degree statistics over any CSR).
// Reference: /root/reference/hovernet_tile_inference.ipynb:1865-1894 (nx.Graph union, weight = min),
// :2969-2975 (i<j edge list); composition / degree per SURVEY A.5 (README.md:127,136).
#include <algorithm>
#include <cstring>
#include "pg_degree.cuh"
#include "pg_query.cuh"

namespace {

constexpr int TPB = 256;
constexpr uint8_t RECIP_INVALID = 255, RECIP_NONE = 254;

// The union is built count -> scan -> push -> rank, one thread per ROW in the first and third step (a row of
// k ids is one or two sectors: vector loads, k independent reads of the neighbours' rows in flight), one lane per
// OUTPUT ENTRY in the last:
//   mark  row i reads the row of each neighbour j and records where i sits in it (the slot, or NONE); every
//         reverse-only edge i->j bumps row_count[j], the row's own valid entries bump row_count[i].
//   scan  row_count -> und_row_ptr (the scan clears row_count behind itself: it is the push cursor next).
//   push  row i writes its own entries (weight = min over both directions) at the front of its range and pushes
//         each reverse-only edge to the BACK of row j's range (cursor[j] counts arrivals).
//   rank  a warp owns 32 consecutive rows = one contiguous range of the staged entries; lane p of that range
//         finds its row by shuffle search, counts the row's smaller ids and writes the entry to its place:
//         rows leave ascending by column whatever order the pushes arrived in, all output traffic coalesced.
// Lists hold ids in "column space" (global ids when the rows are a strip + halo of a larger slide):
// row_id[i] is the id of row i, id_map[id] the row of an id (-1 / >= n: no row here). NULL = identity.
template <int K>
__device__ __forceinline__ void load_row_i32(const int32_t* __restrict__ p, int k, int (&v)[K ? K : 1]) {
  if (K == 0) return;
  if ((K & 3) == 0) {
#pragma unroll
    for (int q = 0; q < K / 4; ++q) {
      const int4 t = reinterpret_cast<const int4*>(p)[q];
      v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int q = 0; q < K; ++q) v[q] = p[q];
  }
}

// slot of `id` in the k-list at `row` (NONE if absent)
template <int K>
__device__ __forceinline__ int find_slot(const int32_t* __restrict__ row, int k, int id) {
  int found = RECIP_NONE;
  if (K != 0) {
    int v[K ? K : 1];
    load_row_i32<K>(row, k, v);
#pragma unroll
    for (int s = K - 1; s >= 0; --s) found = v[s] == id ? s : found;
  } else {
    for (int s = 0; s < k; ++s)
      if (row[s] == id) { found = s; break; }
  }
  return found;
}

// K = compile-time k (rows 16-byte aligned when k % 4 == 0) or 0 = any k
template <int K>
__global__ void __launch_bounds__(TPB)
sym_mark_kernel(const int32_t* __restrict__ knn_idx, int n, int k_rt, const int32_t* __restrict__ row_id,
                const int32_t* __restrict__ id_map, int n_ids, uint8_t* __restrict__ recip,
                int32_t* __restrict__ row_count, int32_t* __restrict__ up_count) {
  // up_count (optional): entries of the final row with column > the row's id, i.e. its share of the i<j edge list
  const int i = blockIdx.x * TPB + threadIdx.x;
  if (i >= n) return;
  const int k = K ? K : k_rt;
  const int my_id = row_id ? row_id[i] : i;
  const int32_t* mine = knn_idx + (int64_t)i * k;
  uint8_t* rc_out = recip + (int64_t)i * k;
  int own = 0, own_up = 0;
  if (K != 0) {
    int ids[K ? K : 1];
    load_row_i32<K>(mine, k, ids);
    int rc[K ? K : 1];
#pragma unroll
    for (int s = 0; s < K; ++s) {
      const int jid = ids[s];
      int r = RECIP_INVALID;
      if (!(jid < 0 || jid == my_id || (id_map && jid >= n_ids) || (!id_map && jid >= n))) {
        const int j = id_map ? id_map[jid] : jid;
        r = RECIP_NONE;
        if (j >= 0 && j < n) {  // else: the neighbour has no row here, own entry only
          r = find_slot<K>(knn_idx + (int64_t)j * k, k, my_id);
          if (r == RECIP_NONE) {
            atomicAdd(&row_count[j], 1);
            if (up_count && my_id > jid) atomicAdd(&up_count[j], 1);
          }
        }
        ++own;
        own_up += jid > my_id;
      }
      rc[s] = r;
    }
    if ((K & 3) == 0) {
#pragma unroll
      for (int q = 0; q < K / 4; ++q)
        reinterpret_cast<uint32_t*>(rc_out)[q] = (uint32_t)rc[4 * q] | ((uint32_t)rc[4 * q + 1] << 8) |
                                                 ((uint32_t)rc[4 * q + 2] << 16) | ((uint32_t)rc[4 * q + 3] << 24);
    } else {
#pragma unroll
      for (int s = 0; s < K; ++s) rc_out[s] = (uint8_t)rc[s];
    }
  } else {
    for (int s = 0; s < k; ++s) {
      const int jid = mine[s];
      int r = RECIP_INVALID;
      if (!(jid < 0 || jid == my_id || (id_map && jid >= n_ids) || (!id_map && jid >= n))) {
        const int j = id_map ? id_map[jid] : jid;
        r = RECIP_NONE;
        if (j >= 0 && j < n) {
          r = find_slot<0>(knn_idx + (int64_t)j * k, k, my_id);
          if (r == RECIP_NONE) {
            atomicAdd(&row_count[j], 1);
            if (up_count && my_id > jid) atomicAdd(&up_count[j], 1);
          }
        }
        ++own;
        own_up += jid > my_id;
      }
      rc_out[s] = (uint8_t)r;
    }
  }
  if (own) atomicAdd(&row_count[i], own);
  if (up_count && own_up) atomicAdd(&up_count[i], own_up);
}

// a row of K items of T as 16-byte vector loads when the row is a whole number of them (the caller checks the
// base alignment), scalar loads otherwise
template <class T, int K>
__device__ __forceinline__ void load_row(const T* __restrict__ p, T (&v)[K]) {
  if ((K * sizeof(T)) % 16 == 0) {
    constexpr int PER = 16 / sizeof(T);
#pragma unroll
    for (int q = 0; q < (int)(K * sizeof(T) / 16); ++q) {
      const uint4 t = reinterpret_cast<const uint4*>(p)[q];
      T tmp[PER];
      memcpy(tmp, &t, 16);
#pragma unroll
      for (int e = 0; e < PER; ++e) v[q * PER + e] = tmp[e];
    }
  } else {
#pragma unroll
    for (int q = 0; q < K; ++q) v[q] = p[q];
  }
}

// push: only the reverse-only edges travel (to the BACK of the target row's range in the staging arrays); a
// row's own entries are read where they are by the rank pass
template <class DT>
__device__ __forceinline__ void push_entry(int s_rc, int jid, DT w, int my_id, int n,
                                           const int32_t* __restrict__ id_map, const int32_t* __restrict__ row_ptr,
                                           int32_t* __restrict__ cursor, int32_t* __restrict__ tmp_col,
                                           DT* __restrict__ tmp_w) {
  if (s_rc != RECIP_NONE) return;
  const int j = id_map ? id_map[jid] : jid;
  if (j < 0 || j >= n) return;
  const int64_t r = (int64_t)row_ptr[j + 1] - 1 - atomicAdd(&cursor[j], 1);
  tmp_col[r] = my_id;
  tmp_w[r] = w;
}

// K = compile-time k with 16-byte aligned rows, or 0 = any k
template <class DT, int K>
__global__ void __launch_bounds__(TPB)
sym_push_kernel(const int32_t* __restrict__ knn_idx, const DT* __restrict__ dist, int n, int k_rt,
                const int32_t* __restrict__ row_id, const int32_t* __restrict__ id_map,
                const uint8_t* __restrict__ recip, const int32_t* __restrict__ row_ptr,
                int32_t* __restrict__ cursor, int32_t* __restrict__ tmp_col, DT* __restrict__ tmp_w) {
  const int i = blockIdx.x * TPB + threadIdx.x;
  if (i >= n) return;
  const int k = K ? K : k_rt;
  const int my_id = row_id ? row_id[i] : i;
  if (K != 0) {
    constexpr int KK = K ? K : 4;
    uint32_t rcw[KK / 4];
    bool any = false;
#pragma unroll
    for (int q = 0; q < KK / 4; ++q) {
      rcw[q] = reinterpret_cast<const uint32_t*>(recip + (int64_t)i * KK)[q];
#pragma unroll
      for (int e = 0; e < 4; ++e) any |= ((rcw[q] >> (8 * e)) & 0xffu) == RECIP_NONE;
    }
    if (!any) return;
    int ids[KK];
    DT ds[KK];
    load_row<int, KK>(knn_idx + (int64_t)i * KK, ids);
    load_row<DT, KK>(dist + (int64_t)i * KK, ds);
#pragma unroll
    for (int s = 0; s < KK; ++s)
      push_entry<DT>((int)((rcw[s >> 2] >> ((s & 3) * 8)) & 0xffu), ids[s], ds[s], my_id, n, id_map, row_ptr, cursor,
                     tmp_col, tmp_w);
  } else {
    for (int s = 0; s < k; ++s)
      push_entry<DT>(recip[(int64_t)i * k + s], knn_idx[(int64_t)i * k + s], dist[(int64_t)i * k + s], my_id, n, id_map,
                     row_ptr, cursor, tmp_col, tmp_w);
  }
}

// rank: a warp owns 32 consecutive rows = one contiguous range of the output. Row r's range is its own valid
// entries (read from its k-list, weight = min over both directions, ipynb:1888-1892) followed by the arrivals
// staged at the back; every lane takes one entry of the range, counts the entries of the row that sort before
// it and writes it to its place.
// optional fused outputs of the rank pass (all NULL: plain symmetrisation)
struct rank_extra {
  const int32_t* row_id;   // id of each row (NULL = identity), for the edge list
  const int32_t* up_ptr;   // [n+1] exclusive scan of the rows' upper-entry counts (NULL: no edge list)
  long long* edges; double* ew64; float* ew32;
  const int32_t* type;     // type by column id
  int n_types;
  int32_t* nbr_count;      // [n][n_types]
  int32_t* degree;
  pg_degree_out deg;
  bool sym_dist;           // the lists' distances are symmetric bit for bit: no reverse read for the min
};

template <class DT, int K>  // K = compile-time k with 16-byte aligned rows (vector loads), or 0 = any k
__global__ void __launch_bounds__(TPB)
sym_rank_kernel(const int32_t* __restrict__ knn_idx, const DT* __restrict__ dist, int n, int k_rt,
                const int32_t* __restrict__ id_map, const uint8_t* __restrict__ recip,
                const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ tmp_col,
                const DT* __restrict__ tmp_w, int32_t* __restrict__ col, double* __restrict__ w64,
                float* __restrict__ w32, rank_extra x) {
  using DG = pg_degree_cta<TPB>;
  __shared__ int s_cnt[TPB / 32][32 * PG_MAX_TYPES];
  __shared__ DG::smem_t s_deg;
  if (DG::on(x.deg)) {  // CTA-wide state: before any warp may leave
    DG::arm(s_deg, x.deg);
    __syncthreads();
  }
  constexpr int KK = K ? K : 4;
  const int k = K ? K : k_rt;
  const int lane = threadIdx.x & 31;
  const int r0 = ((blockIdx.x * TPB + threadIdx.x) >> 5) << 5;
  const bool warp_on = r0 < n;  // warp-uniform (no early exit: the statistics below need every warp at the barriers)
  const int rp = row_ptr[min(r0 + lane, n)];
  const int begin = __shfl_sync(0xffffffffu, rp, 0);
  const int end = warp_on ? row_ptr[min(r0 + 32, n)] : begin;
  const int rp_next = __shfl_down_sync(0xffffffffu, rp, 1);
  const int my_cnt = (lane == 31 ? end : rp_next) - rp;
  // fused extras: my row's id, its slice of the i<j edge list, its type counters
  const int my_rid = (r0 + lane < n) ? (x.row_id ? x.row_id[r0 + lane] : r0 + lane) : 0;
  int my_up = 0, my_upn = 0;
  if (x.up_ptr) { my_up = x.up_ptr[min(r0 + lane, n)]; my_upn = x.up_ptr[min(r0 + lane + 1, n)] - my_up; }
  int* wcnt = s_cnt[threadIdx.x >> 5];
  if (x.nbr_count)
    for (int t = 0; t < x.n_types; ++t) wcnt[lane * x.n_types + t] = 0;
  __syncwarp();
  int my_own = 0;  // valid entries of the lane's row
  if (r0 + lane < n) {
    if (K != 0) {
#pragma unroll
      for (int q = 0; q < KK / 4; ++q) {
        const uint32_t wrd = reinterpret_cast<const uint32_t*>(recip + (int64_t)(r0 + lane) * KK)[q];
#pragma unroll
        for (int e = 0; e < 4; ++e) my_own += ((wrd >> (8 * e)) & 0xffu) != RECIP_INVALID;
      }
    } else {
      for (int s = 0; s < k; ++s) my_own += recip[(int64_t)(r0 + lane) * k + s] != RECIP_INVALID;
    }
  }
  for (int p0 = begin; p0 < end; p0 += 32) {
    const int p = p0 + lane;
    int kk = 0;  // the last row of the 32 that starts at or before p (empty rows share their start with the next row)
#pragma unroll
    for (int step = 16; step > 0; step >>= 1) {
      const int v = __shfl_sync(0xffffffffu, rp, kk + step);
      if (v <= p) kk += step;
    }
    const int rcnt = __shfl_sync(0xffffffffu, my_cnt, kk);
    const int rbase = __shfl_sync(0xffffffffu, rp, kk);
    const int own = __shfl_sync(0xffffffffu, my_own, kk);
    const int rid = __shfl_sync(0xffffffffu, my_rid, kk);
    const int upb = __shfl_sync(0xffffffffu, my_up, kk), upn = __shfl_sync(0xffffffffu, my_upn, kk);
    if (p >= end) continue;
    const int64_t rowk = (int64_t)(r0 + kk) * k;
    const int me = p - rbase;  // position in the row's unsorted range: own entries by slot, then the arrivals
    int c;
    DT w;
    int my_slot = -1;
    int rank = 0;  // place = number of entries that sort before (id, position): any input yields a permutation
    if (K != 0 && own == k) {
      // the common case - every slot of the row is valid: the row's ids in registers (two / four 16-byte loads)
      int ids[KK];
      load_row<int, KK>(knn_idx + rowk, ids);
      if (me < own) {
        my_slot = me;
        c = 0;
#pragma unroll
        for (int s = 0; s < KK; ++s) c = s == me ? ids[s] : c;
        w = dist[rowk + me];
        if (!x.sym_dist) {  // weight = min over directions (ipynb:1888-1892); equal by construction for pg_knn lists
          const int rc = recip[rowk + me];
          if (rc != RECIP_NONE) {
            const int j = id_map ? id_map[c] : c;
            w = min(w, dist[(int64_t)j * k + rc]);
          }
        }
      } else {
        c = tmp_col[p];
        w = tmp_w[p];
      }
#pragma unroll
      for (int s = 0; s < KK; ++s) rank += (ids[s] < c || (ids[s] == c && (my_slot < 0 || s < my_slot))) ? 1 : 0;
    } else {
      if (me < own) {
        int s = me;
        if (own != k) {  // skip the invalid slots
          int seen = 0;
          for (s = 0; s < k; ++s)
            if (recip[rowk + s] != RECIP_INVALID && seen++ == me) break;
        }
        my_slot = s;
        c = knn_idx[rowk + s];
        w = dist[rowk + s];
        const int rc = recip[rowk + s];
        if (rc != RECIP_NONE && !x.sym_dist) {
          const int j = id_map ? id_map[c] : c;
          w = min(w, dist[(int64_t)j * k + rc]);
        }
      } else {
        c = tmp_col[p];
        w = tmp_w[p];
      }
      for (int s = 0; s < k; ++s) {
        const int cu = knn_idx[rowk + s];
        const bool valid = own == k || recip[rowk + s] != RECIP_INVALID;
        rank += (valid && (cu < c || (cu == c && (my_slot < 0 || s < my_slot)))) ? 1 : 0;
      }
    }
    for (int u = own; u < rcnt; ++u) {
      const int cu = tmp_col[rbase + u];
      rank += (cu < c || (cu == c && my_slot < 0 && u < me)) ? 1 : 0;
    }
    const int64_t dst = (int64_t)rbase + rank;
    col[dst] = c;
    if (w64) w64[dst] = (double)w;
    if (w32) w32[dst] = (float)w;
    if (x.up_ptr) {  // the row's last up_n sorted entries are its i<j edges (ipynb:1894 G.edges / :2969-2975)
      const int at = rank - (rcnt - upn);
      if (at >= 0) {
        const int64_t e = (int64_t)upb + at;
        if (x.edges) *reinterpret_cast<longlong2*>(x.edges + 2 * e) = make_longlong2(rid, c);
        if (x.ew64) x.ew64[e] = (double)w;
        if (x.ew32) x.ew32[e] = (float)w;
      }
    }
    if (x.nbr_count) {  // neighbour-type composition (README.md:127): one shared-memory counter per (row, type)
      const int ty = x.type[c];
      if (ty >= 1 && ty <= x.n_types) atomicAdd(&wcnt[kk * x.n_types + ty - 1], 1);
    }
  }
  __syncwarp();
  if (warp_on && x.nbr_count) {  // the warp's 32 rows x n_types counters are one contiguous range of nbr_count
    const int rows_here = min(32, n - r0);
    for (int i = lane; i < rows_here * x.n_types; i += 32) x.nbr_count[(int64_t)r0 * x.n_types + i] = wcnt[i];
  }
  if (x.degree && r0 + lane < n) x.degree[r0 + lane] = my_cnt;
  if (!DG::on(x.deg)) return;
  DG dg(s_deg, x.deg);
  dg.add(my_cnt, r0 + lane < n);
  dg.commit();
  __syncthreads();
  dg.finish(n);
}

// rows are ascending by column: entries above the row's own id start at the first col > id
__global__ void __launch_bounds__(TPB)
upper_count_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                   const int32_t* __restrict__ row_id, int n, int32_t* __restrict__ up_count) {
  const int i = blockIdx.x * TPB + threadIdx.x;
  if (i >= n) return;
  const int id = row_id ? row_id[i] : i;
  int lo = row_ptr[i], hi = row_ptr[i + 1];
  const int end = hi;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (col[mid] > id) hi = mid; else lo = mid + 1;
  }
  up_count[i] = end - lo;
}

// one warp per 32 consecutive rows = one contiguous range of the edge list, one lane per edge (coalesced
// 16-byte stores); the upper entries of a row are the last up_cnt entries of its (ascending) range
__global__ void __launch_bounds__(TPB)
upper_fill_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                  const double* __restrict__ w64, const float* __restrict__ w32,
                  const int32_t* __restrict__ row_id, const int32_t* __restrict__ up_ptr, int n,
                  long long* __restrict__ edges, double* __restrict__ ew64, float* __restrict__ ew32) {
  const int lane = threadIdx.x & 31;
  const int r0 = ((blockIdx.x * TPB + threadIdx.x) >> 5) << 5;
  if (r0 >= n) return;  // warp-uniform
  const int row = min(r0 + lane, n - 1);
  const int up = up_ptr[min(r0 + lane, n)];
  const int row_end = row_ptr[row + 1];
  const int id = row_id ? row_id[row] : row;
  const int begin = __shfl_sync(0xffffffffu, up, 0);
  const int end = up_ptr[min(r0 + 32, n)];
  const bool edges16 = ((uintptr_t)edges & 15) == 0;
  for (int p0 = begin; p0 < end; p0 += 32) {
    const int p = p0 + lane;
    int kk = 0;  // the last row of the 32 whose range starts at or before p
#pragma unroll
    for (int step = 16; step > 0; step >>= 1) {
      const int v = __shfl_sync(0xffffffffu, up, kk + step);
      if (v <= p && r0 + kk + step < n) kk += step;
    }
    const int ubase = __shfl_sync(0xffffffffu, up, kk);
    const int nxt = __shfl_sync(0xffffffffu, up, min(kk + 1, 31));
    const int unext = (kk == 31 || r0 + kk + 1 >= n) ? end : nxt;
    const int rend = __shfl_sync(0xffffffffu, row_end, kk);
    const int rid = __shfl_sync(0xffffffffu, id, kk);
    if (p >= end) continue;
    const int64_t src = (int64_t)rend - (unext - ubase) + (p - ubase);
    if (edges) {
      if (edges16) *reinterpret_cast<longlong2*>(edges + 2 * (int64_t)p) = make_longlong2(rid, col[src]);
      else { edges[2 * (int64_t)p] = rid; edges[2 * (int64_t)p + 1] = col[src]; }
    }
    if (ew64) ew64[p] = w64 ? w64[src] : (double)w32[src];
    if (ew32) ew32[p] = w32 ? w32[src] : (float)w64[src];
  }
}

// ---- K8 over a CSR ------------------------------------------------------------------------
template <int TMAX>
__global__ void __launch_bounds__(TPB)
compose_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
               const int32_t* __restrict__ type, int n, int n_types, int32_t* __restrict__ nbr_count,
               int32_t* __restrict__ degree, pg_degree_out dout) {
  using DG = pg_degree_cta<TPB>;
  __shared__ DG::smem_t s_deg;
  if (DG::on(dout)) {
    DG::arm(s_deg, dout);
    __syncthreads();
  }
  const int i = blockIdx.x * TPB + threadIdx.x;
  const bool valid = i < n;
  int deg = 0;
  if (valid) {
    const int b = row_ptr[i], e = row_ptr[i + 1];
    deg = e - b;
    if (nbr_count) {
      int tc[TMAX];
#pragma unroll
      for (int t = 0; t < TMAX; ++t) tc[t] = 0;
      for (int j = b; j < e; ++j) {
        const int ty = __ldg(&type[col[j]]);
#pragma unroll
        for (int t = 0; t < TMAX; ++t) tc[t] += (ty == t + 1);
      }
#pragma unroll
      for (int t = 0; t < TMAX; ++t)
        if (t < n_types) nbr_count[(int64_t)i * n_types + t] = tc[t];
    }
    if (degree) degree[i] = deg;
  }
  if (!DG::on(dout)) return;
  DG dg(s_deg, dout);
  dg.add(deg, valid);
  dg.commit();
  __syncthreads();
  dg.finish(n);
}

// ---- K11 graph statistics named by the reference (README.md:136 "degree, clustering, centrality"; SURVEY 8f-4)
// Local clustering coefficient over a symmetric CSR with ascending rows (what K6 / K7 emit): one lane per
// directed edge (i, j) of a warp's 32 consecutive rows counts |N(i) & N(j)| by merging the two sorted rows; the
// per-edge counts are added to tri2[i] (integer atomics: order-independent), which ends as twice the number of
// triangles through i; coeff = tri2 / (d (d - 1)), 0 for d < 2 - networkx.clustering's definition.
__global__ void __launch_bounds__(TPB)
clustering_count_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
                        int32_t* __restrict__ tri2) {
  const int lane = threadIdx.x & 31;
  const int r0 = ((blockIdx.x * TPB + threadIdx.x) >> 5) << 5;
  if (r0 >= n) return;  // warp-uniform
  const int rp = row_ptr[min(r0 + lane, n)];
  const int begin = __shfl_sync(0xffffffffu, rp, 0);
  const int end = row_ptr[min(r0 + 32, n)];
  const int rp_next = __shfl_down_sync(0xffffffffu, rp, 1);
  const int my_cnt = (lane == 31 ? end : rp_next) - rp;
  for (int p0 = begin; p0 < end; p0 += 32) {
    const int p = p0 + lane;
    int kk = 0;
#pragma unroll
    for (int step = 16; step > 0; step >>= 1) {
      const int v = __shfl_sync(0xffffffffu, rp, kk + step);
      if (v <= p) kk += step;
    }
    const int rcnt = __shfl_sync(0xffffffffu, my_cnt, kk);
    const int rbase = __shfl_sync(0xffffffffu, rp, kk);
    if (p >= end) continue;
    const int i = r0 + kk, j = col[p];
    if (j == i || j < 0 || j >= n) continue;  // self loops / foreign ids close no triangle here
    int a = rbase, a_end = rbase + rcnt, b = row_ptr[j], b_end = row_ptr[j + 1], common = 0;
    while (a < a_end && b < b_end) {
      const int ca = col[a], cb = col[b];
      common += (ca == cb && ca != i && ca != j) ? 1 : 0;
      a += ca <= cb;
      b += cb <= ca;
    }
    if (common) atomicAdd(&tri2[i], common);
  }
}

__global__ void __launch_bounds__(TPB)
clustering_finish_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ tri2, int n,
                         int32_t* __restrict__ triangles, double* __restrict__ coeff) {
  const int i = blockIdx.x * TPB + threadIdx.x;
  if (i >= n) return;
  const int d = row_ptr[i + 1] - row_ptr[i], t2 = tri2[i];
  if (triangles) triangles[i] = t2 >> 1;
  if (coeff) coeff[i] = d < 2 ? 0.0 : (double)t2 / ((double)d * (double)(d - 1));
}

// type-type interaction counts: inter[a][b] = number of (directed) edges from a node of type a+1 to a node of
// type b+1 = sum of nbr_count rows grouped by the row's own type ("cell-cell interaction patterns", README.md:133)
__global__ void __launch_bounds__(TPB)
interactions_kernel(const int32_t* __restrict__ type, const int32_t* __restrict__ nbr_count, int n, int n_types,
                    unsigned long long* __restrict__ inter) {
  __shared__ unsigned long long s_acc[PG_MAX_TYPES * PG_MAX_TYPES];
  for (int q = threadIdx.x; q < n_types * n_types; q += TPB) s_acc[q] = 0ull;
  __syncthreads();
  for (int i = blockIdx.x * TPB + threadIdx.x; i < n; i += gridDim.x * TPB) {
    const int t = type[i];
    if (t < 1 || t > n_types) continue;
    for (int b = 0; b < n_types; ++b) {
      const int c = nbr_count[(int64_t)i * n_types + b];
      if (c) atomicAdd(&s_acc[(t - 1) * n_types + b], (unsigned long long)c);
    }
  }
  __syncthreads();
  for (int q = threadIdx.x; q < n_types * n_types; q += TPB)
    if (s_acc[q]) atomicAdd(&inter[q], s_acc[q]);
}

}  // namespace

extern "C" {

int pg_knn_union_count(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx, const int32_t* row_id,
                       const int32_t* id_map, int32_t n_ids, int32_t* und_row_ptr, int32_t* up_row_ptr,
                       pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && k >= 1 && k <= PG_MAX_K, "pg_knn_union_count: need n >= 0 and 1 <= k <= %d", PG_MAX_K);
  PG_REQUIRE(h, und_row_ptr != nullptr && (n == 0 || knn_idx != nullptr), "pg_knn_union_count: NULL argument");
  PG_REQUIRE(h, (int64_t)n * k < (int64_t)1 << 31, "pg_knn_union_count: n*k must be < 2^31");
  PG_REQUIRE(h, (row_id == nullptr) == (id_map == nullptr) && (!id_map || n_ids > 0),
             "pg_knn_union_count: row_id and id_map go together (both NULL = identity)");
  int rc;
  if ((rc = pg_reserve(h, h->sym_extra, ((size_t)n + 4) * sizeof(int32_t)))) return rc;
  if ((rc = pg_reserve(h, h->sym_recip, (size_t)n * k + 16))) return rc;
  if (up_row_ptr && (rc = pg_reserve(h, h->sym_cursor, ((size_t)n + 4) * sizeof(int32_t)))) return rc;
  int32_t* row_count = (int32_t*)h->sym_extra.p;
  int32_t* up_count = up_row_ptr ? (int32_t*)h->sym_cursor.p : nullptr;
  if (n > 0) {
    PG_CUDA(h, cudaMemsetAsync(row_count, 0, (size_t)n * sizeof(int32_t), s));
    if (up_count) PG_CUDA(h, cudaMemsetAsync(up_count, 0, (size_t)n * sizeof(int32_t), s));
    const int blocks = pg_div_up(n, TPB);
    const bool vec = ((uintptr_t)knn_idx & 15) == 0;
#define PG_MARK(K) PG_LAUNCH(h, s, "sym_mark_kernel", sym_mark_kernel<K><<<blocks, TPB, 0, s>>>(knn_idx, n, k, row_id, id_map, n_ids, (uint8_t*)h->sym_recip.p, row_count, up_count))
    if (vec && k == 8) PG_MARK(8);
    else if (vec && k == 16) PG_MARK(16);
    else if (vec && k == 4) PG_MARK(4);
    else if (k == 5) PG_MARK(5);
    else PG_MARK(0);
#undef PG_MARK
    PG_LAUNCH_CHECK(h);
  }
  int32_t* totals = (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS);
  // the scan leaves row_count all zero again: pg_knn_union_fill uses it as the push cursor
  if ((rc = pg_scan_i32(h, row_count, und_row_ptr, n, s, totals + 1, true))) return rc;
  if (up_row_ptr && (rc = pg_scan_i32(h, up_count, up_row_ptr, n, s, totals + 2, false))) return rc;
  return PG_OK;
}

int pg_knn_union_total(pg_handle* h, int64_t* total, int64_t* upper_total) {
  if (!h || !total) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  PG_CUDA(h, cudaMemcpyAsync(&h->pinned[1], (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS) + 1, 2 * sizeof(int32_t),
                             cudaMemcpyDeviceToHost, h->last_stream));
  PG_CUDA(h, cudaStreamSynchronize(h->last_stream));
  *total = h->pinned[1];
  if (upper_total) *upper_total = h->pinned[2];  // meaningful after a count pass that was given up_row_ptr
  return PG_OK;
}

int pg_knn_union_fill(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx, const double* dist64,
                      const float* dist32, const int32_t* row_id, const int32_t* id_map,
                      const int32_t* und_row_ptr, const int32_t* up_row_ptr, int32_t* und_col, double* und_w64,
                      float* und_w32, const pg_union_out* extra, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && k >= 1 && k <= PG_MAX_K, "pg_knn_union_fill: bad n / k");
  PG_REQUIRE(h, n == 0 || dist64 || dist32, "pg_knn_union_fill: one of dist64 / dist32 is required");
  PG_REQUIRE(h, und_row_ptr && (n == 0 || (knn_idx && und_col)), "pg_knn_union_fill: NULL argument");
  pg_union_out x{};
  if (extra) x = *extra;
  PG_REQUIRE(h, !(x.edges || x.edge_w64 || x.edge_w32) || up_row_ptr, "pg_knn_union_fill: the edge list needs up_row_ptr from the count pass");
  PG_REQUIRE(h, !x.nbr_count || (x.type && x.n_types >= 1 && x.n_types <= PG_MAX_TYPES),
             "pg_knn_union_fill: nbr_count needs type and 1 <= n_types <= %d", PG_MAX_TYPES);
  PG_REQUIRE(h, !x.hist || x.hist_len >= 1, "pg_knn_union_fill: hist_len must be >= 1");
  PG_REQUIRE(h, ((uintptr_t)x.edges & 15) == 0, "pg_knn_union_fill: edges must be 16-byte aligned");
  rank_extra rx{};
  int rc = pg_degree_prepare(h, x.stats, x.hist, x.hist_len, n, s, &rx.deg);
  if (rc || n == 0) return rc;
  // the total of the matching count pass sizes the staging rows - or, for a caller that has sized its own outputs by
  // their bound and wants no host synchronisation at all, the bound does (every list entry yields at most two entries)
  int64_t total = 0;
  if (x.presized) {
    total = 2 * (int64_t)n * k;
  } else if ((rc = pg_knn_union_total(h, &total, nullptr))) {
    return rc;
  }
  // staging (arrival-order rows) lives in the grid's scratch that is free at this point
  pg_buf& tcol = h->cell_of;
  pg_buf& tw = h->rank;
  if ((rc = pg_reserve(h, tcol, ((size_t)total + 4) * sizeof(int32_t)))) return rc;
  if ((rc = pg_reserve(h, tw, ((size_t)total + 4) * sizeof(double)))) return rc;
  int32_t* cursor = (int32_t*)h->sym_extra.p;  // all zero since the count pass's scan
  const uint8_t* recip = (const uint8_t*)h->sym_recip.p;
  rx.row_id = row_id;
  rx.up_ptr = (x.edges || x.edge_w64 || x.edge_w32) ? up_row_ptr : nullptr;
  rx.edges = (long long*)x.edges; rx.ew64 = x.edge_w64; rx.ew32 = x.edge_w32;
  rx.type = x.type; rx.n_types = x.nbr_count ? x.n_types : 1; rx.nbr_count = x.nbr_count;
  rx.degree = x.degree;
  rx.sym_dist = x.symmetric_dist != 0;
  const int blocks = pg_div_up(n, TPB);
  const bool vec = (((uintptr_t)knn_idx | (uintptr_t)dist64 | (uintptr_t)dist32) & 15) == 0;
#define PG_PUSH(DT, D, K) PG_LAUNCH(h, s, "sym_push_kernel", sym_push_kernel<DT, K><<<blocks, TPB, 0, s>>>(knn_idx, D, n, k, row_id, id_map, recip, und_row_ptr, cursor, (int32_t*)tcol.p, (DT*)tw.p))
#define PG_RANK(DT, D, K) PG_LAUNCH(h, s, "sym_rank_kernel", sym_rank_kernel<DT, K><<<blocks, TPB, 0, s>>>(knn_idx, D, n, k, id_map, recip, und_row_ptr, (const int32_t*)tcol.p, (const DT*)tw.p, und_col, und_w64, und_w32, rx))
  if (dist64) {
    if (vec && k == 8) { PG_PUSH(double, dist64, 8); PG_RANK(double, dist64, 8); }
    else if (vec && k == 16) { PG_PUSH(double, dist64, 16); PG_RANK(double, dist64, 16); }
    else { PG_PUSH(double, dist64, 0); PG_RANK(double, dist64, 0); }
  } else {
    if (vec && k == 8) { PG_PUSH(float, dist32, 8); PG_RANK(float, dist32, 8); }
    else if (vec && k == 16) { PG_PUSH(float, dist32, 16); PG_RANK(float, dist32, 16); }
    else { PG_PUSH(float, dist32, 0); PG_RANK(float, dist32, 0); }
  }
#undef PG_PUSH
#undef PG_RANK
  PG_LAUNCH_CHECK(h);
  // the cursor holds the arrival counts now; the next count pass clears it again
  return PG_OK;
}

// the plain symmetrisation = the union without the fused extras
int pg_knn_symmetrize_count(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx, const int32_t* row_id,
                            const int32_t* id_map, int32_t n_ids, int32_t* und_row_ptr, pg_stream stream) {
  return pg_knn_union_count(h, n, k, knn_idx, row_id, id_map, n_ids, und_row_ptr, nullptr, stream);
}

int pg_knn_symmetrize_total(pg_handle* h, int64_t* total) { return pg_knn_union_total(h, total, nullptr); }

int pg_knn_symmetrize_fill(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx, const double* dist64,
                           const float* dist32, const int32_t* row_id, const int32_t* id_map,
                           const int32_t* und_row_ptr, int32_t* und_col, double* und_w64, float* und_w32,
                           pg_stream stream) {
  return pg_knn_union_fill(h, n, k, knn_idx, dist64, dist32, row_id, id_map, und_row_ptr, nullptr, und_col, und_w64,
                           und_w32, nullptr, stream);
}

int pg_csr_upper_count(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col,
                       const int32_t* row_id, int32_t* up_ptr, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && row_ptr && up_ptr, "pg_csr_upper_count: bad argument");
  int rc;
  if ((rc = pg_reserve(h, h->row_count, ((size_t)n + 4) * sizeof(int32_t)))) return rc;
  if (n > 0) {
    PG_LAUNCH(h, s, "upper_count_kernel", upper_count_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>(row_ptr, col, row_id, n, (int32_t*)h->row_count.p));
    PG_LAUNCH_CHECK(h);
  }
  return pg_scan_i32(h, (const int32_t*)h->row_count.p, up_ptr, n, s, (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS) + 2);
}

int pg_csr_upper_total(pg_handle* h, int64_t* total) {
  if (!h || !total) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  PG_CUDA(h, cudaMemcpyAsync(&h->pinned[2], (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS) + 2, sizeof(int32_t),
                             cudaMemcpyDeviceToHost, h->last_stream));
  PG_CUDA(h, cudaStreamSynchronize(h->last_stream));
  *total = h->pinned[2];
  return PG_OK;
}

int pg_csr_upper_fill(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, const double* w64,
                      const float* w32, const int32_t* row_id, const int32_t* up_ptr, int64_t* edges_i64,
                      double* ew64, float* ew32, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && row_ptr && up_ptr, "pg_csr_upper_fill: bad argument");
  PG_REQUIRE(h, !(ew64 || ew32) || (w64 || w32), "pg_csr_upper_fill: weights requested but none given");
  if (n == 0) return PG_OK;
  PG_LAUNCH(h, s, "upper_fill_kernel", upper_fill_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>(row_ptr, col, w64, w32, row_id, up_ptr, n, (long long*)edges_i64,
                                                     ew64, ew32));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_compose_degree(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, const int32_t* type,
                      int32_t n_types, int32_t* nbr_count, int32_t* degree, pg_degree_stats* stats, int32_t* hist,
                      int32_t hist_len, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && row_ptr, "pg_compose_degree: bad argument");
  PG_REQUIRE(h, !nbr_count || (type && col && n_types >= 1 && n_types <= PG_MAX_TYPES),
             "pg_compose_degree: nbr_count needs type, col and 1 <= n_types <= %d", PG_MAX_TYPES);
  PG_REQUIRE(h, !hist || hist_len >= 1, "pg_compose_degree: hist_len must be >= 1");
  pg_degree_out dout;
  int rc = pg_degree_prepare(h, stats, hist, hist_len, n, s, &dout);
  if (rc || n == 0) return rc;
  if (!nbr_count || n_types <= 8)
    PG_LAUNCH(h, s, "compose_kernel<8>", compose_kernel<8><<<pg_div_up(n, TPB), TPB, 0, s>>>(row_ptr, col, type, n, n_types, nbr_count, degree, dout));
  else
    PG_LAUNCH(h, s, "compose_kernel<16>", compose_kernel<16><<<pg_div_up(n, TPB), TPB, 0, s>>>(row_ptr, col, type, n, n_types, nbr_count, degree, dout));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_clustering(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t* triangles,
                  double* coeff, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && row_ptr, "pg_clustering: bad argument");
  if (n == 0) return PG_OK;
  PG_REQUIRE(h, col != nullptr, "pg_clustering: col is NULL");
  int rc;
  if ((rc = pg_reserve(h, h->row_count, ((size_t)n + 4) * sizeof(int32_t)))) return rc;
  int32_t* tri2 = (int32_t*)h->row_count.p;
  PG_CUDA(h, cudaMemsetAsync(tri2, 0, (size_t)n * sizeof(int32_t), s));
  PG_LAUNCH(h, s, "clustering_count_kernel", clustering_count_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>(row_ptr, col, n, tri2));
  PG_LAUNCH(h, s, "clustering_finish_kernel", clustering_finish_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>(row_ptr, tri2, n, triangles, coeff));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_type_interactions(pg_handle* h, int32_t n, const int32_t* type, const int32_t* nbr_count, int32_t n_types,
                         int64_t* inter, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, n >= 0 && n_types >= 1 && n_types <= PG_MAX_TYPES && inter, "pg_type_interactions: bad argument");
  PG_REQUIRE(h, n == 0 || (type && nbr_count), "pg_type_interactions: type / nbr_count is NULL");
  PG_CUDA(h, cudaMemsetAsync(inter, 0, (size_t)n_types * n_types * sizeof(int64_t), s));
  if (n == 0) return PG_OK;
  const int blocks = std::min(pg_div_up(n, TPB), h->sm_count * 4);
  PG_LAUNCH(h, s, "interactions_kernel", interactions_kernel<<<blocks, TPB, 0, s>>>(type, nbr_count, n, n_types, (unsigned long long*)inter));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
