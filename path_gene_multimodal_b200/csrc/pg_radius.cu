// K6 radius graph with K8 (neighbour-type histogram + degree statistics) fused in.
// Reference: /root/reference/hovernet_tile_inference.ipynb:2964-2975 (cKDTree.query_ball_tree, i<j edge
// loop), :3021 (edge_index), :3041-3042 (np.linalg.norm distances, float32 edge_attr); composition /
// degree per SURVEY A.5. Acceptance test is d2 <= r*r in float64 with d2 = fl(fl(dx*dx)+fl(dy*dy)).
//
// The CSR is built count -> scan -> fill, but every neighbourhood is walked only ONCE and all scattered
// traffic is confined to two single-instruction gathers:
//   walk   (pg_radius_count, kernel 1) one thread per point in CELL order. Cells are strip-ordered
//          (pg_common.cuh), so the lanes of a warp / the threads of a CTA sit in a compact patch and their
//          candidate records (one 32-byte sector each, one 256-bit load) hit in L1. With cell ~ r the 3x3 block
//          of a point is three contiguous runs (one per cell column), walked as ONE merged loop with four loads
//          in flight; the points on a strip edge add a short second loop over the three cells across the edge.
//          Loads past the end of a run are pointed at a sentinel record at infinity, and a point meets itself
//          like any other candidate (undone once after the loop), so the loop body has no special cases.
//          Per point it leaves ONE 32-byte pg_pt_meta {degree, entries, offset, 5 type counts} at its ROW's
//          position (one scattered full-sector store: fire and forget) and parks the row's accepted (id, d2) entries - staged in a
//          small shared-memory slab - in the CTA's own region of a temporary array (space claimed with a
//          shared-memory atomic per warp; a shared overflow region takes what does not fit).
//   rows   (pg_radius_count, kernel 2) one thread per 4 ROWS: reads their meta records (contiguous 256-bit loads)
//          and writes row_ptr (decoupled look-back scan of the entry
//          counts), degree, nbr_count and row_off coalesced; the degree statistics / histogram are reduced
//          here too (CTA -> accumulators; the last CTA publishes them and re-arms the accumulators).
//   gather (pg_radius_fill) warp-flattened over 32 rows: lane p of the warp's contiguous output range finds its
//          row by a 5-step shuffle search, reads one parked entry, ranks it among the row's entries by counting
//          smaller ids (rows are short; ids are distinct) and writes col / dist / edges fully coalesced.
#include <cfloat>
#include <cmath>
#include <cstring>
#include <algorithm>
#include "pg_query.cuh"
#include "pg_scan.cuh"

namespace {

#ifndef PG_WALK_TPB
#define PG_WALK_TPB 128
#endif
#ifndef PG_WALK_MINB
#define PG_WALK_MINB 8
#endif
constexpr int TPB_WALK = PG_WALK_TPB;
#ifndef PG_WALK_SLAB
#define PG_WALK_SLAB 8
#endif
constexpr int SLAB = PG_WALK_SLAB;   // row entries staged per thread in shared memory (12 B x SLAB x TPB_WALK = 12 KB)
#ifndef PG_ROWS_TPB
#define PG_ROWS_TPB 256
#endif
#ifndef PG_ROWS_ITEMS
#define PG_ROWS_ITEMS 4
#endif
constexpr int TPB_ROWS = PG_ROWS_TPB;
constexpr int ROWS_ITEMS = PG_ROWS_ITEMS;
constexpr int ROWS_TILE = TPB_ROWS * ROWS_ITEMS;
constexpr int TPB_GATHER = 256;
constexpr int FIELD_MAX = (1 << PG_TYPE_BITS) - 1;

struct __align__(16) pg_tmp_ent {
  double d2;
  int32_t id;
  int32_t pad;
};

struct __align__(32) pg_pt_meta {
  int32_t deg, cnt, off;
  int32_t c[PG_PACKED_TYPES];
};
static_assert(sizeof(pg_pt_meta) == 32, "pg_pt_meta must be one sector");

__device__ __forceinline__ void st_meta(pg_pt_meta* p, const pg_pt_meta& m) {
  const unsigned long long a = (unsigned long long)(uint32_t)m.deg | ((unsigned long long)(uint32_t)m.cnt << 32);
  const unsigned long long b = (unsigned long long)(uint32_t)m.off | ((unsigned long long)(uint32_t)m.c[0] << 32);
  const unsigned long long c = (unsigned long long)(uint32_t)m.c[1] | ((unsigned long long)(uint32_t)m.c[2] << 32);
  const unsigned long long d = (unsigned long long)(uint32_t)m.c[3] | ((unsigned long long)(uint32_t)m.c[4] << 32);
  asm volatile("st.global.v4.b64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}
__device__ __forceinline__ pg_pt_meta ld_meta(const pg_pt_meta* p) {
  unsigned long long a, b, c, d;
  asm volatile("ld.global.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
  pg_pt_meta m;
  m.deg = (int32_t)(uint32_t)a; m.cnt = (int32_t)(uint32_t)(a >> 32);
  m.off = (int32_t)(uint32_t)b; m.c[0] = (int32_t)(uint32_t)(b >> 32);
  m.c[1] = (int32_t)(uint32_t)c; m.c[2] = (int32_t)(uint32_t)(c >> 32);
  m.c[3] = (int32_t)(uint32_t)d; m.c[4] = (int32_t)(uint32_t)(d >> 32);
  return m;
}

// Merged walk over three runs [b0,e0) [b1,e1) [b2,e2) of the record array: f(record) for every slot; the
// slots past the end read the sentinel record at `pad` (infinitely far away, rejected by every f).
// flush() at least once every FIELD_MAX slots and once at the end.
template <class F, class FL>
__device__ __forceinline__ void walk_runs3(const pg_rec* rec, int b0, int e0, int b1, int e1, int b2, int e2,
                                           int pad, F&& f, FL&& flush) {
  const int n0 = e0 - b0, n01 = n0 + (e1 - b1), tot = n01 + (e2 - b2);
  const int off1 = b1 - n0, off2 = b2 - n01;
  auto pos = [&](int t) { return t < tot ? t + (t < n0 ? b0 : (t < n01 ? off1 : off2)) : pad; };
  for (int t0 = 0; t0 < tot; t0 += FIELD_MAX - 3) {  // FIELD_MAX - 3 is a multiple of 4
    const int t1 = min(tot, t0 + FIELD_MAX - 3);
    for (int t = t0; t < t1; t += 4) {
      const int j0 = pos(t), j1 = pos(t + 1), j2 = pos(t + 2), j3 = pos(t + 3);
      PG_ASSERT(j0 >= 0 && j0 <= pad && j1 >= 0 && j1 <= pad && j2 >= 0 && j2 <= pad && j3 >= 0 && j3 <= pad);
      const pg_rec r0 = pg_ld_rec(rec + j0), r1 = pg_ld_rec(rec + j1);
      const pg_rec r2 = pg_ld_rec(rec + j2), r3 = pg_ld_rec(rec + j3);
      f(r0); f(r1); f(r2); f(r3);
    }
    flush();
  }
}

// Every candidate of the (2R+1)^2 block around (cx, cy), the query point itself included.
template <bool FAST, class F, class FL>
__device__ __forceinline__ void walk_block(const pg_grid_view& g, int R, int cx, int cy, F&& f, FL&& flush) {
  const int pad = g.n;  // the sentinel record
  if (FAST) {           // R == 1
    const int sy = cy >> PG_STRIP_LOG, ly = cy & (PG_STRIP - 1);
    const bool has_l = cx > 0, has_r = cx + 1 < g.nx;
    // pass 0: rows ly-1..ly+1 of the columns cx-1..cx+1 inside this strip (column x+1 starts PG_STRIP cells
    // after column x); pass 1 (strip-edge points only): the one row across the edge, in the adjacent strip
    int edge = -1;
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
      walk_runs3(g.rec, b0, e0, b1, e1, b2, e2, pad, f, flush);
    }
  } else {
    pg_visit_block(g, cx, cy, R, [&](int b, int e) {
      for (int j0 = b; j0 < e; j0 += FIELD_MAX - 3) {
        const int j1 = min(e, j0 + FIELD_MAX - 3);
        for (int j = j0; j < j1; j += 4) {
          const int p1 = j + 1 < j1 ? j + 1 : pad, p2 = j + 2 < j1 ? j + 2 : pad, p3 = j + 3 < j1 ? j + 3 : pad;
          const pg_rec r0 = pg_ld_rec(g.rec + j), r1 = pg_ld_rec(g.rec + p1);
          const pg_rec r2 = pg_ld_rec(g.rec + p2), r3 = pg_ld_rec(g.rec + p3);
          f(r0); f(r1); f(r2); f(r3);
        }
        flush();
      }
    });
  }
}

struct walk_out {
  pg_pt_meta* __restrict__ meta;
  pg_tmp_ent* __restrict__ tmp;
  int cta_cap;                       // entries in one CTA's region of tmp
  unsigned long long ovf_base;       // first entry of the overflow region
  unsigned long long ovf_cap;        // entries in the overflow region
  unsigned long long* ovf_cursor;
  int32_t* __restrict__ nbr_count;   // only the WIDE_TYPES variant writes the type counts itself
  int n_types;
};

// Entries kept: all neighbours (UPPER = false) or only id_j > id_i; degree and type counts are over all neighbours.
template <bool FAST, bool UPPER, bool WIDE_TYPES>
__global__ void __launch_bounds__(TPB_WALK, PG_WALK_MINB)
radius_walk_kernel(pg_grid_view g, double r2, int R, walk_out o) {
  __shared__ double s_d2[SLAB][TPB_WALK];
  __shared__ int s_key[SLAB][TPB_WALK];
  __shared__ int s_alloc;
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) s_alloc = 0;
  pg_pdl_launch();
  __syncthreads();
  pg_pdl_wait();

  const int q = blockIdx.x * TPB_WALK + tid;
  const pg_rec me = pg_ld_rec_ordered(g.rec + min(q, g.n - 1));
  const bool active = q < g.n && me.row < g.n_query;  // halo points own no row
  int cnt = 0, cx = 0, cy = 0;
  pg_pt_meta m;
  m.deg = 0; m.cnt = 0; m.off = -1;
#pragma unroll
  for (int t = 0; t < PG_PACKED_TYPES; ++t) m.c[t] = 0;
  if (active) {
    cx = pg_cell_coord(me.x, g.x0, g.inv_cell, g.nx);
    cy = pg_cell_coord(me.y, g.y0, g.inv_cell, g.ny);
    unsigned long long pk = 0;
    int deg = 0;
    walk_block<FAST>(g, R, cx, cy,
      [&](const pg_rec& c) {
        const double d2 = pg_dist2(me.x, me.y, c.x, c.y);
        const bool a = d2 <= r2;
        deg += a;
        pk += (unsigned long long)a << c.tshift;
        if (a && (UPPER ? c.id > me.id : c.id != me.id)) {
          if (cnt < SLAB) { s_key[cnt][tid] = c.id; s_d2[cnt][tid] = d2; }
          ++cnt;
        }
      },
      [&]() {
#pragma unroll
        for (int t = 0; t < PG_PACKED_TYPES; ++t) m.c[t] += (int)((pk >> (t * PG_TYPE_BITS)) & FIELD_MAX);
        pk = 0;
      });
    // the point met itself (d2 = 0 unless a coordinate is not finite): take it out again
    const int self = pg_dist2(me.x, me.y, me.x, me.y) <= r2;
    m.deg = deg - self;
    const unsigned long long own = (unsigned long long)self << me.tshift;
#pragma unroll
    for (int t = 0; t < PG_PACKED_TYPES; ++t) m.c[t] -= (int)((own >> (t * PG_TYPE_BITS)) & FIELD_MAX);
    m.cnt = cnt;
    if (WIDE_TYPES) {  // more than PG_PACKED_TYPES types: a second walk with counters in local memory (rare)
      int tc[PG_MAX_TYPES];
#pragma unroll
      for (int t = 0; t < PG_MAX_TYPES; ++t) tc[t] = 0;
      walk_block<FAST>(g, R, cx, cy,
        [&](const pg_rec& c) {
          const double d2 = pg_dist2(me.x, me.y, c.x, c.y);
          if (d2 <= r2 && c.id != me.id && c.type >= 1 && c.type <= o.n_types) tc[c.type - 1] += 1;
        },
        [&]() {});
      for (int t = 0; t < o.n_types; ++t) o.nbr_count[(int64_t)me.row * o.n_types + t] = tc[t];
    }
  }

  // ---- park the row's entries: the warp claims space in the CTA's region with one shared-memory atomic
  int incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += y;
  }
  const int wtot = __shfl_sync(0xffffffffu, incl, 31);
  long long wbase = -1;
  if (lane == 0 && wtot > 0) {
    const int loc = atomicAdd(&s_alloc, wtot);
    if (loc + wtot <= o.cta_cap) {
      wbase = (long long)blockIdx.x * o.cta_cap + loc;
    } else {  // the CTA's region is full: shared overflow region (the cursor keeps counting past its end)
      const unsigned long long at = atomicAdd(o.ovf_cursor, (unsigned long long)wtot);
      if (at + (unsigned long long)wtot <= o.ovf_cap) wbase = (long long)(o.ovf_base + at);
    }
  }
  wbase = __shfl_sync(0xffffffffu, wbase, 0);
  if (!active) return;
  if (wbase >= 0 && cnt > 0) {
    const long long off = wbase + (incl - cnt);
    m.off = (int)off;
    PG_ASSERT(off >= 0 && (unsigned long long)off + (unsigned long long)cnt <= o.ovf_base + o.ovf_cap);
    pg_tmp_ent* dst = o.tmp + off;
    if (cnt <= SLAB) {
      for (int t = 0; t < cnt; ++t) {
        pg_tmp_ent e; e.d2 = s_d2[t][tid]; e.id = s_key[t][tid]; e.pad = 0;
        dst[t] = e;
      }
    } else {  // long row: walk this point again and park the entries as they come
      int k = 0;
      walk_block<FAST>(g, R, cx, cy,
        [&](const pg_rec& c) {
          const double d2 = pg_dist2(me.x, me.y, c.x, c.y);
          if (d2 <= r2 && (UPPER ? c.id > me.id : c.id != me.id) && k < cnt) {
            pg_tmp_ent e; e.d2 = d2; e.id = c.id; e.pad = 0;
            dst[k++] = e;
          }
        },
        [&]() {});
    }
  }
  PG_ASSERT(me.row >= 0 && me.row < g.n_query);
  st_meta(o.meta + me.row, m);  // in ROW order: a scattered full-sector store here buys the row pass coalesced loads
}

struct fill_out {
  int32_t* __restrict__ col;
  float* __restrict__ dist32;
  double* __restrict__ dist64;
  long long* __restrict__ edges;
  int32_t* __restrict__ edges32;
  long long* __restrict__ edge_index;
  float* __restrict__ edge_attr;
  long long n_edges;
};

__device__ __forceinline__ void emit_entry(const fill_out& o, long long pos, int my_id, int key, double d2) {
  const double d = sqrt(d2);
  PG_ASSERT(pos >= 0);
  o.col[pos] = key;
  if (o.dist32) o.dist32[pos] = (float)d;
  if (o.dist64) o.dist64[pos] = d;
  if (o.edges) *reinterpret_cast<longlong2*>(o.edges + 2 * pos) = make_longlong2(my_id, key);
  if (o.edges32) *reinterpret_cast<int2*>(o.edges32 + 2 * pos) = make_int2(my_id, key);
  if (o.edge_index) {  // [2, 2E] = hstack(edges.T, edges[:, ::-1].T), ipynb:3021 (see SURVEY B-3)
    o.edge_index[pos] = my_id; o.edge_index[o.n_edges + pos] = key;
    o.edge_index[2 * o.n_edges + pos] = key; o.edge_index[3 * o.n_edges + pos] = my_id;
  }
  if (o.edge_attr) { o.edge_attr[pos] = (float)d; o.edge_attr[o.n_edges + pos] = (float)d; }  // ipynb:3041-3042
}

// The gather of 32 consecutive rows by one warp = one contiguous range [rp(lane 0), end) of the outputs, one lane
// per output entry. rp / off / id / my_cnt: the values of the lane's row.
__device__ __forceinline__ void gather_rows32(int rp, int end, int off, int id, int my_cnt, const pg_tmp_ent* tmp,
                                              const fill_out& o, long long capacity, int32_t* overflow) {
  const int lane = threadIdx.x & 31;
  const int begin = __shfl_sync(0xffffffffu, rp, 0);
  for (int p0 = begin; p0 < end; p0 += 32) {
    const int p = p0 + lane;
    int k = 0;  // the last row of the 32 that starts at or before p (empty rows share their start with the next row)
#pragma unroll
    for (int step = 16; step > 0; step >>= 1) {
      const int v = __shfl_sync(0xffffffffu, rp, k + step);
      if (v <= p) k += step;
    }
    const int roff = __shfl_sync(0xffffffffu, off, k);
    const int rcnt = __shfl_sync(0xffffffffu, my_cnt, k);
    const int rbase = __shfl_sync(0xffffffffu, rp, k);
    const int rid = __shfl_sync(0xffffffffu, id, k);
    if (p >= end) continue;
    if ((long long)rbase + rcnt > capacity || roff < 0) {
      atomicExch(overflow, 1);  // the row does not fit the caller's buffers (or never got parked): dropped, reported
      continue;
    }
    PG_ASSERT(p - rbase >= 0 && p - rbase < rcnt);
    const pg_tmp_ent* src = tmp + roff;
    const pg_tmp_ent e = src[p - rbase];
    int rank = 0;  // ids are distinct, so the place of an entry in its row is the number of smaller ids
    for (int u = 0; u < rcnt; u += 4) {
      const int i0 = src[u].id, i1 = src[min(u + 1, rcnt - 1)].id, i2 = src[min(u + 2, rcnt - 1)].id, i3 = src[min(u + 3, rcnt - 1)].id;
      rank += (i0 < e.id) + (u + 1 < rcnt && i1 < e.id) + (u + 2 < rcnt && i2 < e.id) + (u + 3 < rcnt && i3 < e.id);
    }
    emit_entry(o, (long long)rbase + rank, rid, e.id, e.d2);
  }
}

struct rows_out {
  int32_t* __restrict__ row_ptr;
  int32_t* __restrict__ degree;
  int32_t* __restrict__ nbr_count;   // NULL when not wanted or when the walk wrote it (wide types)
  int32_t* __restrict__ row_off;
  int n_types;
  pg_degree_stats* stats;
  int32_t* hist;
  int hist_len, hist_mode;           // 0 none, 1 shared-memory bins -> accumulators, 2 straight into hist (pre-zeroed)
  pg_stats_acc* acc;
  int32_t* acc_hist;
  int32_t* total_copy;
  unsigned long long* ovf_cursor;    // retired here: *ovf_needed = *ovf_cursor; *ovf_cursor = 0
  unsigned long long* ovf_needed;
};

// The row pass: meta records -> row order. Tiles of ROWS_TILE rows, decoupled look-back over the entry counts
// (tiles are handed out by the scan state's ticket, so a tile only waits on tiles that are running or done).
// The statistics are reduced between publishing the tile's aggregate and reading the predecessors', i.e. inside
// the look-back wait.
struct rows_gather {  // GATHER: the fill pass for the tile's own rows, fused in (outputs given at count time)
  const pg_tmp_ent* tmp;
  const int32_t* row_gid;
  fill_out fo;
  long long capacity;
  int32_t* overflow;
};

template <bool GATHER>
__global__ void __launch_bounds__(TPB_ROWS)
radius_rows_kernel(int n_query, const pg_pt_meta* meta, pg_scan_state st, rows_out o, rows_gather gx) {
  using TS = pg_tile_scan<TPB_ROWS>;
  __shared__ typename TS::smem_t sm;
  __shared__ int s_rp[GATHER ? ROWS_TILE + 1 : 1];
  __shared__ int s_off[GATHER ? ROWS_TILE : 1];
  __shared__ int s_hist[PG_ACC_HIST_MAX];
  __shared__ int s_mn, s_mx, s_last;
  __shared__ unsigned long long s_sum, s_sq;
  const int tid = threadIdx.x;
  const bool want_stats = o.stats != nullptr || o.hist_mode != 0;
  pg_pdl_launch();
  pg_pdl_wait();
  const int tile = TS::take_tile(sm, st);  // a ticket, not blockIdx.x: a tile then only waits on tiles that are already running
  const int row0 = tile * ROWS_TILE + tid * ROWS_ITEMS;
  const bool full = row0 + ROWS_ITEMS <= n_query;

  pg_pt_meta m[ROWS_ITEMS];
  if (o.hist_mode == 1)
    for (int i = tid; i < o.hist_len; i += TPB_ROWS) s_hist[i] = 0;
  if (tid == 0) { s_mn = 0x7fffffff; s_mx = -1; s_sum = 0; s_sq = 0; }
#pragma unroll
  for (int i = 0; i < ROWS_ITEMS; ++i) {
    if (row0 + i < n_query) m[i] = ld_meta(meta + row0 + i);
    else { m[i].deg = 0; m[i].cnt = 0; m[i].off = -1; }
  }
  int v[ROWS_ITEMS], tsum = 0;
#pragma unroll
  for (int i = 0; i < ROWS_ITEMS; ++i) { v[i] = tsum; tsum += m[i].cnt; }
  int tile_sum;
  const int thread_off = TS::local_scan(sm, st, tile, tsum, &tile_sum);  // barrier inside: the shared accumulators are ready

  // ---- everything that does not need the tile's prefix: row_off, degree, type counts, statistics
  if (full) {
    if (!GATHER) *reinterpret_cast<int4*>(o.row_off + row0) = make_int4(m[0].off, m[1].off, m[2].off, m[3].off);
    if (o.degree) *reinterpret_cast<int4*>(o.degree + row0) = make_int4(m[0].deg, m[1].deg, m[2].deg, m[3].deg);
    if (o.nbr_count) {
      if (o.n_types == PG_PACKED_TYPES) {  // 4 rows x 5 counts = 80 contiguous, 16-byte aligned bytes
        int4* d = reinterpret_cast<int4*>(o.nbr_count + (int64_t)row0 * PG_PACKED_TYPES);
        d[0] = make_int4(m[0].c[0], m[0].c[1], m[0].c[2], m[0].c[3]);
        d[1] = make_int4(m[0].c[4], m[1].c[0], m[1].c[1], m[1].c[2]);
        d[2] = make_int4(m[1].c[3], m[1].c[4], m[2].c[0], m[2].c[1]);
        d[3] = make_int4(m[2].c[2], m[2].c[3], m[2].c[4], m[3].c[0]);
        d[4] = make_int4(m[3].c[1], m[3].c[2], m[3].c[3], m[3].c[4]);
      } else {
#pragma unroll
        for (int i = 0; i < ROWS_ITEMS; ++i)
#pragma unroll
          for (int t = 0; t < PG_PACKED_TYPES; ++t)
            if (t < o.n_types) o.nbr_count[(int64_t)(row0 + i) * o.n_types + t] = m[i].c[t];
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < ROWS_ITEMS; ++i) {
      const int row = row0 + i;
      if (row < n_query) {
        if (!GATHER) o.row_off[row] = m[i].off;
        if (o.degree) o.degree[row] = m[i].deg;
        if (o.nbr_count)
#pragma unroll
          for (int t = 0; t < PG_PACKED_TYPES; ++t)
            if (t < o.n_types) o.nbr_count[(int64_t)row * o.n_types + t] = m[i].c[t];
      }
    }
  }
  if (want_stats) {  // thread -> warp -> CTA
    int mn = 0x7fffffff, mx = -1;
    long long sum = 0, sq = 0;
#pragma unroll
    for (int i = 0; i < ROWS_ITEMS; ++i) {
      if (row0 + i < n_query) {
        const int d = m[i].deg;
        mn = min(mn, d); mx = max(mx, d); sum += d; sq += (long long)d * d;
      }
    }
    if (o.hist_mode != 0) {
      // degrees cluster on a few bins: one atomic per distinct bin of the warp instead of one per lane
#pragma unroll
      for (int i = 0; i < ROWS_ITEMS; ++i) {
        const int bin = row0 + i < n_query ? min(m[i].deg, o.hist_len - 1) : -1;
        const unsigned int peers = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0 && (tid & 31) == __ffs(peers) - 1) {
          if (o.hist_mode == 1) atomicAdd(&s_hist[bin], __popc(peers));
          else atomicAdd(&o.hist[bin], __popc(peers));
        }
      }
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, d); sq += __shfl_xor_sync(0xffffffffu, sq, d); }
    if ((tid & 31) == 0) {
      atomicMin(&s_mn, mn); atomicMax(&s_mx, mx);
      atomicAdd(&s_sum, (unsigned long long)sum); atomicAdd(&s_sq, (unsigned long long)sq);
    }
  }

  // ---- the prefix of the tile (barrier inside: the CTA's statistics are complete after it)
  bool last;
  int total;
  const int base = thread_off + TS::look_back(sm, st, tile, tile_sum, &last, &total);
  if (tid == 0 && last) {
    o.row_ptr[n_query] = total;
    if (o.total_copy) *o.total_copy = total;
  }
  if (full) {
    *reinterpret_cast<int4*>(o.row_ptr + row0) = make_int4(v[0] + base, v[1] + base, v[2] + base, v[3] + base);
  } else {
#pragma unroll
    for (int i = 0; i < ROWS_ITEMS; ++i)
      if (row0 + i < n_query) o.row_ptr[row0 + i] = v[i] + base;
  }

  if (GATHER) {
    // ---- the tile's rows are complete: gather their parked entries now (the warp-per-32-rows gather of the fill pass)
#pragma unroll
    for (int i = 0; i < ROWS_ITEMS; ++i) { s_rp[tid * ROWS_ITEMS + i] = v[i] + base; s_off[tid * ROWS_ITEMS + i] = m[i].off; }
    if (tid == TPB_ROWS - 1) s_rp[ROWS_TILE] = (base - thread_off) + tile_sum;  // tile prefix + tile total
    __syncthreads();
    const int lane = tid & 31;
    for (int g = tid >> 5; g < ROWS_TILE / 32; g += TPB_ROWS / 32) {
      const int r0 = tile * ROWS_TILE + g * 32;
      if (r0 >= n_query) break;  // warp-uniform
      const int row = r0 + lane;
      const bool has_row = row < n_query;
      const int rp = s_rp[g * 32 + lane], rp1 = s_rp[g * 32 + lane + 1], end = s_rp[g * 32 + 32];
      gather_rows32(rp, end, has_row ? s_off[g * 32 + lane] : -1, has_row ? (gx.row_gid ? gx.row_gid[row] : row) : 0,
                    rp1 - rp, gx.tmp, gx.fo, gx.capacity, gx.overflow);
    }
  }

  // ---- CTA -> accumulators; the last CTA to get here publishes them and re-arms the accumulators
  if (want_stats) {
    if (tid == 0) {
      atomicMin(&o.acc->min_degree, s_mn); atomicMax(&o.acc->max_degree, s_mx);
      atomicAdd(&o.acc->sum_degree, s_sum); atomicAdd(&o.acc->sumsq_degree, s_sq);
    }
    if (o.hist_mode == 1)
      for (int i = tid; i < o.hist_len; i += TPB_ROWS)
        if (s_hist[i]) atomicAdd(&o.acc_hist[i], s_hist[i]);
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(&o.acc->done, 1u) == (unsigned int)st.num_tiles - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (o.hist_mode == 1)
    for (int i = tid; i < o.hist_len; i += TPB_ROWS) {
      o.hist[i] = *(volatile int32_t*)&o.acc_hist[i];
      o.acc_hist[i] = 0;
    }
  if (tid == 0) {
    volatile pg_stats_acc* a = o.acc;
    if (o.stats) {
      o.stats->min_degree = a->min_degree; o.stats->max_degree = a->max_degree;
      o.stats->sum_degree = (long long)a->sum_degree; o.stats->sumsq_degree = (long long)a->sumsq_degree;
      o.stats->n_nodes = n_query;
    }
    a->min_degree = 0x7fffffff; a->max_degree = -1; a->sum_degree = 0; a->sumsq_degree = 0; a->n_nodes = 0; a->done = 0;
    if (o.ovf_cursor) { *o.ovf_needed = *(volatile unsigned long long*)o.ovf_cursor; *o.ovf_cursor = 0ull; }
  }
}

// nothing to query: empty row_ptr and the statistics of an empty graph
__global__ void empty_graph_kernel(int32_t* row_ptr, int32_t* total_copy, pg_degree_stats* stats, int32_t* hist, int hist_len,
                                   unsigned long long* ovf_needed) {
  if (threadIdx.x == 0) {
    row_ptr[0] = 0;
    *total_copy = 0;
    *ovf_needed = 0;
    if (stats) { stats->min_degree = 0; stats->max_degree = 0; stats->sum_degree = 0; stats->sumsq_degree = 0; stats->n_nodes = 0; }
  }
  if (hist)
    for (int i = threadIdx.x; i < hist_len; i += blockDim.x) hist[i] = 0;
}

// The stand-alone gather (pg_radius_fill): one warp per 32 consecutive rows.
__global__ void __launch_bounds__(TPB_GATHER)
radius_gather_kernel(int n_query, const int32_t* row_ptr, const int32_t* row_off,
                     const pg_tmp_ent* tmp, const int32_t* row_gid,
                     fill_out o, long long capacity, int32_t* overflow) {
  const int lane = threadIdx.x & 31;
  const int r0 = ((blockIdx.x * TPB_GATHER + threadIdx.x) >> 5) << 5;
  pg_pdl_launch();
  pg_pdl_wait();
  if (r0 >= n_query) return;  // warp-uniform
  const int row = r0 + lane;
  const bool has_row = row < n_query;
  const int rp = row_ptr[min(row, n_query)];
  const int off = has_row ? row_off[row] : -1;
  const int id = has_row ? (row_gid ? row_gid[row] : row) : 0;
  const int end = row_ptr[min(r0 + 32, n_query)];
  const int rp_next = __shfl_down_sync(0xffffffffu, rp, 1);
  gather_rows32(rp, end, off, id, (lane == 31 ? end : rp_next) - rp, tmp, o, capacity, overflow);
}

// sizes tmp_ent for the pass described by h->last_count: one region per walk CTA + the overflow region
int size_tmp(pg_handle* h) {
  const pg_grid& gr = h->grid;
  const int64_t n_cta = pg_div_up(std::max(gr.n, 1), TPB_WALK);
  // per point: twice what a past pass produced on average, else a first guess
  const double per_point = h->tmp_hint > 0 && gr.n_query > 0 ? 2.0 * (double)h->tmp_hint / gr.n_query
                                                               : (h->last_count.flags == PG_RADIUS_UPPER ? 4.0 : 8.0);
  int64_t cta_cap = (int64_t)std::ceil(std::min(per_point, 64.0) * TPB_WALK);
  cta_cap = (cta_cap + 7) & ~(int64_t)7;
  const int64_t ovf = std::max<int64_t>(h->tmp_ovf_hint, gr.n_query / 8 + 4096);
  const int64_t total = n_cta * cta_cap + ovf;
  if (total > 0x7ffffff0) return pg_set_error(h, PG_ERR_CAPACITY, "radius graph: more than 2^31 parked entries");
  int rc = pg_reserve(h, h->tmp_ent, (size_t)total * sizeof(pg_tmp_ent));
  if (rc) return rc;
  h->tmp_cta_cap = (int32_t)cta_cap;
  h->tmp_ovf_base = n_cta * cta_cap;
  h->tmp_cap = std::min<int64_t>((int64_t)(h->tmp_ent.cap / sizeof(pg_tmp_ent)), 0x7ffffff0);
  return PG_OK;
}

// enqueue walk + row pass of the pass described by h->last_count
int launch_count_pass(pg_handle* h, cudaStream_t s) {
  const auto& a = h->last_count;
  const pg_grid& gr = h->grid;
  const int nq = gr.n_query;
  unsigned long long* cursor = (unsigned long long*)((char*)h->misc.p + PG_MISC_TMPCUR);
  int32_t* totals = (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS);
  unsigned long long* needed = (unsigned long long*)(totals + 4);
  if (gr.n == 0 || nq == 0) {
    PG_LAUNCH(h, s, "empty_graph_kernel", empty_graph_kernel<<<1, 256, 0, s>>>(a.row_ptr, totals, a.stats, a.hist, a.hist ? a.hist_len : 0, needed));
    PG_LAUNCH_CHECK(h);
    return PG_OK;
  }
  pg_grid_view v = pg_make_view(h);
  const int R = pg_ring_radius(a.r, gr);
  const bool upper = a.flags == PG_RADIUS_UPPER;
  const bool wide = a.nbr_count && a.n_types > PG_PACKED_TYPES;
  walk_out w;
  w.meta = (pg_pt_meta*)h->pt_meta.p;
  w.tmp = (pg_tmp_ent*)h->tmp_ent.p;
  w.cta_cap = h->tmp_cta_cap;
  w.ovf_base = (unsigned long long)h->tmp_ovf_base;
  w.ovf_cap = (unsigned long long)(h->tmp_cap - h->tmp_ovf_base);
  w.ovf_cursor = cursor;
  w.nbr_count = a.nbr_count;
  w.n_types = a.nbr_count ? a.n_types : 1;
  const int blocks = pg_div_up(gr.n, TPB_WALK);
#define PG_WALK_LAUNCH(F, U, W) \
  PG_LAUNCH(h, s, "radius_walk_kernel", pg_launch_pdl(3, radius_walk_kernel<F, U, W>, blocks, TPB_WALK, s, v, a.r * a.r, R, w))
  if (wide) {
    if (R == 1) { if (upper) PG_WALK_LAUNCH(true, true, true); else PG_WALK_LAUNCH(true, false, true); }
    else { if (upper) PG_WALK_LAUNCH(false, true, true); else PG_WALK_LAUNCH(false, false, true); }
  } else {
    if (R == 1) { if (upper) PG_WALK_LAUNCH(true, true, false); else PG_WALK_LAUNCH(true, false, false); }
    else { if (upper) PG_WALK_LAUNCH(false, true, false); else PG_WALK_LAUNCH(false, false, false); }
  }
#undef PG_WALK_LAUNCH
  PG_LAUNCH_CHECK(h);

  rows_out o;
  o.row_ptr = a.row_ptr; o.degree = a.degree; o.nbr_count = wide ? nullptr : a.nbr_count;
  o.row_off = (int32_t*)h->row_off.p;
  o.n_types = a.nbr_count ? a.n_types : 1;
  o.stats = a.stats; o.hist = a.hist; o.hist_len = a.hist_len;
  o.hist_mode = a.hist ? (a.hist_len <= PG_ACC_HIST_MAX ? 1 : 2) : 0;
  if (o.hist_mode == 2) PG_CUDA(h, cudaMemsetAsync(a.hist, 0, (size_t)a.hist_len * sizeof(int32_t), s));
  o.acc = (pg_stats_acc*)((char*)h->misc.p + PG_MISC_ACC);
  o.acc_hist = (int32_t*)((char*)h->misc.p + PG_MISC_ACC_HIST);
  o.total_copy = totals;
  o.ovf_cursor = cursor; o.ovf_needed = needed;
  const int tiles = pg_div_up(nq, ROWS_TILE);
  pg_scan_state st;
  int rc = pg_scan_prepare(h, tiles, TPB_ROWS, s, &st);
  if (rc) return rc;
  rows_gather gx{};
  if (a.fused) {
    gx.tmp = (const pg_tmp_ent*)h->tmp_ent.p;
    gx.row_gid = gr.has_gid ? (const int32_t*)h->s_gid.p : nullptr;
    gx.fo = fill_out{a.col, a.dist32, a.dist64, (long long*)a.edges, a.edges32, nullptr, nullptr, 0};
    gx.capacity = (long long)a.capacity;
    gx.overflow = (int32_t*)((char*)h->misc.p + PG_MISC_OVERFLOW);
    PG_LAUNCH(h, s, "radius_rows_gather_kernel", pg_launch_pdl(4, radius_rows_kernel<true>, tiles, TPB_ROWS, s, nq, (const pg_pt_meta*)h->pt_meta.p, st, o, gx));
  } else {
    PG_LAUNCH(h, s, "radius_rows_kernel", pg_launch_pdl(4, radius_rows_kernel<false>, tiles, TPB_ROWS, s, nq, (const pg_pt_meta*)h->pt_meta.p, st, o, gx));
  }
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // namespace

extern "C" {

int pg_radius_reserve(pg_handle* h, int64_t entries) {
  if (!h) return PG_ERR_INVALID;
  PG_REQUIRE(h, entries >= 0, "pg_radius_reserve: entries < 0");
  if (entries > h->tmp_ovf_hint) h->tmp_ovf_hint = entries;
  return PG_OK;
}

int pg_radius_count(pg_handle* h, double r, int32_t flags, int32_t* row_ptr, int32_t* degree,
                    int32_t* nbr_count, int32_t n_types, pg_degree_stats* stats, int32_t* hist,
                    int32_t hist_len, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  h->last_count.valid = false;
  if (!h->grid.built) return pg_set_error(h, PG_ERR_STATE, "pg_radius_count: call pg_grid_build first");
  PG_REQUIRE(h, r >= 0 && std::isfinite(r), "pg_radius_count: r must be finite and >= 0");
  PG_REQUIRE(h, row_ptr != nullptr, "pg_radius_count: row_ptr is NULL");
  PG_REQUIRE(h, flags == PG_RADIUS_SYMMETRIC || flags == PG_RADIUS_UPPER, "pg_radius_count: bad flags %d", flags);
  PG_REQUIRE(h, !nbr_count || (n_types >= 1 && n_types <= PG_MAX_TYPES), "pg_radius_count: n_types must be in 1..%d", PG_MAX_TYPES);
  PG_REQUIRE(h, !hist || hist_len >= 1, "pg_radius_count: hist_len must be >= 1");
  PG_REQUIRE(h, ((uintptr_t)row_ptr & 15) == 0 && ((uintptr_t)degree & 15) == 0 && ((uintptr_t)nbr_count & 15) == 0,
             "pg_radius_count: row_ptr / degree / nbr_count must be 16-byte aligned");
  const pg_grid& gr = h->grid;
  int rc;
  if ((rc = pg_reserve(h, h->pt_meta, ((size_t)gr.n + 1) * sizeof(pg_pt_meta)))) return rc;
  if ((rc = pg_reserve(h, h->row_off, ((size_t)gr.n_query + 8) * sizeof(int32_t)))) return rc;
  h->radius_r = r;
  h->radius_flags = flags;
  auto& a = h->last_count;
  a.r = r; a.flags = flags; a.row_ptr = row_ptr; a.degree = degree; a.nbr_count = nbr_count; a.n_types = n_types;
  a.stats = stats; a.hist = hist; a.hist_len = hist_len;
  a.fused = false;
  if ((rc = size_tmp(h))) return rc;
  if ((rc = launch_count_pass(h, s))) return rc;
  a.valid = true;
  return PG_OK;
}

int pg_radius_graph(pg_handle* h, double r, int32_t flags, int32_t* row_ptr, int32_t* degree, int32_t* nbr_count,
                    int32_t n_types, pg_degree_stats* stats, int32_t* hist, int32_t hist_len, int32_t* col,
                    float* dist32, double* dist64, int64_t* edges_i64, int32_t* edges_i32, int64_t capacity,
                    pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  h->last_count.valid = false;
  if (!h->grid.built) return pg_set_error(h, PG_ERR_STATE, "pg_radius_graph: call pg_grid_build first");
  PG_REQUIRE(h, r >= 0 && std::isfinite(r), "pg_radius_graph: r must be finite and >= 0");
  PG_REQUIRE(h, row_ptr != nullptr, "pg_radius_graph: row_ptr is NULL");
  PG_REQUIRE(h, flags == PG_RADIUS_SYMMETRIC || flags == PG_RADIUS_UPPER, "pg_radius_graph: bad flags %d", flags);
  PG_REQUIRE(h, !nbr_count || (n_types >= 1 && n_types <= PG_MAX_TYPES), "pg_radius_graph: n_types must be in 1..%d", PG_MAX_TYPES);
  PG_REQUIRE(h, !hist || hist_len >= 1, "pg_radius_graph: hist_len must be >= 1");
  PG_REQUIRE(h, capacity >= 0 && (capacity == 0 || col != nullptr), "pg_radius_graph: capacity < 0 or col is NULL");
  PG_REQUIRE(h, (((uintptr_t)row_ptr | (uintptr_t)degree | (uintptr_t)nbr_count | (uintptr_t)edges_i64 | (uintptr_t)edges_i32) & 15) == 0,
             "pg_radius_graph: row_ptr / degree / nbr_count / edges must be 16-byte aligned");
  const pg_grid& gr = h->grid;
  int rc;
  if ((rc = pg_reserve(h, h->pt_meta, ((size_t)gr.n + 1) * sizeof(pg_pt_meta)))) return rc;
  if ((rc = pg_reserve(h, h->row_off, ((size_t)gr.n_query + 8) * sizeof(int32_t)))) return rc;
  if (capacity > h->tmp_ovf_hint) h->tmp_ovf_hint = capacity;  // as pg_radius_reserve
  h->radius_r = r;
  h->radius_flags = flags;
  auto& a = h->last_count;
  a.r = r; a.flags = flags; a.row_ptr = row_ptr; a.degree = degree; a.nbr_count = nbr_count; a.n_types = n_types;
  a.stats = stats; a.hist = hist; a.hist_len = hist_len;
  a.fused = true; a.col = col; a.dist32 = dist32; a.dist64 = dist64; a.edges = edges_i64; a.edges32 = edges_i32; a.capacity = capacity;
  if ((rc = size_tmp(h))) return rc;
  if ((rc = launch_count_pass(h, s))) return rc;
  a.valid = true;
  return PG_OK;
}

int pg_radius_total(pg_handle* h, int64_t* total) {
  if (!h || !total) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  if (!h->last_count.valid) return pg_set_error(h, PG_ERR_STATE, "pg_radius_total: call pg_radius_count first");
  for (int attempt = 0; attempt < 2; ++attempt) {
    PG_CUDA(h, cudaMemcpyAsync(&h->pinned[0], (char*)h->misc.p + PG_MISC_TOTALS, 8 * sizeof(int32_t),
                               cudaMemcpyDeviceToHost, h->last_stream));
    PG_CUDA(h, cudaMemcpyAsync(&h->pinned[8], (char*)h->misc.p + PG_MISC_BADINPUT, sizeof(int32_t),
                               cudaMemcpyDeviceToHost, h->last_stream));
    PG_CUDA(h, cudaStreamSynchronize(h->last_stream));
    {
      int rc_in = pg_check_input_flag(h);
      if (rc_in) return rc_in;
    }
    int64_t needed;
    memcpy(&needed, &h->pinned[4], sizeof(needed));
    const int64_t produced = h->pinned[0];
    if (produced > h->tmp_hint) h->tmp_hint = produced;
    if (needed <= h->tmp_cap - h->tmp_ovf_base) {
      *total = produced;
      return PG_OK;
    }
    // the overflow region was too small: size it to what the pass needed (and the CTA regions to the new
    // average) and redo the pass
    h->tmp_ovf_hint = std::max(h->tmp_ovf_hint, needed + needed / 4);
    int rc;
    if ((rc = size_tmp(h))) return rc;
    // a fused pass (pg_radius_graph) that ran out of parking space has flagged its dropped rows as a capacity
    // overflow: the redo starts from a clean flag
    if (h->last_count.fused)
      PG_CUDA(h, cudaMemsetAsync((char*)h->misc.p + PG_MISC_OVERFLOW, 0, sizeof(int32_t), h->last_stream));
    if ((rc = launch_count_pass(h, h->last_stream))) return rc;
  }
  return pg_set_error(h, PG_ERR_STATE, "pg_radius_total: the count pass did not settle");
}

int pg_radius_fill(pg_handle* h, const int32_t* row_ptr, int32_t* col, float* dist32, double* dist64,
                   int64_t* edges_i64, int32_t* edges_i32, int64_t* edge_index, float* edge_attr, int64_t n_edges,
                   int64_t capacity, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  if (!h->grid.built || !h->last_count.valid)
    return pg_set_error(h, PG_ERR_STATE, "pg_radius_fill: call pg_grid_build / pg_radius_count first");
  PG_REQUIRE(h, row_ptr != nullptr, "pg_radius_fill: row_ptr is NULL");
  PG_REQUIRE(h, capacity >= 0, "pg_radius_fill: capacity < 0");
  PG_REQUIRE(h, capacity == 0 || col != nullptr, "pg_radius_fill: col is NULL");
  PG_REQUIRE(h, !(edge_index || edge_attr) || (h->radius_flags == PG_RADIUS_UPPER && n_edges >= 0 && n_edges <= capacity),
             "pg_radius_fill: edge_index / edge_attr need the UPPER count pass and 0 <= n_edges <= capacity");
  PG_REQUIRE(h, (((uintptr_t)edges_i64 | (uintptr_t)edges_i32) & 15) == 0, "pg_radius_fill: edges must be 16-byte aligned");
  const pg_grid& gr = h->grid;
  if (gr.n == 0 || gr.n_query == 0) return PG_OK;
  fill_out o{col, dist32, dist64, (long long*)edges_i64, edges_i32, (long long*)edge_index, edge_attr, (long long)n_edges};
  int32_t* ovf = (int32_t*)((char*)h->misc.p + PG_MISC_OVERFLOW);
  const int blocks = pg_div_up(gr.n_query, TPB_GATHER);
  PG_LAUNCH(h, s, "radius_gather_kernel", pg_launch_pdl(5, radius_gather_kernel, blocks, TPB_GATHER, s,
      gr.n_query, row_ptr, (const int32_t*)h->row_off.p, (const pg_tmp_ent*)h->tmp_ent.p,
      gr.has_gid ? (const int32_t*)h->s_gid.p : nullptr, o, (long long)capacity, ovf));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
