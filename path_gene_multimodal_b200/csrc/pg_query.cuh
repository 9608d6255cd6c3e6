// Shared device-side pieces of the grid queries (K5 kNN, K6 radius).
#pragma once
#include <algorithm>
#include <cfloat>
#include <cmath>
#include "pg_common.cuh"

// One point of the cell-ordered array = one 32-byte DRAM sector: the counting-sort scatter writes it
// with a single 256-bit store (a full sector, so L2 never has to fetch the old contents) and a query
// reads coordinates, ids and type of a candidate with a single 256-bit load.
struct __align__(32) pg_rec {
  double x, y;
  int32_t row;     // index of the point in the caller's arrays (its output row; >= n_query: halo point)
  int32_t id;      // id used for ordering / output columns: gid[row] when gids were given, else row
  int32_t type;    // cell type id as given
  int32_t tshift;  // bit offset of the type's 12-bit field in the packed neighbour-type counter
};

#define PG_TYPE_BITS 12
#define PG_PACKED_TYPES 5
#define PG_TYPE_OTHER_SHIFT 60  // types outside 1..5 land in the 4 spare top bits (never read)

struct pg_grid_view {
  const int32_t* cell_start;  // no __restrict__: const + restrict loads become LDG.CONSTANT (see pg_ld_rec)
  const pg_rec* rec;
  int32_t n, n_query, nx, ny, nys;
  double x0, y0, cell, inv_cell;
};

static inline pg_grid_view pg_make_view(const pg_handle* h) {
  pg_grid_view v;
  v.cell_start = (const int32_t*)h->cell_start.p + 3;  // see pg_grid.cu: B[c] = first point of cell c
  v.rec = (const pg_rec*)h->s_rec.p;
  v.n = h->grid.n; v.n_query = h->grid.n_query; v.nx = h->grid.nx; v.ny = h->grid.ny; v.nys = h->grid.nys;
  v.x0 = h->grid.x0; v.y0 = h->grid.y0; v.cell = h->grid.cell; v.inv_cell = h->grid.inv_cell;
  return v;
}

// Block radius of a query of radius r over the grid gr (K6's radius walk, K16's pair histogram).
static inline int pg_ring_radius(double r, const pg_grid& gr) {
  // every point within r lies at most R cells away along each axis. The binning t = fl(fl(v - x0) * inv_cell) rounds
  // twice (each within t eps / 2), so two points r apart can land r * inv_cell + 2 t eps apart; the t that matters is
  // below max(nx, ny) + R + 1 (a pair clamped on the same side shares its border cell), so 4 max(nx, ny) eps covers it
  // with room to spare. A fixed slack does not cover it: at t just below 2^26, r = 13/64 and cell = r (1 + 3e-9),
  // two points exactly r apart bin two rows apart. radius_cell's 2^-20 margin keeps R = 1 up to the 2^28-cell cap.
  // Capped in double before the conversion: a block of radius max(nx, ny) already covers the grid, and a ball far
  // larger than the grid (r / cell past INT_MAX, or cx + R past INT_MAX in the block walk) would not convert or add
  // safely.
  const double cover = (double)std::max(gr.nx, gr.ny);
  const double R = std::ceil(r * gr.inv_cell * (1.0 + 1e-9) + 1e-9 + 4.0 * cover * DBL_EPSILON);
  if (!(R < cover)) return std::max((int)cover, 1);
  return R < 1.0 ? 1 : (int)R;
}

#ifdef __CUDACC__
// 256-bit global load / store (LDG.E.256 / STG.E.256 on sm_100a)
__device__ __forceinline__ pg_rec pg_ld_rec(const pg_rec* p) {
  unsigned long long a, b, c, d;
  // NOT .nc: the query kernels may be scheduled (programmatic dependent launch) while the scatter that writes the
  // records is still running, and ptxas hoists .nc loads above griddepcontrol.wait. Not volatile, so the loads of
  // a batch can be issued back to back.
  asm("ld.global.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
  pg_rec r;
  r.x = __longlong_as_double((long long)a);
  r.y = __longlong_as_double((long long)b);
  r.row = (int32_t)(uint32_t)c; r.id = (int32_t)(uint32_t)(c >> 32);
  r.type = (int32_t)(uint32_t)d; r.tshift = (int32_t)(uint32_t)(d >> 32);
  return r;
}
// same load, but ordered after earlier volatile asm (pg_pdl_wait): for the first read of a kernel
__device__ __forceinline__ pg_rec pg_ld_rec_ordered(const pg_rec* p) {
  unsigned long long a, b, c, d;
  asm volatile("ld.global.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
  pg_rec r;
  r.x = __longlong_as_double((long long)a);
  r.y = __longlong_as_double((long long)b);
  r.row = (int32_t)(uint32_t)c; r.id = (int32_t)(uint32_t)(c >> 32);
  r.type = (int32_t)(uint32_t)d; r.tshift = (int32_t)(uint32_t)(d >> 32);
  return r;
}
__device__ __forceinline__ void pg_st_rec(pg_rec* p, double x, double y, int row, int id, int type, int tshift) {
  const unsigned long long a = (unsigned long long)__double_as_longlong(x), b = (unsigned long long)__double_as_longlong(y);
  const unsigned long long c = (unsigned long long)(uint32_t)row | ((unsigned long long)(uint32_t)id << 32);
  const unsigned long long d = (unsigned long long)(uint32_t)type | ((unsigned long long)(uint32_t)tshift << 32);
  asm volatile("st.global.v4.b64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}

// Rows ya..yb (inclusive, inside the grid) of column x as contiguous runs of the cell-ordered array: one run
// per strip touched (see the cell order in pg_common.cuh).
template <class F>
__device__ __forceinline__ void pg_visit_column(const pg_grid_view& g, int x, int ya, int yb, F&& f) {
  for (int s = ya >> PG_STRIP_LOG; s <= (yb >> PG_STRIP_LOG); ++s) {
    const int s0 = s << PG_STRIP_LOG;
    const int la = max(ya, s0) - s0, lb = min(yb, s0 + PG_STRIP - 1) - s0;
    const int32_t* c = g.cell_start + (((int64_t)s * g.nx + x) << PG_STRIP_LOG);
    f(c[la], c[lb + 1]);
  }
}

// Visit the (2R+1)^2 block of cells around (cx, cy).
template <class F>
__device__ __forceinline__ void pg_visit_block(const pg_grid_view& g, int cx, int cy, int R, F&& f) {
  const int xa = max(cx - R, 0), xb = min(cx + R, g.nx - 1);
  const int ya = max(cy - R, 0), yb = min(cy + R, g.ny - 1);
  for (int x = xa; x <= xb; ++x) pg_visit_column(g, x, ya, yb, f);
}

// Visit only the ring at Chebyshev distance exactly R (R >= 1) around (cx, cy).
template <class F>
__device__ __forceinline__ void pg_visit_ring(const pg_grid_view& g, int cx, int cy, int R, F&& f) {
  const int ya = max(cy - R, 0), yb = min(cy + R, g.ny - 1);
  if (cx - R >= 0) pg_visit_column(g, cx - R, ya, yb, f);
  if (cx + R < g.nx) pg_visit_column(g, cx + R, ya, yb, f);
  const int xa = max(cx - R + 1, 0), xb = min(cx + R - 1, g.nx - 1);
  const bool top = cy - R >= 0, bottom = cy + R < g.ny;
  for (int x = xa; x <= xb; ++x) {
    if (top) { const int c = pg_cell_index(g.nx, x, cy - R); f(g.cell_start[c], g.cell_start[c + 1]); }
    if (bottom) { const int c = pg_cell_index(g.nx, x, cy + R); f(g.cell_start[c], g.cell_start[c + 1]); }
  }
}

// Bounded sorted buffer used to emit a row in ascending key order in chunks of CAP entries:
// pass m keeps the CAP smallest keys greater than the last key already emitted.
template <int CAP>
struct pg_sorted_chunk {
  int key[CAP];
  double val[CAP];
  int m;
  int last;
  __device__ __forceinline__ void reset(int last_key) { m = 0; last = last_key; }
  __device__ __forceinline__ void push(int k, double v) {
    if (k <= last) return;
    if (m == CAP) {
      if (k >= key[CAP - 1]) return;
      m = CAP - 1;
    }
    int s = m;
    while (s > 0 && key[s - 1] > k) { key[s] = key[s - 1]; val[s] = val[s - 1]; --s; }
    key[s] = k; val[s] = v;
    ++m;
  }
};
#endif
