// K2-K4: uniform-grid binning of the centroids - atomic histogram over cells, single-pass scan
// (pg_scan.cu), counting-sort scatter. Plays the role of the cKDTree build at
// /root/reference/hovernet_tile_inference.ipynb:1818 (KNN.from_array) and :2964 (cKDTree(coords)).
//
// Cells are numbered strip by strip, column-major inside a strip (pg_common.cuh: pg_cell_index), so the
// cell-ordered array keeps spatial neighbours close in memory along BOTH axes.
//
// Passes over the points: (1) histogram with fire-and-forget atomics (nothing written per point),
// (2) scatter that re-derives the cell and claims its slot with one atomicAdd on the scanned array.
// The scan writes start(c) into B[c+1] (B[0] = 0 stays put); after the scatter's cursor increments
// B[c+1] = start(c) + count(c) = start(c+1), i.e. B has become the start-of-cell array itself - no
// per-point rank / cell arrays and no cursor copy.
#include <cmath>
#include "pg_query.cuh"

namespace {

#ifndef PG_GRID_TPB
#define PG_GRID_TPB 256
#endif
#ifndef PG_GRID_PTS
#define PG_GRID_PTS 2
#endif
constexpr int TPB = PG_GRID_TPB;

__device__ __forceinline__ unsigned long long dbl_key(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
static inline double key_dbl(unsigned long long k) {
  unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  double d;
  memcpy(&d, &b, sizeof(d));
  return d;
}

// keys[0..1] = min x,y  keys[2..3] = max x,y (monotone uint64 encoding; NaN skipped)
__global__ void __launch_bounds__(TPB)
bounds_kernel(const double2* __restrict__ xy, int n, unsigned long long* keys) {
  unsigned long long lo_x = ~0ull, lo_y = ~0ull, hi_x = 0, hi_y = 0;
  for (int i = blockIdx.x * TPB + threadIdx.x; i < n; i += gridDim.x * TPB) {
    double2 p = xy[i];
    if (p.x == p.x) { unsigned long long k = dbl_key(p.x); lo_x = min(lo_x, k); hi_x = max(hi_x, k); }
    if (p.y == p.y) { unsigned long long k = dbl_key(p.y); lo_y = min(lo_y, k); hi_y = max(hi_y, k); }
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    lo_x = min(lo_x, __shfl_xor_sync(0xffffffffu, lo_x, d));
    lo_y = min(lo_y, __shfl_xor_sync(0xffffffffu, lo_y, d));
    hi_x = max(hi_x, __shfl_xor_sync(0xffffffffu, hi_x, d));
    hi_y = max(hi_y, __shfl_xor_sync(0xffffffffu, hi_y, d));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(&keys[0], lo_x); atomicMin(&keys[1], lo_y);
    atomicMax(&keys[2], hi_x); atomicMax(&keys[3], hi_y);
  }
}

__global__ void init_bounds_kernel(unsigned long long* keys) {
  keys[0] = keys[1] = ~0ull;
  keys[2] = keys[3] = 0ull;
}

// K2: PTS points per thread (independent 256-bit loads in flight, one wave of CTAs for 1M points), reduction
// atomics (no return value, nothing else written)
constexpr int PTS = PG_GRID_PTS;
__device__ __forceinline__ void ld_xy2(const double2* p, double2& a, double2& b) {
  unsigned long long x0, y0, x1, y1;
  // volatile + not .nc: stays behind pg_pdl_wait (the coordinates may come from the kernel before this one)
  asm volatile("ld.global.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(x0), "=l"(y0), "=l"(x1), "=l"(y1) : "l"(p) : "memory");
  a = make_double2(__longlong_as_double((long long)x0), __longlong_as_double((long long)y0));
  b = make_double2(__longlong_as_double((long long)x1), __longlong_as_double((long long)y1));
}

// the PTS points of thread t of CTA b are b*TPB*PTS + k*TPB*2 + t*2 + {0,1} (k < PTS/2): pairs, so that a warp's
// 256-bit loads are contiguous
__device__ __forceinline__ void load_points(const double2* xy, int n, bool aligned32, int base, double2 (&p)[PTS]) {
#pragma unroll
  for (int k = 0; k < PTS / 2; ++k) {
    const int i = base + k * TPB * 2;
    if (aligned32 && i + 1 < n) {
      ld_xy2(xy + i, p[2 * k], p[2 * k + 1]);
    } else {
      if (i < n) p[2 * k] = xy[i];
      if (i + 1 < n) p[2 * k + 1] = xy[i + 1];
    }
  }
}

__global__ void __launch_bounds__(TPB)
histogram_kernel(const double2* xy, int n, bool aligned32, double x0, double y0, double inv_cell, int nx, int ny,
                 int32_t* cell_count, int32_t* bad_input, int epoch) {
  const int base = blockIdx.x * TPB * PTS + threadIdx.x * 2;
  pg_pdl_launch();
  pg_pdl_wait();
  double2 p[PTS];
  load_points(xy, n, aligned32, base, p);
#pragma unroll
  for (int k = 0; k < PTS; ++k) {
    const int i = base + (k >> 1) * TPB * 2 + (k & 1);
    if (i < n) {
      const int c = pg_cell_index(nx, pg_cell_coord(p[k].x, x0, inv_cell, nx), pg_cell_coord(p[k].y, y0, inv_cell, ny));
      PG_ASSERT(c >= 0 && (int64_t)c < (int64_t)nx * (((ny + PG_STRIP - 1) >> PG_STRIP_LOG) << PG_STRIP_LOG));
      atomicAdd(&cell_count[c], 1);
      // cKDTree refuses NaN / inf; here the build goes on (they land in a border cell) and the next call that
      // synchronises reports it
      if (!(isfinite(p[k].x) && isfinite(p[k].y))) *bad_input = epoch;
    }
  }
}

// K4: counting-sort scatter into cell order: one 32-byte record per point, written as one full sector.
// cursor = B + 1: cursor[c] starts as start(c) and ends as start(c+1). PTS points per thread, as in K2.
__global__ void __launch_bounds__(TPB)
scatter_kernel(const double2* xy, const int32_t* type, const int32_t* gid,
               int n, bool aligned32, double x0, double y0, double inv_cell, int nx, int ny, int32_t* cursor,
               pg_rec* rec, int32_t* gid_copy) {
  const int base = blockIdx.x * TPB * PTS + threadIdx.x * 2;
  pg_pdl_launch();
  pg_pdl_wait();
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    // sentinel behind the last record: infinitely far from everything (the queries pad their loads with it)
    const double inf = __longlong_as_double(0x7ff0000000000000ll);
    pg_st_rec(rec + n, inf, inf, 0x7fffffff, 0x7fffffff, 0, PG_TYPE_OTHER_SHIFT);
  }
  double2 p[PTS];
  int t[PTS], id[PTS], dst[PTS];
  load_points(xy, n, aligned32, base, p);
#pragma unroll
  for (int k = 0; k < PTS; ++k) {
    const int i = base + (k >> 1) * TPB * 2 + (k & 1);
    t[k] = (type && i < n) ? type[i] : 0;
    id[k] = i < n ? (gid ? gid[i] : i) : 0;
  }
#pragma unroll
  for (int k = 0; k < PTS; ++k) {
    const int i = base + (k >> 1) * TPB * 2 + (k & 1);
    dst[k] = 0;
    if (i < n) {
      const int c = pg_cell_index(nx, pg_cell_coord(p[k].x, x0, inv_cell, nx), pg_cell_coord(p[k].y, y0, inv_cell, ny));
      dst[k] = atomicAdd(&cursor[c], 1);
    }
  }
#pragma unroll
  for (int k = 0; k < PTS; ++k) {
    const int i = base + (k >> 1) * TPB * 2 + (k & 1);
    if (i < n) {
      const int tshift = (t[k] >= 1 && t[k] <= PG_PACKED_TYPES) ? (t[k] - 1) * PG_TYPE_BITS : PG_TYPE_OTHER_SHIFT;
      PG_ASSERT(dst[k] >= 0 && dst[k] < n);
      pg_st_rec(rec + dst[k], p[k].x, p[k].y, i, id[k], t[k], tshift);
      if (gid) gid_copy[i] = id[k];
    }
  }
}

// the points of the built grid, in cell order, back as plain arrays (a spatial sort of the input: see pg_grid_export)
__global__ void __launch_bounds__(TPB)
export_kernel(const pg_rec* __restrict__ rec, int n, double2* __restrict__ xy, int32_t* __restrict__ type, int32_t* __restrict__ gid) {
  const int p = blockIdx.x * TPB + threadIdx.x;
  if (p >= n) return;
  const pg_rec r = pg_ld_rec(rec + p);
  if (xy) xy[p] = make_double2(r.x, r.y);
  if (type) type[p] = r.type;
  if (gid) gid[p] = r.id;
}

}  // namespace

extern "C" {

int pg_grid_export(pg_handle* h, double* xy, int32_t* type, int32_t* gid, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  if (!h->grid.built) return pg_set_error(h, PG_ERR_STATE, "pg_grid_export: call pg_grid_build first");
  PG_REQUIRE(h, ((uintptr_t)xy & 15) == 0, "pg_grid_export: xy must be 16-byte aligned");
  const int n = h->grid.n;
  if (n == 0) return PG_OK;
  PG_LAUNCH(h, s, "export_kernel", export_kernel<<<pg_div_up(n, TPB), TPB, 0, s>>>((const pg_rec*)h->s_rec.p, n, (double2*)xy, type, gid));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

int pg_grid_build(pg_handle* h, int32_t n, int32_t n_query, const double* xy, const int32_t* type,
                  const int32_t* gid, double cell_size, const double* bounds, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  h->grid.built = false;
  h->build_epoch = h->build_epoch == 0x7fffffff ? 1 : h->build_epoch + 1;
  PG_REQUIRE(h, n >= 0 && n_query >= 0 && n_query <= n, "pg_grid_build: need 0 <= n_query <= n (n=%d n_query=%d)", n, n_query);
  PG_REQUIRE(h, cell_size > 0 && std::isfinite(cell_size), "pg_grid_build: cell_size must be finite and > 0");
  PG_REQUIRE(h, n == 0 || xy != nullptr, "pg_grid_build: xy is NULL");
  PG_REQUIRE(h, ((uintptr_t)xy & 15) == 0, "pg_grid_build: xy must be 16-byte aligned");

  double b[4] = {0, 0, 1, 1};
  if (bounds) {
    for (int i = 0; i < 4; ++i) b[i] = bounds[i];
    PG_REQUIRE(h, std::isfinite(b[0]) && std::isfinite(b[1]) && std::isfinite(b[2]) && std::isfinite(b[3]) &&
                      b[2] >= b[0] && b[3] >= b[1], "pg_grid_build: bad bounds");
  } else if (n > 0) {
    unsigned long long* keys = (unsigned long long*)((char*)h->misc.p + PG_MISC_BOUNDS);
    PG_LAUNCH(h, s, "init_bounds_kernel", init_bounds_kernel<<<1, 1, 0, s>>>(keys));
    int blocks = std::min(pg_div_up(n, TPB), h->sm_count * 8);
    PG_LAUNCH(h, s, "bounds_kernel", bounds_kernel<<<blocks, TPB, 0, s>>>((const double2*)xy, n, keys));
    PG_LAUNCH_CHECK(h);
    unsigned long long hk[4];
    PG_CUDA(h, cudaMemcpyAsync(hk, keys, sizeof(hk), cudaMemcpyDeviceToHost, s));
    PG_CUDA(h, cudaStreamSynchronize(s));
    if (hk[0] == ~0ull || hk[1] == ~0ull)
      return pg_set_error(h, PG_ERR_INVALID, "pg_grid_build: coordinates must be finite (every coordinate is NaN)");
    for (int i = 0; i < 4; ++i) b[i] = key_dbl(hk[i]);
    if (!(std::isfinite(b[0]) && std::isfinite(b[1]) && std::isfinite(b[2]) && std::isfinite(b[3])))
      return pg_set_error(h, PG_ERR_INVALID, "pg_grid_build: coordinates must be finite");
  }

  // finite points can still span more than a double holds (-1e308 .. 1e308): no cell size bins that
  PG_REQUIRE(h, std::isfinite(b[2] - b[0]) && std::isfinite(b[3] - b[1]),
             "pg_grid_build: the coordinate span (%g x %g) overflows double", b[2] - b[0], b[3] - b[1]);

  // cell count is capped; a larger-than-asked cell only makes queries visit more cells (they
  // derive their ring radius from the actual cell size), never changes results.
  const double max_cells = std::min((double)(1 << 28), std::max(8.0 * (double)n, (double)(1 << 20)));
  double cell = cell_size;
  int64_t nx, ny, nys;
  while (true) {
    // backstop: after the span check above a finite span fits one cell long before the cell overflows, so this never
    // fires today; it keeps the loop from spinning should that check ever change
    PG_REQUIRE(h, std::isfinite(cell), "pg_grid_build: no finite cell size bins the span (%g x %g)", b[2] - b[0], b[3] - b[1]);
    const double fx = std::floor((b[2] - b[0]) / cell) + 1, fy = std::floor((b[3] - b[1]) / cell) + 1;
    const double fys = std::ceil(fy / PG_STRIP);
    // rows are padded to whole strips: the padded count may reach 4 x the cap for thin grids (< 2^30 either way)
    if (fx * fy <= max_cells && fx * fys * PG_STRIP <= 4.0 * max_cells) {
      nx = (int64_t)fx; ny = (int64_t)fy; nys = (int64_t)fys;
      break;
    }
    cell *= 2.0;
  }
  const int64_t cells = nx * nys * PG_STRIP;
  pg_grid& g = h->grid;
  g.n = n; g.n_query = n_query; g.nx = (int)nx; g.ny = (int)ny; g.nys = (int)nys;
  g.x0 = b[0]; g.y0 = b[1]; g.cell = cell; g.inv_cell = 1.0 / cell; g.has_gid = gid != nullptr;

  int rc;
  const size_t cc_need = (cells + 4) * sizeof(int32_t);
  if (cc_need > h->cell_count.cap) h->cell_count_clean = false;
  if ((rc = pg_reserve(h, h->cell_count, cc_need))) return rc;
  const size_t cs_need = (cells + 8) * sizeof(int32_t);
  if (cs_need > h->cell_start.cap) {
    if ((rc = pg_reserve(h, h->cell_start, cs_need))) return rc;
    PG_CUDA(h, cudaMemsetAsync(h->cell_start.p, 0, 16, s));  // B[0] = 0 (and the alignment pad) once per allocation
  }
  if ((rc = pg_reserve(h, h->s_rec, (size_t)(n + 2) * sizeof(pg_rec)))) return rc;
  if (gid && (rc = pg_reserve(h, h->s_gid, (size_t)(n + 4) * sizeof(int32_t)))) return rc;
  h->last_count.valid = false;
  const bool aligned32 = ((uintptr_t)xy & 31) == 0;
  int32_t* B = (int32_t*)h->cell_start.p + 3;  // B[0] = 0, B + 1 is 16-byte aligned for the scan

  // the histogram is all zero between builds: the scan below clears every counter it reads
  if (!h->cell_count_clean) {
    PG_CUDA(h, cudaMemsetAsync(h->cell_count.p, 0, h->cell_count.cap, s));
    h->cell_count_clean = true;
  }
  if (n > 0) {
    PG_LAUNCH(h, s, "histogram_kernel", pg_launch_pdl(0, histogram_kernel, pg_div_up(n, TPB * PTS), TPB, s,
        (const double2*)xy, n, aligned32, g.x0, g.y0, g.inv_cell, g.nx, g.ny, (int32_t*)h->cell_count.p,
        (int32_t*)((char*)h->misc.p + PG_MISC_BADINPUT), h->build_epoch));
    PG_LAUNCH_CHECK(h);
  }
  if ((rc = pg_scan_i32(h, (const int32_t*)h->cell_count.p, B + 1, (int32_t)cells, s, nullptr, true))) {
    h->cell_count_clean = false;
    return rc;
  }
  if (n > 0) {
    PG_LAUNCH(h, s, "scatter_kernel", pg_launch_pdl(2, scatter_kernel, pg_div_up(n, TPB * PTS), TPB, s,
        (const double2*)xy, type, gid, n, aligned32, g.x0, g.y0, g.inv_cell, g.nx, g.ny, B + 1, (pg_rec*)h->s_rec.p,
        gid ? (int32_t*)h->s_gid.p : nullptr));
    PG_LAUNCH_CHECK(h);
  }
  g.built = true;
  return PG_OK;
}

int pg_grid_check(pg_handle* h) {
  if (!h) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  PG_CUDA(h, cudaMemcpyAsync(&h->pinned[8], (char*)h->misc.p + PG_MISC_BADINPUT, sizeof(int32_t), cudaMemcpyDeviceToHost, h->last_stream));
  PG_CUDA(h, cudaStreamSynchronize(h->last_stream));
  return pg_check_input_flag(h);
}

int pg_grid_info(pg_handle* h, int32_t* nx, int32_t* ny, double* x0, double* y0, double* cell) {
  if (!h) return PG_ERR_INVALID;
  if (!h->grid.built) return pg_set_error(h, PG_ERR_STATE, "pg_grid_info: no grid built");
  if (nx) *nx = h->grid.nx;
  if (ny) *ny = h->grid.ny;
  if (x0) *x0 = h->grid.x0;
  if (y0) *y0 = h->grid.y0;
  if (cell) *cell = h->grid.cell;
  return PG_OK;
}

}  // extern "C"
