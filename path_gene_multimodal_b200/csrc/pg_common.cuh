// Internal header of libpathgraph.so (sm_100a). Public ABI: include/pathgraph.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <cstdio>
#include "pathgraph.h"

#define PG_WARP 32

struct pg_buf {
  void* p = nullptr;
  size_t cap = 0;
};

// Grid (uniform bins) state kept between pg_grid_build and the queries.
struct pg_grid {
  bool built = false;
  int32_t n = 0, n_query = 0;
  int32_t nx = 0, ny = 0;  // logical cell columns / rows
  int32_t nys = 0;         // strips of PG_STRIP rows (rows are padded up to nys * PG_STRIP; the padding cells are empty)
  double x0 = 0, y0 = 0, cell = 0, inv_cell = 0;
  bool has_gid = false;
};

struct pg_handle {
  int device = 0;
  std::string err;
  // grow-only workspace
  pg_buf cell_count;   // int32 [C+1] histogram; all zero between builds (the scan clears what it reads)
  bool cell_count_clean = false;
  pg_buf cell_start;   // int32 [3 pad | 0 | C+1]: scan output lands one slot late, the scatter's cursor
                       // atomics turn it into the start-of-cell array in place (see pg_grid.cu)
  pg_buf cell_of;      // scratch (K7 staging columns)
  pg_buf rank;         // scratch (K7 staging weights)
  pg_buf s_rec;        // pg_rec [N]    points in cell order, one 32-byte sector each (see pg_query.cuh)
  pg_buf s_pos;        // unused (the walk writes its per-point records in row order)
  pg_buf s_gid;        // int32 [N]     copy of the caller's gids (only when given), for the fill pass
  // radius graph (pg_radius.cu): the walk leaves one 32-byte pg_pt_meta per point IN CELL ORDER (coalesced) and
  // parks the accepted entries of each row in tmp_ent; the row pass un-permutes the meta records into row order
  // (row_ptr scan, degree, type counts, statistics, row_off); the fill pass gathers the parked entries.
  pg_buf pt_meta;      // pg_pt_meta [N]
  pg_buf tmp_ent;      // pg_tmp_ent [tmp_cap]: one fixed region per walk CTA, then a shared overflow region
  pg_buf row_off;      // int32 [n_query] offset of row i's entries in tmp_ent (-1: never parked)
  int64_t tmp_cap = 0;        // entries tmp_ent can hold
  int32_t tmp_cta_cap = 0;    // entries in one CTA's region
  int64_t tmp_ovf_base = 0;   // first entry of the overflow region
  int64_t tmp_hint = 0;       // entries a past count pass produced in total (sizes the CTA regions)
  int64_t tmp_ovf_hint = 0;   // entries the overflow region must hold (a past pass's need / the caller's capacity)
  struct {             // arguments of the last count pass, kept so that it can be redone if tmp_ent was too small
    bool valid = false;
    double r = 0; int32_t flags = 0; int32_t* row_ptr = nullptr; int32_t* degree = nullptr; int32_t* nbr_count = nullptr;
    int32_t n_types = 0; pg_degree_stats* stats = nullptr; int32_t* hist = nullptr; int32_t hist_len = 0;
    // pg_radius_graph: the fill pass fused into the row pass (outputs known at count time)
    bool fused = false; int32_t* col = nullptr; float* dist32 = nullptr; double* dist64 = nullptr; int64_t* edges = nullptr;
    int32_t* edges32 = nullptr;
    int64_t capacity = 0;
  } last_count;
  pg_buf knn_retry;    // int32 [N]     cell-order positions of the points the kNN block pass could not finish
  pg_buf row_count;    // int32 [N+1]   per-row counts before the scan (K7)
  pg_buf scan_state;   // scan descriptors + ticket
  pg_buf misc;         // bounds / flags / cursors
  pg_buf sym_extra;    // int32 [N] K7: undirected row counts, then (cleared by the scan) the push cursor
  pg_buf sym_cursor;   // int32 [N] K7: per-row counts of entries above the row id (the i<j edge list), when asked for
  pg_buf sym_recip;    // uint8 [N*k]
  int32_t* pinned = nullptr;  // host-pinned: [0]=radius total [1]=sym total [2]=upper total [3]=overflow [4..]=scratch
  uint32_t scan_epoch = 0;
  int32_t build_epoch = 0;    // pg_grid_build counter (tags PG_MISC_BADINPUT)
  pg_grid grid;
  double radius_r = 0;
  int32_t radius_flags = 0;
  cudaStream_t last_stream = nullptr;
  int32_t sm_count = 148;
  int32_t contour_labels = -1;   // labels of the last pg_instance_contours_count (-1: none), for the fill call
  bool contour_empty = false;
  int64_t contour_raw = 0;
  size_t morph_smem_set[2][3] = {{0, 0, 0}, {0, 0, 0}};  // K1: dynamic shared memory opted in on this handle's device, per [T][EXTRA]
  double morph_mean_verts = 0;  // pg_map_morph_hint: expected vertices per ring (sizes K1's shared-memory slabs)
  pg_buf hull;         // K14 (pg_hull.cu): chain buffers of the rings that do not fit a warp's slab
  size_t hull_smem_set[2] = {0, 0};  // K14: dynamic shared memory opted in on this handle's device, per T
  pg_buf enrich_lab;   // K15 (pg_enrich.cu): uint8 labels of one chunk of permutations, [rows][n]
  pg_buf enrich_cnt;   // K15: int64 ordered type-pair counts per labelling, [P + 1][T * T]
  pg_buf ac_z;         // K17 (pg_autocorr.cu): centred feature values, node-major groups of 4 columns, [G][n] double4
  pg_buf ac_idx;       // K17: int32 pi_p(i) of one chunk of labellings, [rows][n]
  pg_buf ac_deg;       // K17: int32 in-range entries per row
  pg_buf ac_sims;      // K17: float64 statistic per labelling and column, [P + 1][n_feat] (row 0 = observed)
  pg_buf ac_part;      // K17: float64 CTA partials of the fixed-order reductions
  pg_buf ac_misc;      // K17: pg_ac_misc (column means / m2, S0-S2, integer degree sums) + CTA tickets
  // launch accounting / optional per-kernel CUDA-event timing (pg_profile_*)
  int64_t launches = 0;
  bool profiling = false;
  struct prof_rec { const char* name; cudaEvent_t e0, e1; };
  std::vector<prof_rec> prof;
};

// Brackets one kernel launch: counts it and, when profiling is on, records CUDA events on the
// launching stream around it.
struct pg_kernel_scope {
  pg_handle* h; cudaStream_t s; bool on;
  pg_kernel_scope(pg_handle* h_, cudaStream_t s_, const char* name) : h(h_), s(s_), on(h_->profiling) {
    h->launches += 1;
    if (on) {
      pg_handle::prof_rec r; r.name = name;
      cudaEventCreate(&r.e0); cudaEventCreate(&r.e1);
      cudaEventRecord(r.e0, s);
      h->prof.push_back(r);
    }
  }
  ~pg_kernel_scope() { if (on) cudaEventRecord(h->prof.back().e1, s); }
};
#define PG_LAUNCH(h, s, name, ...)              \
  do {                                          \
    pg_kernel_scope _pg_scope((h), (s), (name)); \
    __VA_ARGS__;                                \
  } while (0)

// misc buffer layout (byte offsets)
#define PG_MISC_BOUNDS 0      // 4 x uint64 ordered-encoded min/max
#define PG_MISC_OVERFLOW 64   // int32 overflow flag
#define PG_MISC_HALOCNT 80    // int32: records packed by the last pg_halo_push
#define PG_MISC_KNN_RETRY 76  // int32: points the kNN select pass handed to the ring pass
#define PG_MISC_BADINPUT 72   // int32: build epoch of the last pg_grid_build that met a non-finite coordinate
#define PG_MISC_TOTALS 128    // int32 x 8 totals copied to pinned memory: [0] radius [1] union [2] upper [3] contour scans; [4..5] uint64 overflow-region entries the last count pass needed
#define PG_MISC_TMPCUR 192    // uint64 allocation cursor of tmp_ent's overflow region (zero between count passes: the row pass moves it to TOTALS[4..5])
#define PG_MISC_SUM64 200     // int64: 64-bit total of the last pg_scan_i32_total (copied to pinned[12..13])
#define PG_MISC_PAIRHIST_TICKET 208  // uint64: point cursor of pair_hist_kernel's CTAs (zeroed before each launch)
#define PG_MISC_FEAT_TICKET 4608  // uint32 [PG_FEAT_MAX_COLS] CTA tickets of feature_stats_kernel, one per column (zero between launches)
#define PG_FEAT_MAX_COLS 256
#define PG_MISC_ACC 256       // pg_stats_acc: degree-statistics accumulators kept in their reset state
#define PG_MISC_ACC_HIST 512  // int32 [PG_ACC_HIST_MAX] histogram accumulators (all zero between launches)
#define PG_ACC_HIST_MAX 1024
#define PG_MISC_BYTES (PG_MISC_FEAT_TICKET + 4 * PG_FEAT_MAX_COLS)

// accumulators behind the fused degree statistics: every CTA adds its share, the last CTA to finish
// copies them to the caller's pg_degree_stats / hist and puts them back into the reset state, so no
// separate init / finish launches are needed.
struct pg_stats_acc {
  int32_t min_degree, max_degree;
  unsigned long long sum_degree, sumsq_degree, n_nodes;
  unsigned int done;  // CTAs finished
};

int pg_set_error(pg_handle* h, int code, const char* fmt, ...);
// after a stream synchronisation that followed the copy of PG_MISC_BADINPUT into h->pinned[8]
int pg_check_input_flag(pg_handle* h);
int pg_reserve(pg_handle* h, pg_buf& b, size_t bytes);

// Launch with programmatic dependent launch allowed: the grid may be scheduled while the kernel before it on the
// stream is still draining; it must execute pg_pdl_wait() before its first global-memory access (every kernel
// launched this way does so at its top), so only launch latency and the prologue overlap - no data hazard.
int pg_pdl_mask();  // PG_PDL_MASK environment variable (debugging aid): bit i allows it for kernels launched with tag i
template <class... KArgs, class... Args>
static inline cudaError_t pg_launch_pdl(int tag, void (*kernel)(KArgs...), int grid, int block, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = (pg_pdl_mask() >> tag) & 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

#define PG_CUDA(h, expr)                                                                      \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess)                                                                    \
      return pg_set_error((h), PG_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                   \
                          cudaGetErrorString(_e), __FILE__, __LINE__);                        \
  } while (0)

#define PG_LAUNCH_CHECK(h) PG_CUDA(h, cudaGetLastError())

#define PG_REQUIRE(h, cond, ...)                                       \
  do {                                                                 \
    if (!(cond)) return pg_set_error((h), PG_ERR_INVALID, __VA_ARGS__); \
  } while (0)

// internal scan entry (pg_scan.cu): out[0..n] exclusive prefix of in[0..n), out[n] = total
// total_copy (optional): a second device location that also receives the total
// clear_in: zero in[0..n) while reading it (the buffer must then be writable)
// publish: degree statistics to hand to the caller from the scan's first CTA (see pg_radius.cu)
struct pg_scan_publish {
  pg_stats_acc* acc = nullptr;   // NULL: no statistics to publish
  int32_t* acc_hist = nullptr;
  pg_degree_stats* stats = nullptr;
  int32_t* hist = nullptr;  // NULL: no histogram to publish
  int32_t hist_len = 0;
};
int pg_scan_i32(pg_handle* h, const int32_t* in, int32_t* out, int32_t n, cudaStream_t s, int32_t* total_copy = nullptr,
                bool clear_in = false, const pg_scan_publish* publish = nullptr);
// pg_scan_i32 of non-negative counts whose total the host needs: the total is also summed in 64 bits and read back
// into *total (synchronises the stream). PG_ERR_INVALID, naming `what`, when it is past INT32_MAX: the int32
// offsets would have wrapped.
int pg_scan_i32_total(pg_handle* h, const int32_t* in, int32_t* out, int32_t n, cudaStream_t s, int32_t* total_copy,
                      const char* what, int64_t* total);

static inline int pg_div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// Cell order. Cells are numbered strip by strip (a strip = PG_STRIP grid rows), column-major inside a strip:
//   c = ((cy / PG_STRIP) * nx + cx) * PG_STRIP + cy % PG_STRIP.
// Consecutive cells - and so consecutive points of the cell-ordered array - sweep a strip column by column,
// which keeps the neighbourhoods of a warp's / CTA's points in a compact, roughly square patch (L1 reuse),
// and the rows cy-1..cy+1 of one column are one contiguous run of the array unless they cross a strip edge.
#ifndef PG_STRIP_LOG
#define PG_STRIP_LOG 5
#endif
#define PG_STRIP (1 << PG_STRIP_LOG)

// compute-sanitizer is closed on the GPU pool this library is developed on, so the bounds it would check are
// asserted by hand in a -DPG_CHECK build (python -m path_gene_multimodal_b200._build with defines=("PG_CHECK=1",);
// the GPU tests are run once per round against that build: profiles/). Compiled out of the product.
#ifdef PG_CHECK
#include <cassert>
#define PG_ASSERT(cond) assert(cond)
#else
#define PG_ASSERT(cond) ((void)0)
#endif

#ifdef __CUDACC__
// programmatic dependent launch: let the next kernel on the stream be scheduled / wait for the previous one
__device__ __forceinline__ void pg_pdl_launch() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pg_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__host__ __device__ __forceinline__ int pg_cell_index(int nx, int cx, int cy) {
  return ((((cy >> PG_STRIP_LOG) * nx) + cx) << PG_STRIP_LOG) + (cy & (PG_STRIP - 1));
}

// cell coordinate along one axis: identical expression everywhere a point is binned.
__device__ __forceinline__ int pg_cell_coord(double v, double v0, double inv_cell, int n_cells) {
  double t = __dmul_rn(__dsub_rn(v, v0), inv_cell);
  int c = __double2int_rd(t);  // NaN -> 0, saturating
  c = c < 0 ? 0 : c;
  c = c >= n_cells ? n_cells - 1 : c;
  return c;
}

// squared distance exactly as scipy's sqeuclidean_distance_double evaluates it for m = 2 on a
// non-FMA build: fl(fl(dx*dx) + fl(dy*dy)). Intrinsics forbid FMA contraction.
__device__ __forceinline__ double pg_dist2(double ax, double ay, double bx, double by) {
  double dx = __dsub_rn(ax, bx);
  double dy = __dsub_rn(ay, by);
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
}
#endif
