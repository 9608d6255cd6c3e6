/*
 * pathgraph.h - C ABI of libpathgraph.so (sm_100a), the B200-native hot path of
 * himangi2003/path_gene_multimodal: nuclei table -> WSI space -> polygon morphology ->
 * kNN / radius spatial cell graph -> neighbour-type composition + degree statistics.
 *
 * The reference has no FFI of its own (pure Python); each entry point below replaces one
 * reference code block, cited as file:line into /root/reference.  The Python functions in
 * path_gene_multimodal_b200/ keep the reference's signatures / column names and call these
 * through ctypes (INTEGRATION.md shows the binding a maintainer would add).
 *
 * Conventions
 *  - every function returns 0 on success, a negative pg_status otherwise; pg_last_error()
 *    gives the text (owned by the library, valid until the next call on that handle).
 *  - all array arguments are DEVICE pointers owned by the caller unless marked "host";
 *    no allocation crosses the boundary; scratch lives in the grow-only per-handle workspace.
 *  - every call is asynchronous on `stream` except pg_create/pg_destroy, the *_total calls
 *    (they synchronise the stream to return a count) and workspace growth (cudaMalloc).
 *  - a handle is bound to one device and is not thread-safe; distinct handles are independent.
 *  - indices are int32 (N, M, E < 2^31); coordinates float64; there is no CPU fallback.
 */
#ifndef PATHGRAPH_H
#define PATHGRAPH_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pg_handle pg_handle;
typedef void* pg_stream; /* cudaStream_t */

typedef enum {
  PG_OK = 0,
  PG_ERR_INVALID = -1,   /* bad argument */
  PG_ERR_CUDA = -2,      /* CUDA runtime error, text in pg_last_error */
  PG_ERR_STATE = -3,     /* call order (e.g. query before pg_grid_build) */
  PG_ERR_CAPACITY = -4,  /* caller buffer smaller than the result */
  PG_ERR_NOMEM = -5
} pg_status;

/* flags of pg_radius_count */
#define PG_RADIUS_SYMMETRIC 0 /* rows hold every j != i with d <= r                          */
#define PG_RADIUS_UPPER 1     /* rows hold only j > i: the reference's `edges` list, i<j    */

#define PG_MAX_TYPES 16
#define PG_MAX_K 64

/* device-side degree statistics block (zeroed / initialised by the library) */
typedef struct {
  int32_t min_degree;
  int32_t max_degree;
  int64_t sum_degree;
  int64_t sumsq_degree;
  int64_t n_nodes;
} pg_degree_stats;

/* optional per-polygon outputs of pg_map_morph (any pointer may be NULL = not wanted) */
typedef struct {
  float* area;            /* |shoelace|; shapely p.area, polygon_morphology.py:247             */
  float* perimeter;       /* closed ring length; shapely p.length, polygon_morphology.py:248   */
  float* eccentricity;    /* sqrt(1 - l2/l1) of the second central moments; ipynb:2415-2429    */
  float* circularity;     /* 4 pi A / max(P,1)^2 = `compactness`; ipynb:2441-2443               */
  float* major_axis;      /* 4 sqrt(l1); ipynb:2423                                            */
  float* minor_axis;      /* 4 sqrt(l2); ipynb:2424                                            */
  double* centroid_x;     /* area centroid in WSI space; p.centroid, polygon_morphology.py:240 */
  double* centroid_y;
  double* poly_bbox;      /* [N,4] xmin,ymin,xmax,ymax of the shifted ring; p.bounds, :241     */
} pg_morph_out;

int pg_version(void);
int pg_create(int device, pg_handle** out);
int pg_destroy(pg_handle* h);
const char* pg_last_error(pg_handle* h); /* h may be NULL: error of the last failed pg_create */
/* bytes currently held by the handle's workspace */
int64_t pg_workspace_bytes(pg_handle* h);

/* ---- K1: fused tile->WSI shift + polygon morphology --------------------------------------
 * replaces add_wsi_coords_to_nuclei's numeric body (aggregated_hovernet_run.py:302-334) and the
 * shapely / cell-18 feature evaluation (polygon_morphology.py:240-248, ipynb:2415-2456).
 *   poly_off  int32 [N+1]   CSR offsets into poly_xy (vertex units)
 *   poly_xy   T     [M,2]   tile-local ring vertices, interleaved x,y; closing vertex optional
 *   nuc_tile  int32 [N]     tile index per nucleus (NULL = no shift)
 *   tile_x/y  int32 [n_tiles]
 *   centroid  f64   [N,2]   tile-local centroid (NULL = skip)   -> wsi_centroid f64 [N,2]
 *   bbox      int32 [N,4]   tile-local bbox     (NULL = skip)   -> wsi_bbox int32 [N,4]
 *   wsi_poly_xy T   [M,2]   shifted vertices (NULL = skip); a separate array: it must not overlap poly_xy
 *                           (the shift is not in place; wsi_poly_xy == poly_xy gives PG_ERR_INVALID)
 * Rows with < 3 vertices give NaN features. */
/* Optional: tell the library how long the rings of the coming pg_map_morph_* calls are (n rings, total_vertices
 * vertices), so that a warp's 32 rings fit its shared-memory staging slab; without it slabs are sized for rings of
 * up to 33 vertices and longer tables take the slower 8-lanes-per-ring path. Results do not depend on it. */
int pg_map_morph_hint(pg_handle* h, int32_t n, int64_t total_vertices);
int pg_map_morph_f32(pg_handle* h, int32_t n, const int32_t* poly_off, const float* poly_xy,
                     const int32_t* nuc_tile, const int32_t* tile_x, const int32_t* tile_y,
                     const double* centroid, const int32_t* bbox, float* wsi_poly_xy,
                     double* wsi_centroid, int32_t* wsi_bbox, const pg_morph_out* out,
                     pg_stream stream);
int pg_map_morph_f64(pg_handle* h, int32_t n, const int32_t* poly_off, const double* poly_xy,
                     const int32_t* nuc_tile, const int32_t* tile_x, const int32_t* tile_y,
                     const double* centroid, const int32_t* bbox, double* wsi_poly_xy,
                     double* wsi_centroid, int32_t* wsi_bbox, const pg_morph_out* out,
                     pg_stream stream);

/* ---- K2-K4: uniform-grid binning (atomic histogram, decoupled look-back scan, counting-sort
 * scatter); the cKDTree build of ipynb:1818 / ipynb:2964.
 *   xy     f64   [N,2]  coordinates (`coords`)
 *   type   int32 [N]    cell type ids (NULL = all 0)
 *   gid    int32 [N]    global ids used for tie-breaks / output columns (NULL = identity);
 *                       set when the points are a strip + halo of a larger slide
 *   n_query             only points with index < n_query are queried / own output rows
 *                       (the rest are halo points); pass N for a whole slide
 *   cell_size           > 0
 *   bounds  host f64[4] xmin,ymin,xmax,ymax (NULL = computed on the device; costs one sync) */
int pg_grid_build(pg_handle* h, int32_t n, int32_t n_query, const double* xy, const int32_t* type,
                  const int32_t* gid, double cell_size, const double* bounds, pg_stream stream);
/* Coordinates must be finite (cKDTree raises on NaN / inf). With bounds = NULL pg_grid_build itself reports it;
 * with caller-given bounds the build is asynchronous, the histogram kernel flags the offending input and
 * PG_ERR_INVALID comes from the next call that synchronises: pg_grid_check (synchronises the stream),
 * pg_radius_total or pg_check_overflow. A span that overflows double (xmax - xmin or ymax - ymin = inf for finite
 * points or bounds, e.g. -1e308 .. 1e308) is PG_ERR_INVALID from pg_grid_build itself. */
int pg_grid_check(pg_handle* h);
/* The points of the built grid in CELL ORDER (a spatial sort of the input, one coalesced pass over the records):
 * xy f64 [n,2], type int32 [n], gid int32 [n] = the id of each point (gid given to pg_grid_build, else its row);
 * any may be NULL. A caller that owns its row order (a strip of a sharded slide: rows are keyed by global id) feeds
 * these back in: every row-indexed access of the later passes - the walk's per-row records, the gather, the
 * neighbours' lists of the kNN union - then stays local. */
int pg_grid_export(pg_handle* h, double* xy, int32_t* type, int32_t* gid, pg_stream stream);
/* host-side view of the grid chosen: nx, ny, x0, y0, cell */
int pg_grid_info(pg_handle* h, int32_t* nx, int32_t* ny, double* x0, double* y0, double* cell);

/* ---- K5: kNN; KNN.from_array(coords, k) + neighbor_distances (ipynb:1815-1850).
 *   knn_idx  int32 [n_query,k] neighbour ids ascending by (d^2, id); self removed by index
 *   dist64   f64   [n_query,k] sqrt(dx*dx+dy*dy) (NULL = skip);  dist32 the same rounded to f32
 *   halo_ok  int32 [1] (NULL = skip) set to 0 if some queried point's k-th distance reaches past
 *            x_lo/x_hi (the region for which all points are present) - see sharding */
int pg_knn(pg_handle* h, int32_t k, int32_t* knn_idx, double* dist64, float* dist32,
           double x_lo, double x_hi, int32_t* halo_ok, pg_stream stream);

/* knn_neighbor_coords of cell 11 (ipynb:1838-1840, copied back at :1950): out_xy f64 [n_rows,k,2] = the
 * coordinates of every list entry, xy f64 [n_points,2] indexed by the ids in knn_idx (NaN for ids outside it). */
int pg_knn_neighbor_coords(pg_handle* h, int32_t n_rows, int32_t k, const int32_t* knn_idx, const double* xy,
                           int32_t n_points, double* out_xy, pg_stream stream);

/* ---- K6 (+K8 fused): radius graph, two-pass CSR; cKDTree.query_ball_tree + the i<j loop +
 * np.linalg.norm (ipynb:2964-2975, ipynb:3041-3042).
 * count pass: row_ptr int32 [n_query+1] (exclusive scan of per-row counts, total in the last slot),
 *   and fused over ALL neighbours regardless of `flags`:
 *   degree int32 [n_query] (NULL = skip), nbr_count int32 [n_query,n_types] for type ids 1..n_types
 *   (NULL = skip), stats (NULL = skip), hist int32 [hist_len] (last bin collects >= hist_len-1). */
int pg_radius_count(pg_handle* h, double r, int32_t flags, int32_t* row_ptr, int32_t* degree,
                    int32_t* nbr_count, int32_t n_types, pg_degree_stats* stats, int32_t* hist,
                    int32_t hist_len, pg_stream stream);
/* optional, before pg_radius_count: announces how many entries the count pass will have to hold (the caller's
 * output capacity), so that a sequence enqueued without ever asking for the total cannot run out of scratch */
int pg_radius_reserve(pg_handle* h, int64_t entries);
/* synchronises `stream`, returns row_ptr[n_query] of the last count pass */
int pg_radius_total(pg_handle* h, int64_t* total);
/* fill pass: col int32 [capacity] ascending per row, dist32 / dist64 (either may be NULL),
 * edges_i64 int64 [capacity,2] rows (i, j) (NULL = skip; the notebook's `edges` when flags=UPPER);
 * edges_i32 the same rows as int32 [capacity,2] (NULL = skip) - half the bytes for callers that move
 * the edge list over PCIe and widen it where it is consumed.
 * With flags=UPPER and the exact total n_edges = E (from pg_radius_total) the notebook's packed
 * tensors can be written directly: edge_index int64 [2,2E] = hstack(edges.T, edges[:, ::-1].T)
 * (ipynb:3021) and edge_attr float32 [2E] = concat(d, d) (ipynb:3041-3042); NULL = skip.
 * Rows that would pass `capacity` are dropped and pg_check_overflow reports it. */
int pg_radius_fill(pg_handle* h, const int32_t* row_ptr, int32_t* col, float* dist32, double* dist64,
                   int64_t* edges_i64, int32_t* edges_i32, int64_t* edge_index, float* edge_attr,
                   int64_t n_edges, int64_t capacity, pg_stream stream);

/* The same graph in ONE call when the caller provides the outputs up front (capacity in entries): the fill pass
 * runs inside the row pass of the count (each CTA gathers the rows it has just scanned), so row offsets never
 * travel through memory and one launch disappears. Rows that do not fit `capacity` are dropped and reported by
 * pg_check_overflow; the valid prefix of col / dist / edges is row_ptr[n_query]. edge_index / edge_attr need the
 * exact total and stay with pg_radius_count + pg_radius_total + pg_radius_fill. */
int pg_radius_graph(pg_handle* h, double r, int32_t flags, int32_t* row_ptr, int32_t* degree,
                    int32_t* nbr_count, int32_t n_types, pg_degree_stats* stats, int32_t* hist,
                    int32_t hist_len, int32_t* col, float* dist32, double* dist64, int64_t* edges_i64,
                    int32_t* edges_i32, int64_t capacity, pg_stream stream);
/* synchronises; PG_ERR_CAPACITY if any fill since the last check overflowed its buffers */
int pg_check_overflow(pg_handle* h);

/* ---- K7: undirected union of the directed kNN lists; nx.Graph loop of ipynb:1865-1894.
 * count: und_row_ptr int32 [N+1]; fill: und_col ascending per row, weights = min over directions.
 * The lists hold ids; for a whole slide ids are row numbers (row_id = id_map = NULL). For a strip +
 * halo, row_id int32 [n] gives the (global) id of each row and id_map int32 [n_ids] the row of an
 * id (-1 = not present); neighbours without a row only contribute their forward entry. */
int pg_knn_symmetrize_count(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx,
                            const int32_t* row_id, const int32_t* id_map, int32_t n_ids,
                            int32_t* und_row_ptr, pg_stream stream);
int pg_knn_symmetrize_total(pg_handle* h, int64_t* total);
int pg_knn_symmetrize_fill(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx,
                           const double* dist64, const float* dist32, const int32_t* row_id,
                           const int32_t* id_map, const int32_t* und_row_ptr, int32_t* und_col,
                           double* und_w64, float* und_w32, pg_stream stream);

/* The same union with the downstream passes fused into it (what build_knn_graph needs in one go): give
 * pg_knn_union_count an up_row_ptr int32 [n+1] and it also scans, per row, the entries above the row's id; then
 * pg_knn_union_fill writes - besides the symmetric CSR - the i<j edge list of ipynb:1894 / :2969-2975 (edges int64
 * [E_und][2] sorted by (i, j), weights), the neighbour-type composition (type int32 indexed by COLUMN id, nbr_count
 * int32 [n][n_types]), the degree and its statistics, from the same rank pass.  Every pointer of pg_union_out may be
 * NULL.  pg_knn_union_total returns both totals (one host synchronisation). */
typedef struct {
  int64_t* edges;
  double* edge_w64;
  float* edge_w32;
  const int32_t* type;
  int32_t n_types;
  int32_t* nbr_count;
  int32_t* degree;
  pg_degree_stats* stats;
  int32_t* hist;
  int32_t hist_len;
  int32_t symmetric_dist; /* non-zero: dist(i->j) == dist(j->i) bit for bit (true for lists made by pg_knn on one
                           * coordinate set), so the weight = min over both directions needs no reverse lookup */
  int32_t presized;       /* non-zero: the caller sized und_col / und_w / edges by their bounds (2 k n entries, k n
                           * edges) without reading the totals; the fill pass then sizes its scratch by the same bound
                           * and never synchronises - the whole count + fill sequence is one enqueue */
} pg_union_out;
int pg_knn_union_count(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx, const int32_t* row_id,
                       const int32_t* id_map, int32_t n_ids, int32_t* und_row_ptr, int32_t* up_row_ptr,
                       pg_stream stream);
int pg_knn_union_total(pg_handle* h, int64_t* total, int64_t* upper_total);
int pg_knn_union_fill(pg_handle* h, int32_t n, int32_t k, const int32_t* knn_idx, const double* dist64,
                      const float* dist32, const int32_t* row_id, const int32_t* id_map,
                      const int32_t* und_row_ptr, const int32_t* up_row_ptr, int32_t* und_col,
                      double* und_w64, float* und_w32, const pg_union_out* extra, pg_stream stream);

/* ---- symmetric CSR (rows ascending by column) -> `edges` (i<j) list; ipynb:2969-2975 / G.edges of
 * ipynb:1894.  row_id int32 [n] = id of each row in column space (NULL = identity; set for strips). */
int pg_csr_upper_count(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col,
                       const int32_t* row_id, int32_t* up_ptr, pg_stream stream);
int pg_csr_upper_total(pg_handle* h, int64_t* total);
int pg_csr_upper_fill(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col,
                      const double* w64, const float* w32, const int32_t* row_id,
                      const int32_t* up_ptr, int64_t* edges_i64, double* ew64, float* ew32,
                      pg_stream stream);

/* ---- K8: neighbour-type composition + degree statistics over any CSR (README.md:127,136; A.5) */
int pg_compose_degree(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col,
                      const int32_t* type, int32_t n_types, int32_t* nbr_count, int32_t* degree,
                      pg_degree_stats* stats, int32_t* hist, int32_t hist_len, pg_stream stream);

/* ---- K9: halo selection for strip-sharded slides (no reference counterpart; SURVEY 8e; csrc/pg_shard.cu).
 * Packs the points with x < lo_edge or x >= hi_edge into 24-byte records {x, y, gid, type}
 * (order unspecified); count_out int32 [1] device.  capacity in records. */
typedef struct {
  double x, y;
  int32_t gid, type;
} pg_halo_rec;
int pg_halo_pack(pg_handle* h, int32_t n, const double* xy, const int32_t* type, const int32_t* gid,
                 double lo_edge, double hi_edge, pg_halo_rec* out, int32_t capacity,
                 int32_t* count_out, pg_stream stream);

/* Device-side exchange steps of the strip sharding (K9, csrc/pg_shard.cu).
 * pg_strip_partition: out = the n points as 24-byte records grouped by owning strip (strip q owns x in
 *   [inner_edges[q-1], inner_edges[q]); inner_edges host f64 [n_strips-1] ascending), input order kept inside every
 *   strip; totals int32 [n_strips] device = records per strip (the send counts of the all-to-all).
 * pg_halo_unpack_multi: appends to xy/type/gid, starting at slot n_base, the records of `recs` whose x lies in an
 *   x-range [x_lo, x_hi) of ranges (host f64 [n_ranges][2], appended in that order) in one enqueue; recs
 *   skip_begin..skip_end-1 are this rank's own contribution and are ignored. counts_out int32 [n_ranges] device =
 *   number appended per range.
 * pg_gid_maps: id_map int32 [n_ids] = row of every global id among the first n_rows points (-1 elsewhere) and
 *   type_by_gid int32 [n_ids] = type of every id among all n points (0 elsewhere); either may be NULL. */
int pg_strip_partition(pg_handle* h, int32_t n, const double* xy, const int32_t* type, const int32_t* gid,
                       int32_t n_strips, const double* inner_edges, pg_halo_rec* out, int32_t* totals,
                       pg_stream stream);
int pg_halo_unpack_multi(pg_handle* h, const pg_halo_rec* recs, int32_t n_recs, int32_t skip_begin,
                         int32_t skip_end, int32_t n_ranges, const double* ranges, double* xy, int32_t* type,
                         int32_t* gid, int32_t n_base, int32_t capacity, int32_t* counts_out, pg_stream stream);
int pg_gid_maps(pg_handle* h, int32_t n, int32_t n_rows, const int32_t* gid, const int32_t* type, int32_t n_ids,
                int32_t* id_map, int32_t* type_by_gid, pg_stream stream);
/* Compact staging of contour vertices (the f1 "table files" row): skimage.measure.find_contours(mask, 0.5)
 * (aggregated_hovernet_run.py:185-197) leaves every vertex on the half-pixel lattice of its tile, so a table may carry
 * its polygons as int16 half-pixels (q = 2 * coordinate): 4 bytes per vertex over the host link instead of 8 / 16.
 * out[i] = 0.5f * in[i], exact; in / out 16-byte aligned. */
int pg_widen_halfpx(pg_handle* h, int64_t n_values, const int16_t* in, float* out, pg_stream stream);
/* The halo exchange as one step over NVLink peer memory (pack + all-gather fused; csrc/pg_shard.cu). Every rank owns a
 * receive slab of world x cap pg_halo_rec followed by world int32 counts, mapped into every rank (symmetric memory);
 * peer_ptrs_dev = device array of the world slab addresses as seen from this rank. pg_halo_push packs like
 * pg_halo_pack and stores each record straight into slot [rank][o] of every peer's slab, then publishes its count
 * (records beyond cap raise the overflow flag). After a barrier across the ranks, pg_halo_unpack_slab appends the
 * valid records of the local slab that fall into the x-ranges (as pg_halo_unpack_multi). */
int pg_halo_push(pg_handle* h, int32_t n, const double* xy, const int32_t* type, const int32_t* gid, double lo_edge,
                 double hi_edge, const uint64_t* peer_ptrs_dev, int32_t world, int32_t rank, int32_t cap,
                 pg_stream stream);
int pg_halo_unpack_slab(pg_handle* h, const void* slab, int32_t world, int32_t rank, int32_t cap, int32_t n_ranges,
                        const double* ranges, double* xy, int32_t* type, int32_t* gid, int32_t n_base,
                        int32_t capacity, int32_t* counts_out, pg_stream stream);
/* int32 counts (degree, nbr_count) -> uint8 (bits = 8) or uint16 (bits = 16) before they cross PCIe; a value that
 * does not fit is stored saturated and reported by pg_check_overflow. */
int pg_narrow_counts(pg_handle* h, const int32_t* src, int64_t n, void* dst, int32_t bits, pg_stream stream);

/* ---- K11: graph statistics the reference names (README.md:133-136 "cell-cell interaction patterns",
 * "degree, clustering, centrality"; SURVEY 8f-4) over a symmetric CSR with ascending rows (K6 / K7 output).
 * triangles int32 [n] (through node i), coeff float64 [n] = 2 T / (d (d - 1)), 0 for d < 2 (networkx.clustering);
 * either may be NULL.  inter int64 [n_types][n_types]: inter[a][b] = directed edges from type a+1 to type b+1. */
int pg_clustering(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col,
                  int32_t* triangles, double* coeff, pg_stream stream);
int pg_type_interactions(pg_handle* h, int32_t n, const int32_t* type, const int32_t* nbr_count,
                         int32_t n_types, int64_t* inter, pg_stream stream);

/* ---- K15: neighbourhood enrichment (csrc/pg_enrich.cu): the type-interaction matrix of an undirected edge list
 * against the same counts under random relabelling of the nodes - the label-permutation z-score of
 * squidpy.gr.nhood_enrichment, which makes "cell-cell interaction patterns" (README.md:133) readable when one type
 * dominates the slide.
 *   edges int32 [n_edges][2] rows (i, j) (build_radius_graph / build_knn_graph's i<j list; any order works); a row
 *         with an id outside [0, n) is skipped, as pg_clustering skips foreign ids. 4-byte alignment suffices.
 *   type  int32 [n]; labels outside 1..n_types count nowhere (but are permuted like every other label).
 * Counting: for a labelling t every edge row (i, j) adds 1 to c[t_i - 1][t_j - 1] and 1 to c[t_j - 1][t_i - 1] (the
 *   directed entries of the symmetric adjacency, squidpy's counting); with the original types c equals
 *   pg_type_interactions of the same graph's composition.
 * Permutation p (0 <= p < n_perms): node i gets the label type[pi_p(i)], pi_p a keyed bijection of [0, n):
 *   h = the least h >= 1 with 4^h >= n; a value x < 4^h is split into L = x >> h, R = x & (2^h - 1);
 *   8 Feistel rounds r = 0..7: (L, R) <- (R, L ^ (splitmix64(R ^ k_{p,r}) & (2^h - 1))),
 *     k_{p,r} = splitmix64(seed ^ (64 p + r));  x <- (L << h) | R;
 *   cycle-walk: repeat the 8 rounds until x < n.  pi_p(i) = that x.
 *   splitmix64(x) (uint64 arithmetic mod 2^64): z = x + 0x9E3779B97F4A7C15; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9;
 *     z = (z ^ (z >> 27)) * 0x94D049BB133111EB; return z ^ (z >> 31).
 *   For h >= 2 a Feistel network only reaches even permutations of its 4^h domain, so for a handful of nodes the
 *   family is visibly not the whole symmetric group; the count statistics match uniform permutations from n ~ 20 on.
 * Statistics, per (a, b), from S1 = sum_p c_p (int64) and S2 = sum_p c_p^2 (128-bit), exact integers each converted
 *   to float64 once:  perm_mean = S1 / P;  perm_std = sqrt(P S2 - S1^2) / P (ddof 0);
 *   zscore = (P count - S1) / sqrt(P S2 - S1^2) - NaN / +-inf where the permutation variance is 0 (IEEE division).
 * n = 0 or n_edges = 0: zero counts, mean and std 0, NaN zscore.  Only integer atomics: the outputs do not depend on
 * the run, the chunking or the handle.  Outputs [n_types][n_types], each pointer may be NULL.  Asynchronous; no host
 * synchronisation beyond workspace growth (labels of at most PG_ENRICH_CHUNK_BYTES / n permutations at a time, and
 * 8 (n_perms + 1) n_types^2 bytes of counts).  PG_ERR_INVALID for n < 0, n_edges < 0, n_types outside
 * 1..PG_MAX_TYPES, n_perms outside 1..PG_ENRICH_MAX_PERMS. */
#define PG_ENRICH_MAX_PERMS 100000
#define PG_ENRICH_CHUNK_BYTES (64 << 20)
typedef struct {
  int64_t* count;     /* observed directed counts */
  double* zscore;
  double* perm_mean;
  double* perm_std;
} pg_enrich_out;
int pg_nhood_enrichment(pg_handle* h, int32_t n, const int32_t* type, int32_t n_types, int64_t n_edges,
                        const int32_t* edges, int32_t n_perms, uint64_t seed, const pg_enrich_out* out,
                        pg_stream stream);

/* ---- K16: type-pair distance histogram over the built grid (csrc/pg_pairhist.cu): the counts behind
 * squidpy.gr.co_occurrence and Ripley's K / L - "cell-cell interaction patterns" (README.md:133) read across distance.
 *   thresholds host f64 [n_thr], finite, >= 0, strictly ascending; 1 <= n_thr <= PG_PAIRHIST_MAX_THR (64)
 *   hist  int64 [n_thr][n_types][n_types]: hist[b][a-1][c-1] = ordered pairs (i, j), i a query row (< n_query),
 *         j any grid point, id_i != id_j, type_i = a, type_j = c, with
 *           b = 0:  d2 <= t_0^2;   b >= 1:  t_{b-1}^2 < d2 <= t_b^2   (pairs past t_{n_thr-1} count nowhere)
 *         d2 = __dadd_rn(__dmul_rn(dx,dx), __dmul_rn(dy,dy)), t_b^2 rounded once in float64 (the radius rule).
 *   type_count int64 [n_types] (may be NULL): query rows of each type.
 * Types outside 1..n_types count nowhere. Integer counts only, so the result does not depend on the run.
 * The walk covers the ball of t_{n_thr-1} on whatever cell the grid was built with (a grid built for a small radius
 * works at a large one, only slower); work is n_query x the points of the (2R+1)^2 block, R = t_max / cell rounded up.
 * With ids (gid) and n_query set for a strip + halo of t_max, the strips' histograms sum to the whole slide's.
 * Asynchronous, no host synchronisation. hist / type_count 8-byte aligned. */
#define PG_PAIRHIST_MAX_THR 64
int pg_pair_dist_hist(pg_handle* h, int32_t n_types, int32_t n_thr, const double* thresholds,
                      int64_t* hist, int64_t* type_count, pg_stream stream);

/* ---- K17: spatial autocorrelation of per-nucleus features over a cell graph (csrc/pg_autocorr.cu): Moran's I or
 * Geary's C of every feature column with permutation statistics - squidpy.gr.spatial_autocorr's statistic - which asks
 * whether a measurement (area, eccentricity, neighbour composition...) is spatially clustered on the slide.
 *   row_ptr int32 [n+1], col int32 [row_ptr[n]]: a symmetric CSR without duplicate entries (build_radius_graph's
 *           symmetric_csr / build_knn_graph's union); entries with col outside [0, n) are skipped, as pg_clustering
 *           skips them, and do not count in any degree.
 *   feat    float64 [n_feat][n] (K10's layout), 1 <= n_feat <= PG_AUTOCORR_MAX_FEAT.
 * Weights: d_i = the in-range entries of row i; w_ij = 1 per entry (binary) or 1 / d_i (PG_AUTOCORR_ROW_STD).
 *   S0 = sum w_ij, S1 = 1/2 sum (w_ij + w_ji)^2, S2 = sum_i (w_i. + w_.i)^2. Binary: S0 = sum d_i, S1 = 2 S0,
 *   S2 = 4 sum d_i^2, exact int64 sums each converted to float64 once. Row-standardised: S0 = the non-isolated nodes,
 *   S1 = 1/2 sum over entries (1/d_i + 1/d_j)^2, S2 = sum over non-isolated i of (1 + sum_{j in N(i)} 1/d_j)^2, float64.
 * Statistic of a column x: z = x - mean(x) over all n nodes, m2 = sum z_i^2;
 *   Moran  I = n sum_ij w_ij z_i z_j / (S0 m2);   Geary  C = (n - 1) sum_ij w_ij (z_i - z_j)^2 / (2 S0 m2)
 *   (Geary's sum is taken per entry, never through its cancelling expansion). m2 = 0 or S0 = 0 gives NaN.
 *   Analytic moments under normality, for the caller: Moran E = -1/(n-1), V = (n^2 S1 - n S2 + 3 S0^2) / ((n^2 - 1)
 *   S0^2) - E^2; Geary E = 1, V = ((2 S1 + S2)(n - 1) - 4 S0^2) / (2 (n + 1) S0^2).
 * Permutations: in labelling p (0 <= p < n_perms) node i takes the values x[pi_p(i)] of ALL columns at once (one
 *   shuffle per permutation shared by the features, squidpy's procedure); pi_p is K15's, bit for bit, for the same seed.
 *   The observed statistic is labelling "identity" and goes through the same arithmetic.
 * Outputs (each pointer may be NULL), per column f:
 *   stat [n_feat] float64; perm_mean, perm_var (ddof 0) [n_feat] float64 (NaN when n_perms = 0);
 *   n_ge [n_feat] int64 = #{p : stat_p >= stat} (0 for a NaN stat); sims [n_perms][n_feat] float64 = stat_p;
 *   s012 float64 [3] = S0, S1, S2.
 * Every float sum has a fixed order (a thread's share, a shuffle tree, the warps in index order, the CTA partials in
 * index order), so the outputs do not depend on the run, the chunking or the handle; no float atomics. A non-finite
 * value in a column makes that column's outputs NaN (n_ge 0) and touches no other column. Asynchronous: no host
 * synchronisation beyond workspace growth (32 n_feat/4 n bytes of centred values, int32 indices of at most
 * PG_AUTOCORR_CHUNK_BYTES / 4n permutations at a time, 8 (n_perms + 1) n_feat bytes of statistics). PG_ERR_INVALID for
 * n < 0, n_feat outside 1..PG_AUTOCORR_MAX_FEAT, n_perms outside 0..PG_ENRICH_MAX_PERMS, unknown flags, NULL inputs. */
#define PG_AUTOCORR_GEARY 1    /* Geary's C instead of Moran's I */
#define PG_AUTOCORR_ROW_STD 2  /* row-standardised weights w_ij = 1 / d_i instead of binary */
#define PG_AUTOCORR_MAX_FEAT 256
#define PG_AUTOCORR_CHUNK_BYTES (32 << 20)
typedef struct {
  double* stat;
  double* perm_mean;
  double* perm_var;
  int64_t* n_ge;
  double* sims;
  double* s012;
} pg_autocorr_out;
int pg_spatial_autocorr(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t n_feat,
                        const double* feat, int32_t flags, int32_t n_perms, uint64_t seed, const pg_autocorr_out* out,
                        pg_stream stream);

/* ---- K18: local indicators of spatial association (csrc/pg_lisa.cu): one value per node and feature column, which
 * says WHERE a feature clusters (immune hot spots, regions of large nuclei, the cold margin around them) where K17 says
 * whether. Local Moran's I_i (Anselin 1995; PySAL esda Moran_Local) or Getis-Ord Gi / Gi* z-scores (Ord & Getis 1995;
 * esda G_Local), with conditional permutation tests.
 *   row_ptr / col: a symmetric CSR as for K17. Entries with col outside [0, n) and self entries (col == i) are skipped:
 *           conditional randomisation keeps node i fixed (esda separates self weights for the same reason).
 *           d_i = the remaining entries of row i.
 *   feat    float64 [n_feat][n] (K10's layout), 1 <= n_feat <= PG_AUTOCORR_MAX_FEAT.
 * Weights: w = 1 (binary) or w = 1 / d_i (PG_AUTOCORR_ROW_STD). Per column, z = x - mean over all n nodes (K17's
 * centring, bit for bit), m2 = sum z^2.
 *   lag     S_i = sum_{j in N(i)} z_j in CSR entry order; L_i = S_i (binary) or S_i / d_i (row-standardised; 0 when
 *           d_i = 0).
 *   Moran   I_i = c z_i L_i, c = (n - 1) / m2 (esda's n_1 z lz / den).
 *   Gi*     (PG_LOCAL_GETIS_ORD | PG_LOCAL_STAR): the self term belongs to the neighbourhood. Binary: W_i = S1_i = d_i + 1,
 *           w_ii = w = 1; row-standardised: W_i = 1, S1_i = w_ii = w = 1 / (d_i + 1).
 *           Z_i = (w_ii z_i + w S_i) / (sqrt(m2 / n) sqrt((n S1_i - W_i^2) / (n - 1))).
 *   Gi      (PG_LOCAL_GETIS_ORD): binary W_i = S1_i = d_i; row-standardised W_i = 1, S1_i = 1 / d_i.
 *           N_i = L_i + W_i z_i / (n - 1), s_i^2 = (m2 - z_i^2 n / (n - 1)) / (n - 1),
 *           Z_i = N_i / (s_i sqrt(((n - 1) S1_i - W_i^2) / (n - 2)))
 *           (Ord & Getis's x(i) mean and S(i) over the other n - 1 values, rewritten on z so that nothing cancels).
 *   A quantity <= 0 under a square root, m2 = 0 or n too small for the formula (Gi*: n < 2, Gi: n < 3) gives NaN.
 * Draws: K = max d_i. Permutation p draws r_p[j] = pi'_p(j), j < K, pi'_p K15's keyed bijection (same round keys
 *   k_{p,r}) on [0, n - 1): a uniform K-subset in random order, the role of esda's permutation(n - 1)[:max_card]. Node i's
 *   j-th neighbour in permutation p is s = r_p[j] + (r_p[j] >= i) (never i itself); S_ip = sum_{j < d_i} z_s in ascending
 *   j, and stat_ip follows from S_ip through the same arithmetic as stat_i from S_i. All nodes and columns share the
 *   draws of a permutation.
 * Outputs, each pointer may be NULL, [n_feat][n] unless stated:
 *   stat, lag float64: I_i or Z_i, and L_i;
 *   n_ge int32 = #{p : stat_ip >= stat_i} (0 for a NaN stat or d_i = 0);
 *   perm_mean, perm_var float64 (ddof 0) from d1 = sum_p delta_p and d2 = sum_p delta_p^2, delta_p = stat_ip - stat_i,
 *     both in ascending p: perm_mean = stat_i + d1 / P, perm_var = max(0, d2 / P - (d1 / P)^2); NaN when n_perms = 0 or
 *     d_i = 0;
 *   sims float64 [n_perms][n_feat][n] = stat_ip (NaN where d_i = 0), for tests on small graphs;
 *   mean, m2 float64 [n_feat].
 * Isolated nodes (d_i = 0) keep the formula's statistic and get no permutation outputs. A non-finite value in a column
 * makes that column NaN (n_ge 0) and touches no other column. Every float sum has a fixed order and every node's
 * permutation sums live in one thread, so the outputs do not depend on the run or the handle; no float atomics.
 * Asynchronous: no host synchronisation beyond workspace growth (K17's 32 n_feat/4 n bytes of centred values, 12 n
 * bytes of degrees and degree order). PG_ERR_INVALID on K17's conditions, and PG_LOCAL_STAR without
 * PG_LOCAL_GETIS_ORD. */
#define PG_LOCAL_GETIS_ORD 4  /* Getis-Ord Gi instead of local Moran */
#define PG_LOCAL_STAR 8       /* Gi*: node i counts in its own neighbourhood */
typedef struct {
  double* stat;
  double* lag;
  int32_t* n_ge;
  double* perm_mean;
  double* perm_var;
  double* sims;
  double* mean;
  double* m2;
} pg_local_out;
int pg_local_autocorr(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t n_feat,
                      const double* feat, int32_t flags, int32_t n_perms, uint64_t seed, const pg_local_out* out,
                      pg_stream stream);

/* ---- K19: cell clusters (csrc/pg_cluster.cu): connected components and DBSCAN over a cell graph, and a table with
 * one row per cluster - the lymphocyte aggregates, tumour nests and stroma islands a pathologist counts.
 * pg_connected_components: any CSR, row_ptr int32 [n+1], col int32. Every entry (i, j) with j in [0, n) and j != i
 *   joins i and j; other entries are skipped, as pg_clustering skips them. A CSR that is not symmetric gives the weak
 *   components (scipy.sparse.csgraph.connected_components with directed=False).
 *   label int32 [n] = the rank of the node's component in the order of the components' smallest member (scipy's
 *   numbering); n_labels int32 [1] (device) = the components.
 * pg_dbscan: row_ptr / col the symmetric radius CSR of the points (K6 with flags 0: d2 <= eps^2, no self entries).
 *   d_i = the entries of row i with j in [0, n) and j != i; core_i = (d_i + 1 >= min_samples) (the point counts itself,
 *   as in sklearn). Only entries between two core nodes join. Clusters are numbered in the order of their smallest core
 *   node; label int32 [n] = the cluster of a core node; a non-core node takes the smallest label among its core
 *   neighbours, -1 (noise) when it has none. core uint8 [n] = core_i. n_labels int32 [1] (device) = the clusters.
 *   This is sklearn.cluster.DBSCAN's result exactly: its dbscan_inner visits the points in index order, starts a new
 *   cluster at each unlabelled core point and finishes that cluster (labelling every neighbour of its core points that
 *   has no label yet) before it starts the next. So the clusters get their labels in the order of their smallest core
 *   point, and a border point reachable from several clusters keeps the label of the first of them to reach it: the
 *   smallest label among its core neighbours.
 * Both: union-find (links only ever hang a root under a smaller root, so each root ends as its component's smallest
 *   member) and a scan of the roots; the labels do not depend on the run or the handle. Asynchronous, no host
 *   synchronisation beyond workspace growth (12 n bytes). PG_ERR_INVALID for n < 0, min_samples < 1, NULL pointers.
 * pg_cluster_props: the clusters 0..n_clusters-1 of label int32 [n] (n_labels of the calls above; a label outside
 *   [0, n_clusters) belongs to no cluster); xy float64 [n][2] (16-byte aligned); type int32 [n] (types outside
 *   1..n_types count nowhere); core uint8 [n]. Outputs per cluster c, each may be NULL:
 *     n_members int32 [K]; n_core int32 [K] (needs core); type_count int32 [K][n_types] (needs type);
 *     centroid float64 [K][2] = the coordinate sums / n_members, each sum taken in one fixed order over the members in
 *       ascending node index (lane l of a warp adds members l, l + 32, ... in turn, then a shuffle tree adds the lanes);
 *     bbox float64 [K][4] = xmin, ymin, xmax, ymax (NaN centroid and bbox for a cluster without members);
 *     member_off int32 [K+1], member_xy float64 [M][2] (16-byte aligned, M = member_off[K] = the members): the members'
 *       coordinates grouped by cluster in ascending node index - a polygon CSR that pg_ring_hull_f64 takes as it is.
 *   The grouping is a stable LSD counting sort on 8-bit digits of the label; every output position follows from counts
 *   and scans, none from the order of atomics, so the outputs do not depend on the run or the handle. Asynchronous, no
 *   host synchronisation beyond workspace growth (8 n + 4 K bytes and 8 max(K, 256 ceil(n / 2048)) bytes); the caller knows K
 *   from n_labels (one read-back, as pg_radius_total). PG_ERR_INVALID for n < 0, n_clusters < 0, n_types outside
 *   1..PG_MAX_TYPES, NULL required pointers. */
typedef struct {
  int32_t* n_members;
  int32_t* n_core;
  int32_t* type_count;
  double* centroid;
  double* bbox;
  int32_t* member_off;
  double* member_xy;
} pg_cluster_out;
int pg_connected_components(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t* label,
                            int32_t* n_labels, pg_stream stream);
int pg_dbscan(pg_handle* h, int32_t n, const int32_t* row_ptr, const int32_t* col, int32_t min_samples,
              int32_t* label, uint8_t* core, int32_t* n_labels, pg_stream stream);
int pg_cluster_props(pg_handle* h, int32_t n, const int32_t* label, int32_t n_clusters, const double* xy,
                     const int32_t* type, int32_t n_types, const uint8_t* core, const pg_cluster_out* out,
                     pg_stream stream);

/* ---- K12: raster region properties of an instance map (SURVEY 8f-3): what skimage regionprops gives
 * aggregated_hovernet_run.py:172-181 (bbox per instance) and hovernet_tile_inference.ipynb:2415-2429 (cell 18:
 * area, perimeter, eccentricity, major / minor axis length, orientation).  inst_map int32 [height][width], labels
 * 1..n_labels (0 = background; labels outside are ignored); every output is indexed by label - 1 and may be NULL.
 * bbox = {min_row, min_col, max_row + 1, max_col + 1}; centroid = {row, col}; absent labels: area 0, NaN features. */
typedef struct {
  int32_t* area;        /* [n_labels] */
  int32_t* bbox;        /* [n_labels][4] */
  double* centroid;     /* [n_labels][2] */
  double* perimeter;    /* [n_labels] */
  double* eccentricity;
  double* major_axis;
  double* minor_axis;
  double* orientation;
} pg_raster_out;
int pg_raster_props(pg_handle* h, int32_t height, int32_t width, const int32_t* inst_map,
                    int32_t n_labels, const pg_raster_out* out, pg_stream stream);

/* solidity = area / convex area (skimage regionprops: convex_hull_image of the region - the hull of the pixels' diamond
 * corners, rasterised with its border - cell 18's fourth property). area / bbox: pg_raster_props outputs of the same map.
 * convex_area int32 [n_labels], solidity float64 [n_labels] (NaN for absent labels); either may be NULL. Exact integer
 * arithmetic; one host synchronisation (workspace size). PG_ERR_INVALID when the workspace, sum 4 (2 rows + 1) over
 * the labels' boxes, is past INT32_MAX entries. */
int pg_raster_solidity(pg_handle* h, int32_t height, int32_t width, const int32_t* inst_map, int32_t n_labels,
                       const int32_t* area, const int32_t* bbox, int32_t* convex_area, double* solidity,
                       pg_stream stream);

/* ---- K14: per-ring convex hull (cell 18's `solidity` and `orientation`, ipynb:2415-2456, for the polygons K1 measures).
 *   poly_off   int32 [N+1]  CSR offsets into poly_xy (vertex units), as for pg_map_morph
 *   n_vertices              vertices in poly_xy (M); sizes the workspace of rings that do not fit a shared-memory slab
 *   poly_xy    T     [M,2]  ring vertices, interleaved x,y, any order or self-intersection; closing vertex optional
 * Outputs float64 [N], each may be NULL:
 *   convex_area  area of the convex hull of the ring's vertices (Andrew's monotone chain)
 *   solidity     |shoelace area| / convex_area
 *   orientation  skimage's: 0.5 atan2(-2b, c - a) with (a, b, c) = (mu_xx, -mu_xy, mu_yy) of the ring's area moments,
 *                x = column, y = row (+-pi/4 when a == c): pi/2 in magnitude for a ring long along x, 0 along y.
 * Rows with < 3 vertices give NaN everywhere; zero area gives NaN solidity / orientation; zero convex area gives
 * convex_area 0 and NaN solidity. Exact (float64 terms are integers / 4) for vertices on the half-pixel lattice. */
typedef struct {
  double* convex_area;
  double* solidity;
  double* orientation;
} pg_hull_out;
int pg_ring_hull_f32(pg_handle* h, int32_t n, int64_t n_vertices, const int32_t* poly_off, const float* poly_xy,
                     const pg_hull_out* out, pg_stream stream);
int pg_ring_hull_f64(pg_handle* h, int32_t n, int64_t n_vertices, const int32_t* poly_off, const double* poly_xy,
                     const pg_hull_out* out, pg_stream stream);

/* ---- K13: instance map -> one polygon per instance (SURVEY 8f-3): aggregated_hovernet_run.py:183-198 -
 * find_contours(inst_map == id, 0.5), the longest contour, (x, y) = (col, row), approximate_polygon(tolerance).
 * area / bbox are pg_raster_props outputs for the same map. count: poly_off int32 [n_labels + 1] (device, 16-byte
 * aligned; labels without pixels get empty rings); total: vertices to allocate (one host synchronisation, two more
 * inside count for the scratch); fill: poly_xy float64 [total][2], closed rings (first == last vertex) as skimage
 * returns them. Douglas-Peucker decisions are taken in exact integer arithmetic on the half-pixel lattice (a distance
 * equal to the tolerance is not "greater"; the first maximum splits) - skimage's float evaluation breaks such ties
 * by libm rounding. fill must follow its count on the same handle (the contours wait in the workspace). count
 * returns PG_ERR_INVALID when its scratch (visited bits: a quarter byte per square of every label's window; raw
 * contour vertices) is past INT32_MAX bytes / entries: many labels whose windows span a large map. */
int pg_instance_contours_count(pg_handle* h, int32_t height, int32_t width, const int32_t* inst_map,
                               int32_t n_labels, const int32_t* area, const int32_t* bbox, double tolerance,
                               int32_t* poly_off, pg_stream stream);
int pg_instance_contours_total(pg_handle* h, int64_t* total);
int pg_instance_contours_fill(pg_handle* h, int32_t n_labels, const int32_t* poly_off, double* poly_xy,
                              pg_stream stream);

/* ---- K10: node features for the GNN input (SURVEY 8f-2).  hovernet_tile_inference.ipynb:2903 (cell 21:
 * z = (v - mean) / std(ddof=0), NaN-skipping statistics, a column with sigma 0 / NaN becomes all 0.0) and
 * ipynb:2950 (cell 23: pd.get_dummies(type, prefix="type"), features = one-hot columns then the *_z columns).
 * feat float64 [n_feat][n] (one contiguous column per feature), type int32 [n], onehot_values int32 [n_onehot]
 * (the distinct type values, ascending) -> x float32 [n][n_onehot + n_feat] row-major, stats float64
 * [n_feat][2] = {mean, sigma} (device); n_feat <= 256.  Deterministic (pandas' two-pass mean / variance, fixed-order sums). */
int pg_node_features(pg_handle* h, int32_t n, int32_t n_feat, const double* feat, const int32_t* type,
                     const int32_t* onehot_values, int32_t n_onehot, float* x, double* stats,
                     pg_stream stream);

/* ---- launch accounting and per-kernel timing (CUDA events recorded on the launching stream) ----
 * pg_launch_count: kernels launched through this handle so far.
 * pg_profile_enable(1) starts recording one (name, start, stop) event pair per kernel launch and
 * clears earlier records; pg_profile_count synchronises the device and returns how many records
 * there are; pg_profile_get returns the kernel name (library-owned) and its duration in ms. */
int64_t pg_launch_count(pg_handle* h);
int pg_profile_enable(pg_handle* h, int on);
int pg_profile_count(pg_handle* h);
int pg_profile_get(pg_handle* h, int i, const char** name, float* ms);

/* ---- exclusive scan (decoupled look-back), exposed for tests: out[i] = sum in[0..i), out[n] = total */
int pg_exclusive_scan_i32(pg_handle* h, const int32_t* in, int32_t* out, int32_t n, pg_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* PATHGRAPH_H */
