// K13: instance map -> one polygon per instance (SURVEY 8f-3, second half).
// Reference: /root/reference/aggregated_hovernet_run.py:183-198 - per instance: mask = (inst_map == inst_id),
// find_contours(mask, 0.5), the longest contour, (x, y) = (col, row), approximate_polygon(tolerance = 0.5).
// The reference masks the whole tile once per instance and walks Python dictionaries; here one thread owns one
// instance and only ever looks at the 2x2 squares around its bounding box (from K12):
//   pass A  the marching-squares segments of the instance's mask form disjoint directed cycles (open chains only at
//           the image border). The squares are scanned in skimage's order; every segment not seen yet is followed
//           through its component (the successor of a segment is in the square across the edge it ends on), which
//           gives the component's length, its first and its last segment. skimage's dictionary bookkeeping
//           (_assemble_contours) reduces to: a cycle starts at the to-point of its LAST segment, contours are numbered
//           by their FIRST segment, max(key = len) takes the first longest (oracle/contours.py checks this closed form
//           against the literal bookkeeping).
//   pass B  the chosen contour is written out in doubled integer coordinates and simplified by Douglas-Peucker with
//           every decision in integer arithmetic (distance^2 as a fraction; a tie is "not greater"; the first maximum
//           splits). skimage evaluates the same decisions through arctan2 / sin / cos in floating point, where ties -
//           frequent on the half-pixel lattice - fall either way depending on libm: the exact rule is the one result
//           that does not depend on the platform (DESIGN.md, oracle/contours.py).
//   pass C  the kept vertices as float64 (x, y), CSR over the labels.
#include <algorithm>
#include "pg_common.cuh"

namespace {

constexpr int TPB = 128;
enum { E_T = 0, E_B = 1, E_L = 2, E_R = 3 };

__constant__ signed char c_nseg[16] = {0, 1, 1, 1, 1, 1, 2, 1, 1, 2, 1, 1, 1, 1, 1, 0};
// from / to edge of the (up to two) segments of every case, in skimage's append order
__constant__ signed char c_from[16][2] = {{-1, -1}, {E_T, -1}, {E_R, -1}, {E_R, -1}, {E_L, -1}, {E_T, -1}, {E_R, E_L}, {E_R, -1},
                                          {E_B, -1}, {E_T, E_B}, {E_B, -1}, {E_B, -1}, {E_L, -1}, {E_T, -1}, {E_L, -1}, {-1, -1}};
__constant__ signed char c_to[16][2] = {{-1, -1}, {E_L, -1}, {E_T, -1}, {E_L, -1}, {E_B, -1}, {E_B, -1}, {E_T, E_B}, {E_B, -1},
                                        {E_R, -1}, {E_L, E_R}, {E_T, -1}, {E_L, -1}, {E_R, -1}, {E_R, -1}, {E_T, -1}, {-1, -1}};

struct window {  // the squares (sr, sc) around one instance: sr in [sr0, sr0 + wh), sc in [sc0, sc0 + ww)
  int sr0, sc0, wh, ww;
};

__device__ __forceinline__ window make_window(const int32_t* bbox, int h, int w) {
  window x;
  x.sr0 = max(bbox[0] - 1, 0);
  x.sc0 = max(bbox[1] - 1, 0);
  x.wh = max(min(bbox[2] - 1, h - 2) - x.sr0 + 1, 0);
  x.ww = max(min(bbox[3] - 1, w - 2) - x.sc0 + 1, 0);
  return x;
}

struct walker {
  const int32_t* m;
  int h, w, lab;
  window win;
  __device__ __forceinline__ int square_case(int sr, int sc) const {
    const int32_t* p = m + (int64_t)sr * w + sc;
    return (p[0] == lab ? 1 : 0) | (p[1] == lab ? 2 : 0) | (p[w] == lab ? 4 : 0) | (p[w + 1] == lab ? 8 : 0);
  }
  __device__ __forceinline__ int sid_of(int sr, int sc, int sub) const { return (((sr - win.sr0) * win.ww + (sc - win.sc0)) << 1) | sub; }
  __device__ __forceinline__ void square_of(int sid, int& sr, int& sc, int& sub) const {
    const int idx = sid >> 1;
    sub = sid & 1;
    sr = win.sr0 + idx / win.ww;
    sc = win.sc0 + idx % win.ww;
  }
  // the segment that starts (FWD) where `sid` ends, or ends where it starts (!FWD); -1 at the image border
  template <bool FWD>
  __device__ __forceinline__ int step(int sid) const {
    int sr, sc, sub;
    square_of(sid, sr, sc, sub);
    const int k = square_case(sr, sc);
    const int e = FWD ? c_to[k][sub] : c_from[k][sub];
    int nr = sr, nc = sc, enter;
    if (e == E_T) { nr = sr - 1; enter = E_B; }
    else if (e == E_B) { nr = sr + 1; enter = E_T; }
    else if (e == E_L) { nc = sc - 1; enter = E_R; }
    else { nc = sc + 1; enter = E_L; }
    if (nr < 0 || nr > h - 2 || nc < 0 || nc > w - 2) return -1;
    const int k2 = square_case(nr, nc);
    const int s2 = (FWD ? c_from[k2][0] : c_to[k2][0]) == enter ? 0 : 1;
    return sid_of(nr, nc, s2);
  }
  // doubled (row, col) of the from / to point of a segment
  __device__ __forceinline__ int2 point(int sid, bool to) const {
    int sr, sc, sub;
    square_of(sid, sr, sc, sub);
    const int k = square_case(sr, sc);
    const int e = to ? c_to[k][sub] : c_from[k][sub];
    if (e == E_T) return make_int2(2 * sr, 2 * sc + 1);
    if (e == E_B) return make_int2(2 * sr + 2, 2 * sc + 1);
    if (e == E_L) return make_int2(2 * sr + 1, 2 * sc);
    return make_int2(2 * sr + 1, 2 * sc + 2);
  }
};

// visited bits needed by one instance (bytes)
__global__ void __launch_bounds__(TPB)
contour_window_kernel(const int32_t* __restrict__ area, const int32_t* __restrict__ bbox, int n_labels, int h, int w,
                      int32_t* __restrict__ bytes) {
  const int l = blockIdx.x * TPB + threadIdx.x;
  if (l >= n_labels) return;
  int b = 0;
  if (area[l] > 0) {
    const window x = make_window(bbox + 4 * l, h, w);
    b = (x.wh * x.ww * 2 + 7) >> 3;
  }
  bytes[l] = b;
}

struct pick {  // the contour chosen for one instance
  int start_seg;  // first segment of the raw contour (-1: none)
  int n_seg;      // segments = raw vertices - 1
};

__global__ void __launch_bounds__(TPB)
contour_pick_kernel(const int32_t* __restrict__ m, int h, int w, const int32_t* __restrict__ area,
                    const int32_t* __restrict__ bbox, int n_labels, const int32_t* __restrict__ vis_off,
                    uint8_t* __restrict__ vis, pick* __restrict__ picks, int32_t* __restrict__ n_raw) {
  const int l = blockIdx.x * TPB + threadIdx.x;
  if (l >= n_labels) return;
  pick best{-1, 0};
  if (area[l] > 0) {
    walker wk{m, h, w, l + 1, make_window(bbox + 4 * l, h, w)};
    uint8_t* v = vis + vis_off[l];
    const int n_sq = wk.win.wh * wk.win.ww;
    for (int b = 0; b < ((n_sq * 2 + 7) >> 3); ++b) v[b] = 0;
    auto seen = [&](int sid) { return (v[sid >> 3] >> (sid & 7)) & 1; };
    auto mark = [&](int sid) { v[sid >> 3] |= (uint8_t)(1u << (sid & 7)); };
    for (int idx = 0; idx < n_sq; ++idx) {
      const int sr = wk.win.sr0 + idx / wk.win.ww, sc = wk.win.sc0 + idx % wk.win.ww;
      const int ns = c_nseg[wk.square_case(sr, sc)];
      for (int sub = 0; sub < ns; ++sub) {
        const int sid = (idx << 1) | sub;
        if (seen(sid)) continue;
        // follow the component forwards from its first segment
        int len = 0, last = sid, cur = sid;
        bool closed = false;
        while (true) {
          mark(cur);
          ++len;
          last = max(last, cur);
          const int nx = wk.step<true>(cur);
          if (nx < 0) break;
          if (nx == sid) { closed = true; break; }
          cur = nx;
        }
        int start = sid;
        if (closed) {
          start = wk.step<true>(last);  // a cycle leaves skimage's bookkeeping starting right after its closing segment
        } else {                        // an open chain (image border): it starts where nothing precedes it
          cur = sid;
          while (true) {
            const int pv = wk.step<false>(cur);
            if (pv < 0) break;
            cur = pv;
            mark(cur);
            ++len;
          }
          start = cur;
        }
        if (len > best.n_seg) { best.start_seg = start; best.n_seg = len; }  // the first longest wins
      }
    }
  }
  picks[l] = best;
  n_raw[l] = best.start_seg >= 0 ? best.n_seg + 1 : 0;
}

// exact Douglas-Peucker over raw[0..n) (doubled integer coordinates); keep[] marks the surviving vertices;
// stack holds (start, end) pairs. tol2 = (2 * tolerance)^2 in doubled units.
__device__ int simplify(const int2* __restrict__ raw, int n, double tol2, uint8_t* __restrict__ keep, int2* __restrict__ stack) {
  for (int i = 0; i < n; ++i) keep[i] = 0;
  keep[0] = 1; keep[n - 1] = 1;
  int kept = n > 1 ? 2 : 1;
  int sp = 0;
  stack[sp++] = make_int2(0, n - 1);
  while (sp > 0) {
    const int2 se = stack[--sp];
    const int2 a = raw[se.x], b = raw[se.y];
    const long long dx = b.x - a.x, dy = b.y - a.y;
    const long long L2 = dx * dx + dy * dy;
    long long best_num = 0, best_den = 1;
    int best_i = -1;
    for (int i = se.x + 1; i < se.y; ++i) {
      const int2 p = raw[i];
      const long long pax = p.x - a.x, pay = p.y - a.y, pbx = p.x - b.x, pby = p.y - b.y;
      long long num, den;
      if (pax * dx + pay * dy > 0 && -(pbx * dx + pby * dy) > 0) {
        const long long cr = dx * pay - dy * pax;
        num = cr * cr; den = L2;
      } else {
        num = min(pax * pax + pay * pay, pbx * pbx + pby * pby); den = 1;
      }
      // num / den > best_num / best_den, dens in {1, L2}: never more than one L2 factor on either side
      bool greater;
      if (den == best_den) greater = num > best_num;
      else if (den == 1) greater = (unsigned long long)num * (unsigned long long)L2 > (unsigned long long)best_num;
      else greater = (unsigned long long)num > (unsigned long long)best_num * (unsigned long long)L2;
      if (best_i < 0 || greater) { best_num = num; best_den = den; best_i = i; }
    }
    if (best_i >= 0 && (double)best_num > tol2 * (double)best_den) {
      stack[sp++] = make_int2(best_i, se.y);
      stack[sp++] = make_int2(se.x, best_i);
      keep[best_i] = 1;
      ++kept;
    }
  }
  return kept;
}

__global__ void __launch_bounds__(TPB)
contour_trace_kernel(const int32_t* __restrict__ m, int h, int w, const int32_t* __restrict__ bbox, int n_labels,
                     const pick* __restrict__ picks, const int32_t* __restrict__ raw_off, double tol2,
                     int2* __restrict__ raw, uint8_t* __restrict__ keep, int2* __restrict__ stack,
                     int32_t* __restrict__ n_keep) {
  const int l = blockIdx.x * TPB + threadIdx.x;
  if (l >= n_labels) return;
  const pick pk = picks[l];
  if (pk.start_seg < 0) { n_keep[l] = 0; return; }
  walker wk{m, h, w, l + 1, make_window(bbox + 4 * l, h, w)};
  const int o = raw_off[l], n = pk.n_seg + 1;
  int cur = pk.start_seg;
  raw[o] = wk.point(cur, false);
  for (int i = 1; i < n; ++i) {
    raw[o + i] = wk.point(cur, true);
    if (i + 1 < n) cur = wk.step<true>(cur);
  }
  n_keep[l] = simplify(raw + o, n, tol2, keep + o, stack + o);
}

__global__ void __launch_bounds__(TPB)
contour_emit_kernel(int n_labels, const int32_t* __restrict__ raw_off, const int2* __restrict__ raw,
                    const uint8_t* __restrict__ keep, const int32_t* __restrict__ poly_off, double2* __restrict__ poly_xy) {
  const int l = blockIdx.x * TPB + threadIdx.x;
  if (l >= n_labels) return;
  const int o = raw_off[l], n = raw_off[l + 1] - o;
  int at = poly_off[l];
  for (int i = 0; i < n; ++i)
    if (keep[o + i]) poly_xy[at++] = make_double2(0.5 * raw[o + i].y, 0.5 * raw[o + i].x);  // (x, y) = (col, row)
}

}  // namespace

extern "C" {

int pg_instance_contours_count(pg_handle* h, int32_t height, int32_t width, const int32_t* inst_map, int32_t n_labels,
                               const int32_t* area, const int32_t* bbox, double tolerance, int32_t* poly_off,
                               pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  h->contour_labels = -1;
  PG_REQUIRE(h, height >= 0 && width >= 0 && n_labels >= 0 && poly_off, "pg_instance_contours_count: bad argument");
  PG_REQUIRE(h, height <= 16384 && width <= 16384, "pg_instance_contours_count: maps up to 16384 pixels a side");
  PG_REQUIRE(h, tolerance >= 0 && tolerance < 1e6, "pg_instance_contours_count: bad tolerance");
  PG_REQUIRE(h, n_labels == 0 || (inst_map && area && bbox), "pg_instance_contours_count: NULL argument");
  PG_REQUIRE(h, ((uintptr_t)poly_off & 15) == 0, "pg_instance_contours_count: poly_off must be 16-byte aligned");
  int rc;
  const int blocks = pg_div_up(std::max(n_labels, 1), TPB);
  // per-label scratch offsets: [0] visited bytes, [1] raw vertices, [2] counts before the scans
  const size_t per = (((size_t)n_labels + 8) * sizeof(int32_t) + 15) & ~(size_t)15;  // 16-byte aligned sub-arrays
  if ((rc = pg_reserve(h, h->row_count, 4 * per + (size_t)n_labels * sizeof(pick)))) return rc;
  int32_t* cnt = (int32_t*)h->row_count.p;
  int32_t* vis_off = (int32_t*)((char*)h->row_count.p + per);
  int32_t* raw_off = (int32_t*)((char*)h->row_count.p + 2 * per);
  pick* picks = (pick*)((char*)h->row_count.p + 4 * per);
  int32_t* totals = (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS);
  if (n_labels == 0 || height < 2 || width < 2) {  // no squares: no contours (skimage needs a 2 x 2 image)
    PG_CUDA(h, cudaMemsetAsync(poly_off, 0, ((size_t)n_labels + 1) * sizeof(int32_t), s));
    PG_CUDA(h, cudaMemsetAsync(totals + 3, 0, sizeof(int32_t), s));
    h->contour_labels = n_labels;
    h->contour_empty = true;
    return PG_OK;
  }
  h->contour_empty = false;
  PG_LAUNCH(h, s, "contour_window_kernel", contour_window_kernel<<<blocks, TPB, 0, s>>>(area, bbox, n_labels, height, width, cnt));
  PG_LAUNCH_CHECK(h);
  int64_t n_vis;  // visited bytes, then raw vertices: both totals are checked against the int32 offsets in 64 bits
  if ((rc = pg_scan_i32_total(h, cnt, vis_off, n_labels, s, totals + 3, "pg_instance_contours_count (visited bits)", &n_vis))) return rc;
  if ((rc = pg_reserve(h, h->cell_of, (size_t)n_vis + 64))) return rc;
  PG_LAUNCH(h, s, "contour_pick_kernel", contour_pick_kernel<<<blocks, TPB, 0, s>>>(inst_map, height, width, area, bbox, n_labels, vis_off,
                                                                                       (uint8_t*)h->cell_of.p, picks, cnt));
  PG_LAUNCH_CHECK(h);
  int64_t n_raw64;
  if ((rc = pg_scan_i32_total(h, cnt, raw_off, n_labels, s, totals + 3, "pg_instance_contours_count (raw vertices)", &n_raw64))) return rc;
  const size_t n_raw = (size_t)n_raw64;
  // raw vertices (int2) + stack (int2) in `rank`, keep flags in `cell_of` (the visited bits are done with)
  if ((rc = pg_reserve(h, h->rank, 2 * (n_raw + 8) * sizeof(int2)))) return rc;
  if ((rc = pg_reserve(h, h->cell_of, n_raw + 64))) return rc;
  int2* raw = (int2*)h->rank.p;
  int2* stack = raw + n_raw + 8;
  const double t2 = 2.0 * tolerance;
  PG_LAUNCH(h, s, "contour_trace_kernel", contour_trace_kernel<<<blocks, TPB, 0, s>>>(inst_map, height, width, bbox, n_labels, picks, raw_off, t2 * t2,
                                                                                         raw, (uint8_t*)h->cell_of.p, stack, cnt));
  PG_LAUNCH_CHECK(h);
  if ((rc = pg_scan_i32(h, cnt, poly_off, n_labels, s, totals + 3))) return rc;
  h->contour_labels = n_labels;
  h->contour_raw = (int64_t)n_raw;
  return PG_OK;
}

int pg_instance_contours_total(pg_handle* h, int64_t* total) {
  if (!h || !total) return PG_ERR_INVALID;
  PG_CUDA(h, cudaSetDevice(h->device));
  if (h->contour_labels < 0) return pg_set_error(h, PG_ERR_STATE, "pg_instance_contours_total: call pg_instance_contours_count first");
  PG_CUDA(h, cudaMemcpyAsync(&h->pinned[10], (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS) + 3, sizeof(int32_t),
                             cudaMemcpyDeviceToHost, h->last_stream));
  PG_CUDA(h, cudaStreamSynchronize(h->last_stream));
  *total = h->pinned[10];
  return PG_OK;
}

int pg_instance_contours_fill(pg_handle* h, int32_t n_labels, const int32_t* poly_off, double* poly_xy, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  if (h->contour_labels < 0 || h->contour_labels != n_labels)
    return pg_set_error(h, PG_ERR_STATE, "pg_instance_contours_fill: call pg_instance_contours_count for the same labels first");
  PG_REQUIRE(h, poly_off != nullptr, "pg_instance_contours_fill: poly_off is NULL");
  PG_REQUIRE(h, ((uintptr_t)poly_xy & 15) == 0, "pg_instance_contours_fill: poly_xy must be 16-byte aligned");
  if (n_labels == 0 || h->contour_empty) return PG_OK;
  const size_t per = (((size_t)n_labels + 8) * sizeof(int32_t) + 15) & ~(size_t)15;
  const int32_t* raw_off = (const int32_t*)((char*)h->row_count.p + 2 * per);
  PG_LAUNCH(h, s, "contour_emit_kernel", contour_emit_kernel<<<pg_div_up(n_labels, TPB), TPB, 0, s>>>(n_labels, raw_off, (const int2*)h->rank.p,
                                                                                                         (const uint8_t*)h->cell_of.p, poly_off, (double2*)poly_xy));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // extern "C"
