// K12: raster region properties of a HoverNeXt instance map (SURVEY 8f-3, first half).
// Reference: /root/reference/aggregated_hovernet_run.py:172-181 (regionprops(inst_map): per-instance bbox) and
// /root/reference/hovernet_tile_inference.ipynb:2415-2429 (cell 18: regionprops_table area, perimeter,
// eccentricity, major / minor axis length, orientation). skimage's definitions (SURVEY A.4):
//   area = pixel count; bbox = [min_row, min_col, max_row + 1, max_col + 1]; centroid = mean (row, col);
//   inertia tensor T = [[mu02, -mu11], [-mu11, mu20]] / mu00 (axis 0 = rows), eigenvalues l1 >= l2 >= 0;
//   eccentricity = sqrt(1 - l2 / l1) (0 when l1 == 0); major / minor = 4 sqrt(l1 / l2);
//   orientation = 0.5 atan2(-2 b, c - a) with (a, b, c) = (T00, T01, T11), +-pi/4 when a == c;
//   perimeter (4-neighbourhood): border = pixels with a 4-neighbour outside the region; every border pixel gets
//   the code sum of [[10,2,10],[2,1,2],[10,2,10]] over the border pixels around it and contributes 1 for codes
//   5,7,15,17,25,27, sqrt(2) for 21,33 and (1+sqrt(2))/2 for 13,23.
// The reference does this with one full-mask pass PER INSTANCE (inst_map == inst_id, :183); here the map is read
// twice in total. All accumulators are integers (pixel coordinates are integers: raw moments are exact in int64,
// perimeter is three counters), so the result does not depend on the order of the atomics.
#include <algorithm>
#include "pg_common.cuh"

namespace {

constexpr int TPB = 256;

struct raster_acc {  // one per label
  unsigned long long sr, sc, srr, scc, src;
  int area, min_r, min_c, max_r, max_c;
  int p1, p2, p3;  // perimeter code classes: weight 1, sqrt(2), (1 + sqrt(2)) / 2
};

__global__ void __launch_bounds__(TPB)
raster_init_kernel(raster_acc* acc, int n_labels) {
  const int i = blockIdx.x * TPB + threadIdx.x;
  if (i >= n_labels) return;
  raster_acc a;
  a.sr = a.sc = a.srr = a.scc = a.src = 0ull;
  a.area = 0; a.min_r = a.min_c = 0x7fffffff; a.max_r = a.max_c = -1;
  a.p1 = a.p2 = a.p3 = 0;
  acc[i] = a;
}

__device__ __forceinline__ int label_at(const int32_t* __restrict__ m, int h, int w, int r, int c) {
  return (r >= 0 && r < h && c >= 0 && c < w) ? m[(int64_t)r * w + c] : 0;
}

// pass 1: moments, bbox, border map. One thread per pixel; the lanes of a warp that carry the same label (a run
// of a nucleus along the row) are folded together before they touch the accumulators.
__global__ void __launch_bounds__(TPB)
raster_moments_kernel(const int32_t* __restrict__ m, int h, int w, int n_labels, raster_acc* __restrict__ acc,
                      uint8_t* __restrict__ border) {
  const int64_t px = (int64_t)blockIdx.x * TPB + threadIdx.x;
  const bool in = px < (int64_t)h * w;
  const int r = in ? (int)(px / w) : 0, c = in ? (int)(px - (int64_t)r * w) : 0;
  int lab = in ? m[px] : 0;
  if (lab < 0 || lab > n_labels) lab = 0;
  bool is_border = false;
  if (lab > 0)
    is_border = label_at(m, h, w, r - 1, c) != lab || label_at(m, h, w, r + 1, c) != lab ||
                label_at(m, h, w, r, c - 1) != lab || label_at(m, h, w, r, c + 1) != lab;
  if (in) border[px] = is_border ? 1 : 0;
  const unsigned peers = __match_any_sync(0xffffffffu, lab);
  if (lab == 0) return;
  const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
  // group sums: values are < 2^31 per lane for maps up to 46340 pixels a side; 64-bit sums via two 32-bit halves
  const unsigned cnt = __popc(peers);
  const unsigned s_r = __reduce_add_sync(peers, (unsigned)r), s_c = __reduce_add_sync(peers, (unsigned)c);
  const unsigned long long rr = (unsigned long long)r * r, cc = (unsigned long long)c * c, rc = (unsigned long long)r * c;
  const unsigned long long s_rr = (unsigned long long)__reduce_add_sync(peers, (unsigned)(rr & 0xffffu)) +
                                  ((unsigned long long)__reduce_add_sync(peers, (unsigned)(rr >> 16)) << 16);
  const unsigned long long s_cc = (unsigned long long)__reduce_add_sync(peers, (unsigned)(cc & 0xffffu)) +
                                  ((unsigned long long)__reduce_add_sync(peers, (unsigned)(cc >> 16)) << 16);
  const unsigned long long s_rc = (unsigned long long)__reduce_add_sync(peers, (unsigned)(rc & 0xffffu)) +
                                  ((unsigned long long)__reduce_add_sync(peers, (unsigned)(rc >> 16)) << 16);
  const int mn_r = __reduce_min_sync(peers, r), mx_r = __reduce_max_sync(peers, r);
  const int mn_c = __reduce_min_sync(peers, c), mx_c = __reduce_max_sync(peers, c);
  if (lane != leader) return;
  raster_acc* a = acc + (lab - 1);
  atomicAdd(&a->area, (int)cnt);
  atomicAdd(&a->sr, (unsigned long long)s_r); atomicAdd(&a->sc, (unsigned long long)s_c);
  atomicAdd(&a->srr, s_rr); atomicAdd(&a->scc, s_cc); atomicAdd(&a->src, s_rc);
  atomicMin(&a->min_r, mn_r); atomicMax(&a->max_r, mx_r);
  atomicMin(&a->min_c, mn_c); atomicMax(&a->max_c, mx_c);
}

// pass 2: perimeter codes of the border pixels
__global__ void __launch_bounds__(TPB)
raster_perimeter_kernel(const int32_t* __restrict__ m, const uint8_t* __restrict__ border, int h, int w,
                        int n_labels, raster_acc* __restrict__ acc) {
  const int64_t px = (int64_t)blockIdx.x * TPB + threadIdx.x;
  if (px >= (int64_t)h * w || !border[px]) return;
  const int lab = m[px];
  const int r = (int)(px / w), c = (int)(px - (int64_t)r * w);
  int code = 1;
#pragma unroll
  for (int dr = -1; dr <= 1; ++dr)
#pragma unroll
    for (int dc = -1; dc <= 1; ++dc) {
      if (dr == 0 && dc == 0) continue;
      const int rr = r + dr, cc = c + dc;
      if (rr < 0 || rr >= h || cc < 0 || cc >= w) continue;
      const int64_t q = (int64_t)rr * w + cc;
      if (border[q] && m[q] == lab) code += (dr != 0 && dc != 0) ? 10 : 2;
    }
  raster_acc* a = acc + (lab - 1);
  if (code == 5 || code == 7 || code == 15 || code == 17 || code == 25 || code == 27) atomicAdd(&a->p1, 1);
  else if (code == 21 || code == 33) atomicAdd(&a->p2, 1);
  else if (code == 13 || code == 23) atomicAdd(&a->p3, 1);
}

__global__ void __launch_bounds__(TPB)
raster_finish_kernel(const raster_acc* __restrict__ acc, int n_labels, pg_raster_out o) {
  const int i = blockIdx.x * TPB + threadIdx.x;
  if (i >= n_labels) return;
  const raster_acc a = acc[i];
  const double nan_ = __longlong_as_double(0x7ff8000000000000ll);
  if (o.area) o.area[i] = a.area;
  const bool some = a.area > 0;
  if (o.bbox) {
    o.bbox[4 * i + 0] = some ? a.min_r : 0; o.bbox[4 * i + 1] = some ? a.min_c : 0;
    o.bbox[4 * i + 2] = some ? a.max_r + 1 : 0; o.bbox[4 * i + 3] = some ? a.max_c + 1 : 0;
  }
  double cr = nan_, cc = nan_, ecc = nan_, major = nan_, minor = nan_, orient = nan_, per = nan_;
  if (some) {
    const double n = (double)a.area;
    cr = (double)a.sr / n; cc = (double)a.sc / n;
    // exact integer central moments, each rounded once: n mu20 = n sum r^2 - (sum r)^2, ... in __int128
    // (n < 2^31, sum r^2 < 2^63: every product < 2^95), and the tensor entry mu20 / n = (n mu20) / n^2.
    // Subtracting the raw moments in float64 instead loses digits with the square of the region's distance
    // from the origin (1e-7 in the axis lengths at 46000 px).
    const __int128 n_ = a.area;
    const __int128 sr = (__int128)a.sr, sc = (__int128)a.sc;
    const double num20 = (double)(n_ * (__int128)a.srr - sr * sr);
    const double num02 = (double)(n_ * (__int128)a.scc - sc * sc);
    const double num11 = (double)(n_ * (__int128)a.src - sr * sc);
    const double n2 = n * n;
    const double ta = num02 / n2, tb = -(num11 / n2), tc = num20 / n2;  // inertia tensor [[ta, tb], [tb, tc]]
    const double mid = 0.5 * (ta + tc), hd = 0.5 * (ta - tc);
    const double rad = sqrt(hd * hd + tb * tb);
    const double l1 = fmax(mid + rad, 0.0), l2 = fmax(mid - rad, 0.0);
    ecc = l1 == 0.0 ? 0.0 : sqrt(1.0 - l2 / l1);
    major = 4.0 * sqrt(l1);
    minor = 4.0 * sqrt(l2);
    const double pi = 3.14159265358979323846;
    orient = (ta - tc == 0.0) ? (tb < 0.0 ? pi / 4.0 : -pi / 4.0) : 0.5 * atan2(-2.0 * tb, tc - ta);
    per = (double)a.p1 + (double)a.p2 * 1.4142135623730951 + (double)a.p3 * ((1.0 + 1.4142135623730951) / 2.0);
  }
  if (o.centroid) { o.centroid[2 * i] = cr; o.centroid[2 * i + 1] = cc; }
  if (o.eccentricity) o.eccentricity[i] = ecc;
  if (o.major_axis) o.major_axis[i] = major;
  if (o.minor_axis) o.minor_axis[i] = minor;
  if (o.orientation) o.orientation[i] = orient;
  if (o.perimeter) o.perimeter[i] = per;
}

// ---- solidity = area / area of the convex hull image (skimage convex_hull_image: the hull of the pixels' diamond
// corners (r +- 1/2, c), (r, c +- 1/2), rasterised including its border). One thread per instance, doubled integer
// coordinates, everything exact: per doubled row the extent [lo, hi] of the diamond points, the hull's left / right
// chains by a monotone-chain stack over the rows, then per pixel row the integer columns between the two chains.
__global__ void __launch_bounds__(TPB)
raster_rows_kernel(const int32_t* __restrict__ area, const int32_t* __restrict__ bbox, int n_labels, int32_t* __restrict__ need) {
  const int l = blockIdx.x * TPB + threadIdx.x;
  if (l >= n_labels) return;
  need[l] = area[l] > 0 ? 4 * (2 * (bbox[4 * l + 2] - bbox[4 * l]) + 1) : 0;
}

__device__ __forceinline__ long long floor_div(long long a, long long b) {  // b > 0
  long long q = a / b;
  return (a % b != 0 && a < 0) ? q - 1 : q;
}

__global__ void __launch_bounds__(TPB)
raster_solidity_kernel(const int32_t* __restrict__ m, int h, int w, const int32_t* __restrict__ area,
                       const int32_t* __restrict__ bbox, int n_labels, const int32_t* __restrict__ off,
                       int32_t* __restrict__ scratch, int32_t* __restrict__ convex_area, double* __restrict__ solidity) {
  const int l = blockIdx.x * TPB + threadIdx.x;
  if (l >= n_labels) return;
  const double nan_ = __longlong_as_double(0x7ff8000000000000ll);
  if (area[l] <= 0) {
    if (convex_area) convex_area[l] = 0;
    if (solidity) solidity[l] = nan_;
    return;
  }
  const int lab = l + 1;
  const int r0 = bbox[4 * l], c0 = bbox[4 * l + 1], r1 = bbox[4 * l + 2], c1 = bbox[4 * l + 3];
  const int nd = 2 * (r1 - r0) + 1;  // doubled rows 2 r0 - 1 .. 2 (r1 - 1) + 1, index j = R - (2 r0 - 1)
  int32_t* lo = scratch + off[l];
  int32_t* hi = lo + nd;
  int32_t* sl = hi + nd;  // hull stacks (row indices)
  int32_t* sr = sl + nd;
  const int NONE_LO = 0x7fffffff, NONE_HI = -0x7fffffff;
  for (int j = 0; j < nd; ++j) { lo[j] = NONE_LO; hi[j] = NONE_HI; }
  for (int r = r0; r < r1; ++r) {
    const int32_t* row = m + (int64_t)r * w;
    int cmin = -1, cmax = -1;
    for (int c = c0; c < c1; ++c)
      if (row[c] == lab) { if (cmin < 0) cmin = c; cmax = c; }
    if (cmin < 0) continue;
    const int j = 2 * (r - r0);
    lo[j] = min(lo[j], 2 * cmin); hi[j] = max(hi[j], 2 * cmax);
    lo[j + 1] = min(lo[j + 1], 2 * cmin - 1); hi[j + 1] = max(hi[j + 1], 2 * cmax + 1);
    lo[j + 2] = min(lo[j + 2], 2 * cmin); hi[j + 2] = max(hi[j + 2], 2 * cmax);
  }
  // monotone chains over the rows that hold points: left = lower convex envelope of (j, lo), right = upper of (j, hi)
  int nl = 0, nr = 0;
  for (int j = 0; j < nd; ++j) {
    if (lo[j] == NONE_LO) continue;
    while (nl >= 2) {
      const long long ax = sl[nl - 2], bx = sl[nl - 1];
      const long long cr = (bx - ax) * ((long long)lo[j] - lo[ax]) - ((long long)lo[bx] - lo[ax]) * (j - ax);
      if (cr <= 0) --nl; else break;  // b on or above the chord a -> j: not a vertex of the lower envelope
    }
    sl[nl++] = j;
    while (nr >= 2) {
      const long long ax = sr[nr - 2], bx = sr[nr - 1];
      const long long cr = (bx - ax) * ((long long)hi[j] - hi[ax]) - ((long long)hi[bx] - hi[ax]) * (j - ax);
      if (cr >= 0) --nr; else break;
    }
    sr[nr++] = j;
  }
  // pixel rows: doubled row R = 2 r has index j = 2 (r - r0) + 1; count the columns c with L(j) <= 2 c <= U(j)
  long long count = 0;
  int il = 0, ir = 0;
  const int j_first = sl[0], j_last = sl[nl - 1];
  for (int r = r0; r < r1; ++r) {
    const int j = 2 * (r - r0) + 1;
    if (j < j_first || j > j_last) continue;
    while (il + 1 < nl - 1 && sl[il + 1] <= j) ++il;
    while (ir + 1 < nr - 1 && sr[ir + 1] <= j) ++ir;
    long long c_lo, c_hi;
    {
      const long long a = sl[il], b = sl[min(il + 1, nl - 1)];
      if (b == a) c_lo = -floor_div(-(long long)lo[a], 2);
      else {
        const long long den = b - a, num = (long long)lo[a] * den + ((long long)lo[b] - lo[a]) * (j - a);
        c_lo = -floor_div(-num, 2 * den);  // ceil(num / (2 den))
      }
    }
    {
      const long long a = sr[ir], b = sr[min(ir + 1, nr - 1)];
      if (b == a) c_hi = floor_div((long long)hi[a], 2);
      else {
        const long long den = b - a, num = (long long)hi[a] * den + ((long long)hi[b] - hi[a]) * (j - a);
        c_hi = floor_div(num, 2 * den);
      }
    }
    if (c_hi >= c_lo) count += c_hi - c_lo + 1;
  }
  if (convex_area) convex_area[l] = (int32_t)count;
  if (solidity) solidity[l] = count > 0 ? (double)area[l] / (double)count : nan_;
}

}  // namespace

extern "C" int pg_raster_props(pg_handle* h, int32_t height, int32_t width, const int32_t* inst_map, int32_t n_labels,
                               const pg_raster_out* out, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, height >= 0 && width >= 0 && n_labels >= 0 && out, "pg_raster_props: bad argument");
  PG_REQUIRE(h, height <= 46340 && width <= 46340, "pg_raster_props: maps up to 46340 pixels a side");
  if (n_labels == 0) return PG_OK;
  const int64_t pixels = (int64_t)height * width;
  PG_REQUIRE(h, pixels == 0 || inst_map, "pg_raster_props: inst_map is NULL");
  int rc;
  if ((rc = pg_reserve(h, h->rank, (size_t)n_labels * sizeof(raster_acc)))) return rc;
  if ((rc = pg_reserve(h, h->cell_of, (size_t)pixels + 16))) return rc;
  raster_acc* acc = (raster_acc*)h->rank.p;
  uint8_t* border = (uint8_t*)h->cell_of.p;
  PG_LAUNCH(h, s, "raster_init_kernel", raster_init_kernel<<<pg_div_up(n_labels, TPB), TPB, 0, s>>>(acc, n_labels));
  if (pixels > 0) {
    const int blocks = pg_div_up(pixels, TPB);
    PG_LAUNCH(h, s, "raster_moments_kernel", raster_moments_kernel<<<blocks, TPB, 0, s>>>(inst_map, height, width, n_labels, acc, border));
    PG_LAUNCH(h, s, "raster_perimeter_kernel", raster_perimeter_kernel<<<blocks, TPB, 0, s>>>(inst_map, border, height, width, n_labels, acc));
  }
  PG_LAUNCH(h, s, "raster_finish_kernel", raster_finish_kernel<<<pg_div_up(n_labels, TPB), TPB, 0, s>>>(acc, n_labels, *out));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

extern "C" int pg_raster_solidity(pg_handle* h, int32_t height, int32_t width, const int32_t* inst_map, int32_t n_labels,
                                  const int32_t* area, const int32_t* bbox, int32_t* convex_area, double* solidity,
                                  pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  PG_REQUIRE(h, height >= 0 && width >= 0 && n_labels >= 0, "pg_raster_solidity: bad argument");
  if (n_labels == 0) return PG_OK;
  PG_REQUIRE(h, inst_map && area && bbox, "pg_raster_solidity: NULL argument");
  int rc;
  const size_t per = (((size_t)n_labels + 8) * sizeof(int32_t) + 15) & ~(size_t)15;
  if ((rc = pg_reserve(h, h->row_count, 2 * per))) return rc;
  int32_t* need = (int32_t*)h->row_count.p;
  int32_t* off = (int32_t*)((char*)h->row_count.p + per);
  int32_t* totals = (int32_t*)((char*)h->misc.p + PG_MISC_TOTALS);
  const int blocks = pg_div_up(n_labels, TPB);
  PG_LAUNCH(h, s, "raster_rows_kernel", raster_rows_kernel<<<blocks, TPB, 0, s>>>(area, bbox, n_labels, need));
  PG_LAUNCH_CHECK(h);
  int64_t n_scratch;
  if ((rc = pg_scan_i32_total(h, need, off, n_labels, s, totals + 3, "pg_raster_solidity", &n_scratch))) return rc;
  if ((rc = pg_reserve(h, h->rank, ((size_t)n_scratch + 16) * sizeof(int32_t)))) return rc;
  PG_LAUNCH(h, s, "raster_solidity_kernel", raster_solidity_kernel<<<blocks, TPB, 0, s>>>(inst_map, height, width, area, bbox, n_labels, off,
                                                                                             (int32_t*)h->rank.p, convex_area, solidity));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}
