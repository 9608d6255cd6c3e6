// K1: fused tile->WSI shift + polygon morphology over CSR-packed rings.
// Reference: /root/reference/aggregated_hovernet_run.py:302-334 (centroid / bbox / polygon shift),
// /root/reference/polygon_morphology.py:240-248 and create_and_overlay_polygon_from_prediction.py:298-299
// (shapely area / length / centroid / bounds), hovernet_tile_inference.ipynb:2415-2456 (eccentricity,
// axes, compactness). Formulas: SURVEY A.4 (Green's-theorem area moments in a frame at vertex 0).
//
// Work split: a warp owns 32 consecutive polygons = ONE contiguous range of the vertex array.
//   staged path (the range fits the warp's shared-memory slab - every nuclei table): lane 0 brings the range in
//     with one bulk copy (cp.async.bulk, completion on a per-warp mbarrier) while the lanes do the per-polygon
//     centroid / bbox shifts; then each LANE walks ITS polygon out of shared memory - no shuffles, no reductions,
//     one load per vertex - adding the tile offset in place, and lane 0 sends the shifted slab back with one bulk
//     store. The ring is cyclic, so lane l starts at the vertex that puts it on shared-memory bank (l mod 16):
//     32 lanes walking rings 256 B apart stay conflict-free. Global traffic is two full-line bulk transfers.
//   group path (a warp whose range exceeds the slab, e.g. tissue-region rings of thousands of vertices):
//     sub-warps of 8 lanes walk one ring each straight from global memory, 3-step butterfly, totals handed to
//     the polygon's lane.
// Both leave the Green's-theorem sums of a polygon (frame at one of its own vertices, float64) in its lane; the
// closed-form epilogue and all per-polygon loads / stores run one polygon per lane, fully coalesced.
#include <algorithm>
#include <cmath>
#include "pg_common.cuh"
#include "pg_ring.cuh"

namespace {

constexpr int TPB = 128;
constexpr int WARPS = TPB / 32;
constexpr int SLAB_VERTS_MIN = 32 * 33 + 2;  // 32 rings of 32 vertices, explicitly closed (+1), + alignment slack
constexpr size_t SLAB_BYTES_MAX = 200 * 1024;  // per CTA

__device__ __forceinline__ double bfly_add(double v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}
__device__ __forceinline__ float bfly_addf(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}
template <typename T> __device__ __forceinline__ T bfly_min(T v) {
  v = min(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = min(v, __shfl_xor_sync(0xffffffffu, v, 2));
  v = min(v, __shfl_xor_sync(0xffffffffu, v, 4));
  return v;
}
template <typename T> __device__ __forceinline__ T bfly_max(T v) {
  v = max(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = max(v, __shfl_xor_sync(0xffffffffu, v, 2));
  v = max(v, __shfl_xor_sync(0xffffffffu, v, 4));
  return v;
}

// length of one edge in float32: MUFU.SQRT (sqrt.approx, relative error <= 2^-22) instead of the IEEE sqrtf sequence
// (MUFU.RSQ + Newton step + a guarded slow path: ~9 instructions and a branch per vertex of the inner loop). The
// perimeter is a float32 output compared at 1e-5; the sum of <= 32 such terms is folded into float64 (ring_sums).
__device__ __forceinline__ float edge_len(float dx, float dy) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(fmaf(dx, dx, dy * dy)));
  return r;
}

// MINB = CTAs per SM the register allocation leaves room for. The kernel is latency-bound per warp (bulk load ->
// walk -> bulk store), so what it delivers follows the warps per SM: MINB = 7 (72 registers instead of 80 for float32
// vertices) is picked by the launcher whenever the slabs are small enough for 7 CTAs to fit shared memory.
template <typename T, bool EXTRA, int MINB>
__global__ void __launch_bounds__(TPB, MINB)
map_morph_kernel(int n, const int32_t* __restrict__ poly_off, const typename vec2_of<T>::type* __restrict__ poly,
                 const int32_t* __restrict__ nuc_tile, const int32_t* __restrict__ tile_x,
                 const int32_t* __restrict__ tile_y, const double2* __restrict__ centroid,
                 const int4* __restrict__ bbox, typename vec2_of<T>::type* __restrict__ wsi_poly,
                 double2* __restrict__ wsi_centroid, int4* __restrict__ wsi_bbox, pg_morph_out out,
                 int slab_verts) {
  using V2 = typename vec2_of<T>::type;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t s_bar[WARPS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int warp_global = (blockIdx.x * TPB + threadIdx.x) >> 5;
  const int my_poly = warp_global * 32 + lane;
  if (warp_global * 32 >= n) return;  // whole warp out of range (no CTA-wide barrier below)

  // ---- the warp's vertex range
  const int off0 = poly_off[min(my_poly, n)];
  const int off_last = poly_off[min(warp_global * 32 + 32, n)];
  const int off_next = __shfl_down_sync(0xffffffffu, off0, 1);
  const int nv = (lane == 31 ? off_last : off_next) - off0;
  const int wbeg = __shfl_sync(0xffffffffu, off0, 0);
  const int total = off_last - wbeg;

  // slab: vertex i of the range lives at slab[i]; the bulk transfers need 16-byte alignment on both sides, so
  // the slab is placed with the same alignment phase as the global range (`head` vertices precede the first
  // 16-byte boundary: 0 or 1 for float2, always 0 for double2) and the odd head / tail vertices move by hand
  V2* slab_base = reinterpret_cast<V2*>(smem_raw) + (size_t)wid * slab_verts;
  const V2* gsrc = poly + wbeg;
  V2* gdst = wsi_poly ? wsi_poly + wbeg : nullptr;
  const int head = (int)(((16u - (uint32_t)((uintptr_t)gsrc & 15u)) & 15u) / sizeof(V2));
  const bool same_phase = !gdst || (((uintptr_t)gsrc ^ (uintptr_t)gdst) & 15u) == 0;
  const bool staged = total > 0 && total <= slab_verts - 2 && same_phase;  // warp-uniform
  V2* slab = slab_base + (head ? (int)(16 / sizeof(V2)) - head : 0);       // &slab[head] is 16-byte aligned
  int nbulk = 0;
  if (staged) {
    const int h = min(head, total);
    nbulk = ((total - h) * (int)sizeof(V2) & ~15) / (int)sizeof(V2);
    const int tail0 = h + nbulk;  // [tail0, total) moves by hand
    if (lane == 0) {
      mbar_init(&s_bar[wid], 1);
      if (nbulk > 0) {
        mbar_expect_tx(&s_bar[wid], (uint32_t)nbulk * sizeof(V2));
        bulk_load(slab + h, gsrc + h, (uint32_t)nbulk * sizeof(V2), &s_bar[wid]);
      }
    } else if (lane == 1) {
      for (int i = 0; i < h; ++i) slab[i] = gsrc[i];
    } else if (lane == 2) {
      for (int i = tail0; i < total; ++i) slab[i] = gsrc[i];
    }
  }

  // ---- one polygon per lane: tile shift, centroid / bbox shift (aggregated_hovernet_run.py:302-319); this
  // runs while the bulk load is in flight
  int itx = 0, ity = 0;
  if (my_poly < n) {
    if (nuc_tile) { const int t = nuc_tile[my_poly]; itx = tile_x[t]; ity = tile_y[t]; }
    if (centroid) { const double2 c = centroid[my_poly]; wsi_centroid[my_poly] = make_double2(c.x + (double)itx, c.y + (double)ity); }
    if (bbox) { const int4 b = bbox[my_poly]; wsi_bbox[my_poly] = make_int4(b.x + itx, b.y + ity, b.z + itx, b.w + ity); }
  }

  ring_sums r;
  r.S = r.Sx = r.Sy = r.Ixx = r.Iyy = r.Ixy = 0; r.P = 0; r.Pd = 0; r.fx = r.fy = 0;
  T bx0 = 0, by0 = 0, bx1 = 0, by1 = 0;

  if (staged) {
    __syncwarp();                       // barrier initialised, hand-moved vertices visible
    if (nbulk > 0) mbar_wait(&s_bar[wid], 0);
    if (nv > 0) {
      V2* mine = slab + (off0 - wbeg);
      // start vertex: bank (pair / quad) of slab[..] advances by one per vertex; put lane l on bank l
      constexpr int BANKS = 128 / (int)sizeof(V2);  // distinct vertex slots per shared-memory wavefront
      const int phase = (int)((smem_u32(mine) / sizeof(V2)) & (BANKS - 1));
      int idx = (lane - phase) & (BANKS - 1);
      if (idx >= nv) idx %= nv;
      const T tsx = (T)itx, tsy = (T)ity;
      V2 v = mine[idx];
      if (wsi_poly) { V2 w; w.x = v.x + tsx; w.y = v.y + tsy; mine[idx] = w; }  // :322-334
      r.fx = (double)v.x; r.fy = (double)v.y;
      if (EXTRA) { bx0 = bx1 = v.x; by0 = by1 = v.y; }
      double xa = 0, ya = 0;
      T px = v.x, py = v.y;
      const T fxT = v.x, fyT = v.y;
#pragma unroll 2
      for (int k = 1; k < nv; ++k) {
        idx = idx + 1 == nv ? 0 : idx + 1;
        v = mine[idx];
        if (wsi_poly) { V2 w; w.x = v.x + tsx; w.y = v.y + tsy; mine[idx] = w; }
        const double xb = (double)v.x - r.fx, yb = (double)v.y - r.fy;
        edge_terms(r, xa, ya, xb, yb);
        const float dx = (float)(v.x - px), dy = (float)(v.y - py);
        r.P += edge_len(dx, dy);
        if ((k & 31) == 0) { r.Pd += (double)r.P; r.P = 0.f; }
        if (EXTRA) { bx0 = min(bx0, v.x); bx1 = max(bx1, v.x); by0 = min(by0, v.y); by1 = max(by1, v.y); }
        xa = xb; ya = yb; px = v.x; py = v.y;
      }
      {  // closing edge back to the start vertex (the frame origin: no area terms)
        const float dx = (float)(fxT - px), dy = (float)(fyT - py);
        r.P += edge_len(dx, dy);
      }
    }
    if (wsi_poly) {
      fence_async_smem();               // generic-proxy writes -> visible to the bulk store
      __syncwarp();
      const int h = min(head, total), tail0 = h + nbulk;
      if (lane == 0) {
        if (nbulk > 0) { bulk_store(gdst + h, slab + h, (uint32_t)nbulk * sizeof(V2)); bulk_store_wait_read(); }
      } else if (lane == 1) {
        for (int i = 0; i < h; ++i) gdst[i] = slab[i];
      } else if (lane == 2) {
        for (int i = tail0; i < total; ++i) gdst[i] = slab[i];
      }
    }
  } else {
    // ---- group path: 8 lanes per ring, straight from global memory
    const int grp = lane >> 3, sub = lane & 7;
#pragma unroll 1
    for (int t = 0; t < 8; ++t) {
      const int src = (grp << 3) + t;
      const int o = __shfl_sync(0xffffffffu, off0, src);
      const int cnt = __shfl_sync(0xffffffffu, nv, src);
      const int sx = __shfl_sync(0xffffffffu, itx, src);
      const int sy = __shfl_sync(0xffffffffu, ity, src);
      ring_sums a;
      a.S = a.Sx = a.Sy = a.Ixx = a.Iyy = a.Ixy = 0; a.P = 0; a.Pd = 0;
      V2 v0; v0.x = 0; v0.y = 0;
      T mnx = 0, mny = 0, mxx = 0, mxy = 0;
      if (cnt > 0) {
        v0 = poly[o];
        if (EXTRA) { mnx = mxx = v0.x; mny = mxy = v0.y; }
        const T tsx = (T)sx, tsy = (T)sy;
        for (int e = sub; e < cnt; e += 8) {
          const V2 va = poly[o + e];
          const V2 vb = poly[o + ((e + 1 == cnt) ? 0 : e + 1)];
          if (wsi_poly) { V2 w; w.x = va.x + tsx; w.y = va.y + tsy; wsi_poly[o + e] = w; }
          const double xa = (double)va.x - (double)v0.x, ya = (double)va.y - (double)v0.y;
          const double xb = (double)vb.x - (double)v0.x, yb = (double)vb.y - (double)v0.y;
          edge_terms(a, xa, ya, xb, yb);
          const float dx = (float)(vb.x - va.x), dy = (float)(vb.y - va.y);
          a.Pd += (double)edge_len(dx, dy);  // long rings live on this path: float64 accumulation throughout
          if (EXTRA) { mnx = min(mnx, va.x); mxx = max(mxx, va.x); mny = min(mny, va.y); mxy = max(mxy, va.y); }
        }
      }
      a.S = bfly_add(a.S); a.Sx = bfly_add(a.Sx); a.Sy = bfly_add(a.Sy);
      a.Ixx = bfly_add(a.Ixx); a.Iyy = bfly_add(a.Iyy); a.Ixy = bfly_add(a.Ixy);
      a.Pd = bfly_add(a.Pd);
      if (EXTRA) { mnx = bfly_min(mnx); mny = bfly_min(mny); mxx = bfly_max(mxx); mxy = bfly_max(mxy); }
      if (sub == t) {
        r = a;
        r.fx = (double)v0.x; r.fy = (double)v0.y;
        if (EXTRA) { bx0 = mnx; by0 = mny; bx1 = mxx; by1 = mxy; }
      }
    }
  }

  // ---- epilogue: one polygon per lane
  if (my_poly >= n) return;
  const double S = r.S, Sx = r.Sx, Sy = r.Sy, Ixx = r.Ixx, Iyy = r.Iyy, Ixy = r.Ixy, fx = r.fx, fy = r.fy;
  const double per = r.Pd + (double)r.P;
  const float P = (float)per;
  const float nanf_ = __int_as_float(0x7fc00000);
  const double nand_ = __longlong_as_double(0x7ff8000000000000ll);
  const bool ok = nv >= 3;
  const double A = 0.5 * S;
  const double area = fabs(A);
  if (out.area) out.area[my_poly] = ok ? (float)area : nanf_;
  if (out.perimeter) out.perimeter[my_poly] = ok ? P : nanf_;
  if (out.circularity) {
    const double pm = fmax(per, 1.0);
    out.circularity[my_poly] = ok ? (float)(4.0 * 3.14159265358979323846 * area / (pm * pm)) : nanf_;
  }
  const bool good = ok && A != 0.0;
  double ecc = nand_, major = nand_, minor = nand_, cxw = nand_, cyw = nand_;
  if (good) {
    const double inv = 1.0 / A;
    const double cx = Sx * inv * (1.0 / 6.0), cy = Sy * inv * (1.0 / 6.0);
    const double mu20 = Iyy * inv * (1.0 / 12.0) - cx * cx;
    const double mu02 = Ixx * inv * (1.0 / 12.0) - cy * cy;
    const double mu11 = Ixy * inv * (1.0 / 24.0) - cx * cy;
    const double m = 0.5 * (mu20 + mu02);
    const double hd = 0.5 * (mu20 - mu02);
    const double c = sqrt(hd * hd + mu11 * mu11);
    const double l1 = m + c;
    const double l2 = fmax(m - c, 0.0);
    ecc = l1 > 0.0 ? sqrt(1.0 - l2 / l1) : 0.0;
    major = 4.0 * sqrt(fmax(l1, 0.0));
    minor = 4.0 * sqrt(l2);
    cxw = cx + fx + (double)itx;
    cyw = cy + fy + (double)ity;
  }
  if (out.eccentricity) out.eccentricity[my_poly] = (float)ecc;
  if (EXTRA) {
    if (out.major_axis) out.major_axis[my_poly] = (float)major;
    if (out.minor_axis) out.minor_axis[my_poly] = (float)minor;
    if (out.centroid_x) out.centroid_x[my_poly] = cxw;
    if (out.centroid_y) out.centroid_y[my_poly] = cyw;
    if (out.poly_bbox) {
      double* b = out.poly_bbox + (int64_t)my_poly * 4;
      b[0] = ok ? (double)bx0 + (double)itx : nand_; b[1] = ok ? (double)by0 + (double)ity : nand_;
      b[2] = ok ? (double)bx1 + (double)itx : nand_; b[3] = ok ? (double)by1 + (double)ity : nand_;
    }
  }
}

template <typename T>
int launch_map_morph(pg_handle* h, int32_t n, const int32_t* poly_off, const T* poly_xy, const int32_t* nuc_tile,
                     const int32_t* tile_x, const int32_t* tile_y, const double* centroid, const int32_t* bbox,
                     T* wsi_poly_xy, double* wsi_centroid, int32_t* wsi_bbox, const pg_morph_out* out, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  using V2 = typename vec2_of<T>::type;
  PG_REQUIRE(h, n >= 0, "pg_map_morph: n < 0");
  PG_REQUIRE(h, n == 0 || poly_off, "pg_map_morph: poly_off is NULL");
  PG_REQUIRE(h, !nuc_tile || (tile_x && tile_y), "pg_map_morph: nuc_tile given without tile_x / tile_y");
  PG_REQUIRE(h, !centroid || wsi_centroid, "pg_map_morph: centroid given without wsi_centroid");
  PG_REQUIRE(h, !bbox || wsi_bbox, "pg_map_morph: bbox given without wsi_bbox");
  PG_REQUIRE(h, (((uintptr_t)poly_xy | (uintptr_t)wsi_poly_xy) & (sizeof(V2) - 1)) == 0 &&
                    (((uintptr_t)centroid | (uintptr_t)wsi_centroid | (uintptr_t)bbox | (uintptr_t)wsi_bbox) & 15) == 0,
             "pg_map_morph: vertex / centroid / bbox arrays must be aligned to their vector width");
  if (n == 0) return PG_OK;
  pg_morph_out o{};
  if (out) o = *out;
  const bool extra = o.major_axis || o.minor_axis || o.centroid_x || o.centroid_y || o.poly_bbox;
  const int blocks = pg_div_up(n, TPB);  // 32 polygons per warp
  // slab per warp: the default holds 32 rings of up to 33 vertices (6 CTAs per SM for float32); tables with longer
  // rings (mean from pg_map_morph_hint - the Python layer knows M) get 32 rings of the mean length + 40 % spread
  int slab_verts = SLAB_VERTS_MIN;
  if (h->morph_mean_verts > 33.0) slab_verts = (int)std::ceil(46.0 * h->morph_mean_verts) + 2;
  else if (h->morph_mean_verts > 0.0 && h->morph_mean_verts <= 23.0)  // short rings: smaller slabs, more CTAs per SM
    slab_verts = std::max(512, (int)std::ceil(40.0 * h->morph_mean_verts) + 2);  // 32 rings of the mean length + 25 %
  slab_verts = std::min(slab_verts, (int)(SLAB_BYTES_MAX / (WARPS * sizeof(V2))));
  slab_verts &= ~1;  // whole 16-byte units per warp
  const size_t smem = (size_t)WARPS * slab_verts * sizeof(V2);
  // 7 CTAs per SM fit shared memory (227 KB minus 1 KB per CTA) -> the 72-register build of the float32 kernel
  // register caps that cost no spills: 6 CTAs per SM for float32 vertices (5 with the extra outputs), 5 / 4 for float64
  constexpr int MINB0 = sizeof(T) == 4 ? 6 : 5, MINB0X = sizeof(T) == 4 ? 5 : 4;
#ifndef PG_MORPH_DENSE
#define PG_MORPH_DENSE 7
#endif
  const bool dense = PG_MORPH_DENSE > 0 && sizeof(T) == 4 && !extra && PG_MORPH_DENSE * (smem + 1024 + 128) <= 227 * 1024;
  auto kern = extra ? map_morph_kernel<T, true, MINB0X> : (dense ? map_morph_kernel<T, false, PG_MORPH_DENSE> : map_morph_kernel<T, false, MINB0>);
  // the opt-in above 48 KB of dynamic shared memory belongs to the DEVICE the handle lives on (cudaFuncSetAttribute
  // acts on the current device only) and SETS the limit rather than raising it: every handle therefore opts in, once,
  // for the one largest size any launch can ask for, so handles sharing a device cannot lower each other's limit
  size_t& granted = h->morph_smem_set[sizeof(T) == 8 ? 1 : 0][extra ? 1 : (dense ? 2 : 0)];
  if (granted == 0) {
    PG_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SLAB_BYTES_MAX));
    granted = SLAB_BYTES_MAX;
  }
  PG_LAUNCH(h, s, extra ? "map_morph_kernel<T, true>" : "map_morph_kernel<T, false>",
            kern<<<blocks, TPB, smem, s>>>(n, poly_off, (const V2*)poly_xy, nuc_tile, tile_x, tile_y,
                                           (const double2*)centroid, (const int4*)bbox, (V2*)wsi_poly_xy,
                                           (double2*)wsi_centroid, (int4*)wsi_bbox, o, slab_verts));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // namespace

extern "C" {

int pg_map_morph_hint(pg_handle* h, int32_t n, int64_t total_vertices) {
  if (!h) return PG_ERR_INVALID;
  PG_REQUIRE(h, n >= 0 && total_vertices >= 0, "pg_map_morph_hint: negative size");
  h->morph_mean_verts = n > 0 ? (double)total_vertices / (double)n : 0.0;
  return PG_OK;
}

int pg_map_morph_f32(pg_handle* h, int32_t n, const int32_t* poly_off, const float* poly_xy, const int32_t* nuc_tile,
                     const int32_t* tile_x, const int32_t* tile_y, const double* centroid, const int32_t* bbox,
                     float* wsi_poly_xy, double* wsi_centroid, int32_t* wsi_bbox, const pg_morph_out* out,
                     pg_stream stream) {
  return launch_map_morph<float>(h, n, poly_off, poly_xy, nuc_tile, tile_x, tile_y, centroid, bbox, wsi_poly_xy,
                                 wsi_centroid, wsi_bbox, out, stream);
}

int pg_map_morph_f64(pg_handle* h, int32_t n, const int32_t* poly_off, const double* poly_xy, const int32_t* nuc_tile,
                     const int32_t* tile_x, const int32_t* tile_y, const double* centroid, const int32_t* bbox,
                     double* wsi_poly_xy, double* wsi_centroid, int32_t* wsi_bbox, const pg_morph_out* out,
                     pg_stream stream) {
  return launch_map_morph<double>(h, n, poly_off, poly_xy, nuc_tile, tile_x, tile_y, centroid, bbox, wsi_poly_xy,
                                  wsi_centroid, wsi_bbox, out, stream);
}

}  // extern "C"
