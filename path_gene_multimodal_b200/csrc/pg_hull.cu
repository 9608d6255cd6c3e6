// K14: per-ring convex hull over CSR-packed rings -> convex area, solidity = |shoelace area| / convex area, and the
// skimage orientation of the ring's area moments (cell 18 of hovernet_tile_inference.ipynb:2415-2456 asks
// regionprops_table for both; pg_map_morph (K1) computes neither).
//
// The hull is Andrew's monotone chain, which is correct for any point set: approximate_polygon can emit
// self-intersecting rings, so an algorithm for simple polygons (Melkman) is not enough. Orientation tests and hull-area
// terms are float64 differences in a frame at one of the ring's own vertices: on the half-pixel lattice of every
// HoverNeXt vertex they are small multiples of 1/4, so convex area and solidity are exact there.
//
// Work split (K1's): a warp owns 32 consecutive rings = ONE contiguous range of the vertex array.
//   staged path (the range fits the warp's shared-memory slab - every nuclei table): lane 0 brings the range in with
//     one bulk copy; then each LANE handles ITS ring in shared memory: area moments in ring order, then the points in
//     (x, y) order - merged in O(n) from the ring's two x-monotone chains when it has only two (most nuclei), sorted in
//     place otherwise - into a lower and an upper chain whose stacks hold uint16 indices in a second per-warp slab.
//   chain path (a warp whose range exceeds the slab: tissue islands of 10^3..10^5 vertices): the warp takes its rings
//     one at a time. Every vertex starts as a one-point run; level l merges pairs of runs of 2^(l-1) vertices. A run is
//     its lower and upper hull chains, both sorted by (x, y), and the chains of a union are the monotone chains of the
//     linear merge of the two runs' chains, so no level needs a sort. Chains live in the grow-only workspace at the
//     ring's own vertex positions (two ping-pong buffers per chain), so scratch is sized by n_vertices alone.
// Both paths end with the same chains in the same order and sum the hull area the same way.
#include <algorithm>
#include <cmath>
#include "pg_common.cuh"
#include "pg_ring.cuh"

namespace {

constexpr int TPB = 128;
constexpr int WARPS = TPB / 32;
constexpr int SLAB_VERTS_MIN = 32 * 33 + 2;    // 32 rings of 32 vertices, explicitly closed (+1), + alignment slack
constexpr size_t SLAB_BYTES_MAX = 200 * 1024;  // per CTA, vertex slabs and index slabs together
constexpr int IDX_SLACK = 64;                  // index slab entries beyond the vertex slab: 2 per lane (see below)

template <typename V2> __device__ __forceinline__ bool lex_less(V2 a, V2 b) {
  return a.x < b.x || (a.x == b.x && a.y < b.y);
}

// twice the signed area of (o, a, b), > 0 for a left turn
template <typename V2> __device__ __forceinline__ double turn(V2 o, V2 a, V2 b) {
  const double ax = (double)a.x - (double)o.x, ay = (double)a.y - (double)o.y;
  const double bx = (double)b.x - (double)o.x, by = (double)b.y - (double)o.y;
  return ax * by - ay * bx;
}

__device__ __forceinline__ double bfly_add32(double v) {
#pragma unroll
  for (int m = 1; m < 32; m <<= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

// Twice the hull area: the lower chain left to right, then the upper chain right to left, in a frame at the chains'
// common first point (the (x, y)-smallest vertex). L(j) / U(j) give the j-th point of a chain, both left to right.
template <typename V2, typename FL, typename FU>
__device__ __forceinline__ double chain_area2(int nl, int nu, FL L, FU U) {
  const V2 f = L(0);
  double s = 0.0;
  for (int j = 0; j + 1 < nl; ++j) s += turn(f, L(j), L(j + 1));
  for (int j = nu - 1; j > 0; --j) s += turn(f, U(j), U(j - 1));
  return s;
}

// One level of the chain path: merge the (x, y)-sorted chains a [la] and b [lb] and keep the monotone chain of the
// result (lower: left turns only; upper: right turns only), written to out, which is the chain's own stack.
template <typename V2, bool UPPER>
__device__ int merge_chain(const V2* a, int la, const V2* b, int lb, V2* out) {
  int k = 0, ia = 0, ib = 0;
  while (ia < la || ib < lb) {
    V2 p;
    if (ib >= lb || (ia < la && !lex_less(b[ib], a[ia]))) p = a[ia++];
    else p = b[ib++];
    while (k >= 2) {
      const double t = turn(out[k - 2], out[k - 1], p);
      if (UPPER ? t >= 0.0 : t <= 0.0) --k;
      else break;
    }
    out[k++] = p;
  }
  return k;
}

template <typename T, int MINB>
__global__ void __launch_bounds__(TPB, MINB)
ring_hull_kernel(int n, int64_t n_vertices, const int32_t* __restrict__ poly_off,
                 const typename vec2_of<T>::type* __restrict__ poly, pg_hull_out out, int slab_verts,
                 typename vec2_of<T>::type* __restrict__ chain_buf, int2* __restrict__ chain_len) {
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
  PG_ASSERT(wbeg >= 0 && off_last <= n_vertices && nv >= 0);

  // slab: vertex i of the range lives at slab[i], placed with the alignment phase of the global range (as in K1)
  V2* slab_base = reinterpret_cast<V2*>(smem_raw) + (size_t)wid * slab_verts;
  uint16_t* idx_slab = reinterpret_cast<uint16_t*>(reinterpret_cast<V2*>(smem_raw) + (size_t)WARPS * slab_verts) +
                       (size_t)wid * (slab_verts + IDX_SLACK);
  const V2* gsrc = poly + wbeg;
  const int head = (int)(((16u - (uint32_t)((uintptr_t)gsrc & 15u)) & 15u) / sizeof(V2));
  const bool staged = total > 0 && total <= slab_verts - 2;  // warp-uniform
  V2* slab = slab_base + (head ? (int)(16 / sizeof(V2)) - head : 0);  // &slab[head] is 16-byte aligned
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

  ring_sums r;
  r.S = r.Sx = r.Sy = r.Ixx = r.Iyy = r.Ixy = 0; r.P = 0; r.Pd = 0; r.fx = r.fy = 0;
  double hull2 = 0.0;

  if (staged) {
    __syncwarp();  // barrier initialised, hand-moved vertices visible
    if (nbulk > 0) mbar_wait(&s_bar[wid], 0);
    if (nv >= 3) {
      V2* mine = slab + (off0 - wbeg);
      PG_ASSERT(off0 - wbeg + nv <= total);
      // ---- area moments in ring order (before the sort below reorders the slab). Start vertex as in K1: lane l on
      // shared-memory bank l. The same walk finds the (x, y)-extreme vertices and counts the direction changes of
      // the ring in (x, y) order: at most two = the ring is two x-monotone chains.
      constexpr int BANKS = 128 / (int)sizeof(V2);
      const int phase = (int)((smem_u32(mine) / sizeof(V2)) & (BANKS - 1));
      int idx = (lane - phase) & (BANKS - 1);
      if (idx >= nv) idx %= nv;
      V2 v = mine[idx];
      r.fx = (double)v.x; r.fy = (double)v.y;
      const V2 v0 = v;
      const int rot = idx;
      int imin = idx, imax = idx;
      V2 vmin = v, vmax = v;
      int first_dir = 0, last_dir = 0, changes = 0;
      double xa = 0, ya = 0;
      V2 prev = v;
      for (int k = 1; k <= nv; ++k) {
        idx = idx + 1 == nv ? 0 : idx + 1;
        v = k < nv ? mine[idx] : v0;
        if (k < nv) {
          const double xb = (double)v.x - r.fx, yb = (double)v.y - r.fy;
          edge_terms(r, xa, ya, xb, yb);
          xa = xb; ya = yb;
          if (lex_less(v, vmin)) { vmin = v; imin = idx; }
          if (lex_less(vmax, v)) { vmax = v; imax = idx; }
        }
        const int dir = lex_less(prev, v) ? 1 : (lex_less(v, prev) ? -1 : 0);
        if (dir != 0) {
          if (first_dir == 0) first_dir = dir;
          else if (dir != last_dir) ++changes;
          last_dir = dir;
        }
        prev = v;
      }
      if (last_dir != first_dir) ++changes;
      const bool two_chains = changes <= 2;

      // ---- the points in (x, y) order, fed to a lower and an upper monotone chain. Stacks of indices into `mine`:
      // the lower one grows up from stk[0], the upper one down from stk[nv + 1]. Apart from the first and the last
      // point fed so far, a point is on at most one of the two chains, so they never hold more than nv + 2 entries.
      uint16_t* stk = idx_slab + (off0 - wbeg) + 2 * lane;
      const int top = nv + 1;
      // sorted position i lives at mine[at(i)]: rotated like the walk above, so that lanes at the same i of the sort
      // and of the feed loop below sit on different banks
      auto at = [&](int i) { const int q = i + rot; return q >= nv ? q - nv : q; };
      if (!two_chains) {  // in-place Shell sort, gaps 1, 4, 13, 40, ... (Knuth)
        int gap = 1;
        while (3 * gap + 1 < nv) gap = 3 * gap + 1;
#pragma unroll 1
        for (; gap > 0; gap = (gap - 1) / 3) {
#pragma unroll 1
          for (int i = gap; i < nv; ++i) {
            const V2 t = mine[at(i)];
            int j = i;
            while (j >= gap && lex_less(t, mine[at(j - gap)])) { mine[at(j)] = mine[at(j - gap)]; j -= gap; }
            mine[at(j)] = t;
          }
        }
      }
      // two chains: A runs forward from imin to imax, B backward from imin - 1 to imax + 1, both ascending
      const int la = two_chains ? (imax - imin + nv) % nv + 1 : nv;
      const int lb = nv - la;
      int ia = 0, ib = 0, nl = 0, nu = 0;
      V2 lo0 = v0, lo1 = v0, up0 = v0, up1 = v0;  // the two top points of each stack (second, top)
#pragma unroll 1
      for (int k = 0; k < nv; ++k) {
        int i;
        if (!two_chains) {
          i = at(k);
        } else {
          int ja = imin + ia; ja -= ja >= nv ? nv : 0;
          int jb = imin - 1 - ib; jb += jb < 0 ? nv : 0;
          if (ib >= lb || (ia < la && !lex_less(mine[jb], mine[ja]))) { i = ja; ++ia; }
          else { i = jb; ++ib; }
        }
        const V2 p = mine[i];
        while (nl >= 2 && turn(lo0, lo1, p) <= 0.0) {
          --nl; lo1 = lo0;
          if (nl >= 2) lo0 = mine[stk[nl - 2]];
        }
        while (nu >= 2 && turn(up0, up1, p) >= 0.0) {
          --nu; up1 = up0;
          if (nu >= 2) up0 = mine[stk[top - (nu - 2)]];
        }
        PG_ASSERT(nl + nu + 2 <= nv + 2);
        stk[nl++] = (uint16_t)i;
        stk[top - nu++] = (uint16_t)i;
        lo0 = lo1; lo1 = p; up0 = up1; up1 = p;
      }
      hull2 = chain_area2<V2>(nl, nu, [&](int j) { return mine[stk[j]]; }, [&](int j) { return mine[stk[top - j]]; });
    }
  } else {
    // ---- chain path: the whole warp on one ring at a time
    auto bufL = [&](int b) { return chain_buf + (size_t)b * n_vertices; };
    auto bufU = [&](int b) { return chain_buf + (size_t)(2 + b) * n_vertices; };
#pragma unroll 1
    for (int t = 0; t < 32; ++t) {
      const int o = __shfl_sync(0xffffffffu, off0, t);
      const int cnt = __shfl_sync(0xffffffffu, nv, t);
      if (warp_global * 32 + t >= n || cnt < 3) continue;  // warp-uniform
      ring_sums a;
      a.S = a.Sx = a.Sy = a.Ixx = a.Iyy = a.Ixy = 0; a.P = 0; a.Pd = 0;
      const V2 v0 = poly[o];
      for (int e = lane; e < cnt; e += 32) {
        const V2 va = poly[o + e];
        const V2 vb = poly[o + ((e + 1 == cnt) ? 0 : e + 1)];
        const double xa = (double)va.x - (double)v0.x, ya = (double)va.y - (double)v0.y;
        const double xb = (double)vb.x - (double)v0.x, yb = (double)vb.y - (double)v0.y;
        edge_terms(a, xa, ya, xb, yb);
      }
      a.S = bfly_add32(a.S); a.Sx = bfly_add32(a.Sx); a.Sy = bfly_add32(a.Sy);
      a.Ixx = bfly_add32(a.Ixx); a.Iyy = bfly_add32(a.Iyy); a.Ixy = bfly_add32(a.Ixy);

      // level l: runs of 2^l vertices from pairs of runs of 2^(l-1); level 1 reads the ring itself
      int levels = 0;
      while ((1 << levels) < cnt) ++levels;
#pragma unroll 1
      for (int l = 1; l <= levels; ++l) {
        const int w = 1 << l, half = w >> 1;
        const int dst = (l - 1) & 1, src = dst ^ 1;
        for (int pa = lane * w; pa < cnt; pa += 32 * w) {
          const int pb = pa + half;
          const int2 lena = l == 1 ? make_int2(1, 1) : chain_len[o + pa];
          const int2 lenb = pb >= cnt ? make_int2(0, 0) : (l == 1 ? make_int2(1, 1) : chain_len[o + pb]);
          const V2* aL = l == 1 ? poly + o + pa : bufL(src) + o + pa;
          const V2* aU = l == 1 ? poly + o + pa : bufU(src) + o + pa;
          const V2* bL = l == 1 ? poly + o + pb : bufL(src) + o + pb;
          const V2* bU = l == 1 ? poly + o + pb : bufU(src) + o + pb;
          PG_ASSERT(o + pa + lena.x + lenb.x <= n_vertices && o + pa + lena.y + lenb.y <= n_vertices);
          const int nl = merge_chain<V2, false>(aL, lena.x, bL, lenb.x, bufL(dst) + o + pa);
          const int nu = merge_chain<V2, true>(aU, lena.y, bU, lenb.y, bufU(dst) + o + pa);
          PG_ASSERT(nl <= min(w, cnt - pa) && nu <= min(w, cnt - pa));
          chain_len[o + pa] = make_int2(nl, nu);
        }
        __syncwarp();  // this level's chains and lengths visible to every lane
      }
      if (lane == t) {
        const int fin = (levels - 1) & 1;
        const V2* L = bufL(fin) + o;
        const V2* U = bufU(fin) + o;
        const int2 len = chain_len[o];
        r = a;
        r.fx = (double)v0.x; r.fy = (double)v0.y;
        hull2 = chain_area2<V2>(len.x, len.y, [&](int j) { return L[j]; }, [&](int j) { return U[j]; });
      }
      __syncwarp();  // the lanes move on to the next ring's buffers only after lane t has read this one's
    }
  }

  // ---- epilogue: one ring per lane
  if (my_poly >= n) return;
  const double nand_ = __longlong_as_double(0x7ff8000000000000ll);
  const bool ok = nv >= 3;
  const double A = 0.5 * r.S;
  const double area = fabs(A);
  const double cvx = 0.5 * hull2;
  const bool good = ok && A != 0.0;
  if (out.convex_area) out.convex_area[my_poly] = ok ? cvx : nand_;
  if (out.solidity) out.solidity[my_poly] = good && cvx != 0.0 ? area / cvx : nand_;
  if (out.orientation) {
    double o = nand_;
    if (good) {  // skimage: (a, b, c) = (mu_xx, -mu_xy, mu_yy) of the inertia tensor, x = column, y = row
      const double inv = 1.0 / A;
      const double cx = r.Sx * inv * (1.0 / 6.0), cy = r.Sy * inv * (1.0 / 6.0);
      const double mu20 = r.Iyy * inv * (1.0 / 12.0) - cx * cx;
      const double mu02 = r.Ixx * inv * (1.0 / 12.0) - cy * cy;
      const double mu11 = r.Ixy * inv * (1.0 / 24.0) - cx * cy;
      const double ta = mu20, tb = -mu11, tc = mu02;
      o = ta - tc == 0.0 ? (tb < 0.0 ? 0.25 * 3.14159265358979323846 : -0.25 * 3.14159265358979323846)
                         : 0.5 * atan2(-2.0 * tb, tc - ta);
    }
    out.orientation[my_poly] = o;
  }
}

template <typename T>
int launch_ring_hull(pg_handle* h, int32_t n, int64_t n_vertices, const int32_t* poly_off, const T* poly_xy,
                     const pg_hull_out* out, pg_stream stream) {
  if (!h) return PG_ERR_INVALID;
  cudaStream_t s = (cudaStream_t)stream;
  PG_CUDA(h, cudaSetDevice(h->device));
  h->last_stream = s;
  using V2 = typename vec2_of<T>::type;
  PG_REQUIRE(h, n >= 0 && n_vertices >= 0, "pg_ring_hull: negative size");
  PG_REQUIRE(h, n_vertices < ((int64_t)1 << 31), "pg_ring_hull: n_vertices >= 2^31");
  PG_REQUIRE(h, n == 0 || poly_off, "pg_ring_hull: poly_off is NULL");
  PG_REQUIRE(h, n_vertices == 0 || poly_xy, "pg_ring_hull: poly_xy is NULL");
  PG_REQUIRE(h, ((uintptr_t)poly_xy & (sizeof(V2) - 1)) == 0, "pg_ring_hull: poly_xy must be aligned to one vertex");
  if (n == 0) return PG_OK;
  pg_hull_out o{};
  if (out) o = *out;
  // slabs as K1's (mean ring length from n_vertices), each with an index slab of uint16 beside it
  const double mean = (double)n_vertices / (double)n;
  int slab_verts = SLAB_VERTS_MIN;
  if (mean > 33.0) slab_verts = (int)std::ceil(46.0 * mean) + 2;
  else if (mean > 0.0 && mean <= 23.0) slab_verts = std::max(512, (int)std::ceil(40.0 * mean) + 2);
  const size_t per_vert = sizeof(V2) + sizeof(uint16_t);
  slab_verts = (slab_verts + 7) & ~7;  // whole 16-byte units per warp in both slabs
  slab_verts = std::min(slab_verts, (int)((SLAB_BYTES_MAX / WARPS - IDX_SLACK * sizeof(uint16_t)) / per_vert) & ~7);
  const size_t smem = (size_t)WARPS * (slab_verts * per_vert + IDX_SLACK * sizeof(uint16_t));
  // chain path scratch: lower / upper chains x two ping-pong buffers of n_vertices points, and the run lengths
  const size_t chain_bytes = 4 * (size_t)n_vertices * sizeof(V2);
  int rc;
  if ((rc = pg_reserve(h, h->hull, chain_bytes + (size_t)n_vertices * sizeof(int2) + 64))) return rc;
  V2* chain_buf = (V2*)h->hull.p;
  int2* chain_len = (int2*)((char*)h->hull.p + chain_bytes);
  constexpr int MINB = sizeof(T) == 4 ? 4 : 3;
  auto kern = ring_hull_kernel<T, MINB>;
  size_t& granted = h->hull_smem_set[sizeof(T) == 8 ? 1 : 0];
  if (granted == 0) {
    PG_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SLAB_BYTES_MAX));
    granted = SLAB_BYTES_MAX;
  }
  PG_LAUNCH(h, s, "ring_hull_kernel<T>",
            kern<<<pg_div_up(n, TPB), TPB, smem, s>>>(n, n_vertices, poly_off, (const V2*)poly_xy, o, slab_verts,
                                                      chain_buf, chain_len));
  PG_LAUNCH_CHECK(h);
  return PG_OK;
}

}  // namespace

extern "C" {

int pg_ring_hull_f32(pg_handle* h, int32_t n, int64_t n_vertices, const int32_t* poly_off, const float* poly_xy,
                     const pg_hull_out* out, pg_stream stream) {
  return launch_ring_hull<float>(h, n, n_vertices, poly_off, poly_xy, out, stream);
}

int pg_ring_hull_f64(pg_handle* h, int32_t n, int64_t n_vertices, const int32_t* poly_off, const double* poly_xy,
                     const pg_hull_out* out, pg_stream stream) {
  return launch_ring_hull<double>(h, n, n_vertices, poly_off, poly_xy, out, stream);
}

}  // extern "C"
