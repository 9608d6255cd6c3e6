// Internal header: pieces shared by the kernels that walk CSR-packed rings out of a warp's shared-memory slab
// (K1 pg_morph.cu, K14 pg_hull.cu): bulk-copy (TMA) plumbing and the Green's-theorem ring sums.
#pragma once
#include <stdint.h>

namespace {

template <typename T> struct vec2_of;
template <> struct vec2_of<float> { using type = float2; };
template <> struct vec2_of<double> { using type = double2; };

// ---- bulk-copy (TMA) plumbing: 1-D global <-> shared transfers, 16-byte granularity
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "W:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@!p bra W;\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Green's-theorem sums of one ring in a frame at one of its vertices.
struct ring_sums {
  double S, Sx, Sy, Ixx, Iyy, Ixy;
  float P;        // ring length: float32 edge lengths (each within an ulp) summed in float32 over at most 32 edges ...
  double Pd;      // ... and those partial sums in float64, so the error does not grow with the ring (shapely's
                  // p.length is float64: polygon_morphology.py:247-248 measures tissue islands of 10^4..10^5 vertices)
  double fx, fy;  // frame origin
};

// one edge (xa,ya) -> (xb,yb), frame coordinates
__device__ __forceinline__ void edge_terms(ring_sums& r, double xa, double ya, double xb, double yb) {
  const double a = xa * yb - xb * ya;
  const double sxx = xa + xb, syy = ya + yb;
  r.S += a;
  r.Sx += sxx * a;
  r.Sy += syy * a;
  r.Ixx += (syy * syy - ya * yb) * a;             // ya^2 + ya*yb + yb^2
  r.Iyy += (sxx * sxx - xa * xb) * a;             // xa^2 + xa*xb + xb^2
  r.Ixy += (sxx * syy + xa * ya + xb * yb) * a;   // xa*yb + 2xa*ya + 2xb*yb + xb*ya
}

}  // namespace
