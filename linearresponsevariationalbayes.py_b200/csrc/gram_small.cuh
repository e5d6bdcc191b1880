// Packed formulation of the weighted Grams of the beta block on the FP64 tensor cores (DMMA.8x8x4), sm_100a.
//
//   G_a = X^T diag(a) X      G_b = X^T diag(b) S      G_c = S^T diag(c) S        S = X * X
//
// (the second derivatives of sum_n l_n wrt (beta.mean, beta.var); SURVEY.md A.2).  The three
// families are ONE weighted Gram of the packed row z_n = [x_n | s_n] (2K columns) whose weight
// depends on the classes of the two columns: (x,x) -> a, (x,s) -> b, (s,s) -> c.  Packing 2K
// columns into T2 = ceil(2K/8) tiles instead of 2*ceil(K/8) executes 16 instead of 21 DMMAs per
// 4 observations at K = 20.  Only the upper triangle of the packed tile grid is computed.
//
// Tile classes (template parameters): tiles [0, T0) hold x columns only, tile T0 straddles the
// x|s boundary when HAS_M, the remaining tiles hold s columns only.
//   row tile i pure x :  A = z_i                    B = z_j * (a | b by the class of B's column)
//   row tile i pure s :  A = z_i                    B = z_j * c
//   straddle row, straddle column: two DMMAs into one accumulator,
//                        A = z_i masked to its x columns, B = z_j * (a | b)
//                        A = z_i masked to its s columns, B = z_j * c
//   straddle row, pure-s column:   A = z_i * (b | c by the class of A's column),  B = z_j
//
// This header keeps what the packed Gram kernels (gram_mid.cuh, gram_wide.cuh, fused.cuh) and the other
// bulk-copy kernels share: the mbarrier / bulk async copy helpers and the shape of the packed tile grid.
// Their partials use one layout: part (n_cta, NT, 64) with NT = T2 (T2+1) / 2, tile (i <= j) at slot
// j (j+1)/2 + i, element (r, c) of a tile at r * 8 + c.
#pragma once
#include "common.cuh"

namespace lrvb {

// ---- mbarrier + bulk async copy (TMA, SASS UBLKCP) ------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) {
  return (unsigned)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LRVB_MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra LRVB_MBAR_DONE;\n"
      "bra LRVB_MBAR_WAIT;\n"
      "LRVB_MBAR_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// non-blocking: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(unsigned bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}

__device__ __forceinline__ double lds_f64(unsigned addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];\n" : "=d"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ double vmul(double a, double b) {
  double v;
  asm volatile("mul.f64 %0, %1, %2;\n" : "=d"(v) : "d"(a), "d"(b));
  return v;
}

// shape of the packed tile grid for a given K
struct GramSmallShape {
  int T2, T0, has_m, NT;
};
inline GramSmallShape gram_small_shape(int K) {
  GramSmallShape s;
  s.T2 = (2 * K + 7) / 8;
  s.T0 = K / 8;
  s.has_m = (K % 8) != 0;
  s.NT = s.T2 * (s.T2 + 1) / 2;
  return s;
}

}  // namespace lrvb
