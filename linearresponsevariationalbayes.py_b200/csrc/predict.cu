// Prediction on new rows with mean-field and linear-response (LRVB) variances, fp64, sm_100a.
//
// For a new row x (K) in group g (g = -1: population level, mu in place of u_g), at the point of the
// last evaluation:
//   z_m = E[u_g] + x.E[beta],  z_v = Var[u_g] + x^2.Var[beta],  p = sum what sigma(t_q),
//   p2 = sum what sigma(t_q)^2,  a = dp/dz_m,  b = dp/dz_v      (the training quadrature, obs_fused.cuh)
// and, for the LR pass, j H^-1 j^T with j = dp/dfree, nonzero on beta (a x, b x~) and on the two columns
// of the row's random effect (l = (a, b d_g)).  With the arrowhead blocks of H^-1
//   var = j_b^T P j_b + 2 j_b^T C_g l + l^T Sigma_g l,     P = (H^-1)_{beta beta}
// and, with x~_k = s_k x_k^2, s_k = -(i_k - lb) / i_k^2, the first term splits into three forms that do
// not depend on (a, b):
//   j_b^T P j_b = a^2 x^T P_mm x + 2ab x^T P'_ms x^2 + b^2 x^2^T P'_ss x^2     (P' = P scaled by s)
// which the FP64 tensor cores evaluate for 32 rows at a time as [x | x | x^2] times Bt = [P_mm | P'_ms | P'_ss]
// (K x 3K, built by k_predict_pmat) followed by row dot products with [x | x^2 | x^2].  eta = z_m uses
// a = 1, b = 0.  No per-row intermediate leaves the SM.
//
// Approximate leave-one-out (LOO) over the handle's own training rows (lrvb_glmm_loo, DESIGN.md 3c) runs the LR pass
// with a = 1, b = 0 and a = 0, b = 1 at once: the three quadratic forms, the cross dot products and Sigma_g give
//   Q_n = [j_m; j_v] H^-1 [j_m; j_v]^T,   j_m = d z_m / d free,  j_v = d z_v / d free,
// and with W_m = w_n l_m, W_v = w_n l_v (rows 0, 1 of the handle's W, written by the last evaluation) the infinitesimal
// jackknife moves the row's moments by (dz_m, dz_v) = -Q_n (W_m, W_v).  The epilogue evaluates log E_q[p(y_n | z)]
// by the Gauss-Hermite rule before and after the shift (y = 0 as log E[sigma(-z)]: no cancellation when p -> 1).
//
// Every row's result depends on that row alone and is computed in the same order wherever the row sits
// in a tile, so a permutation of the rows permutes the outputs bitwise.  Rows of one group read the same
// C_g / Sigma_g, which stay in L1 when the rows are visited group by group: `order` (optional) is the
// visiting order, a permutation of [0, M); rows are read from and written to their own places in X, g
// and out, so no sorted copy of X is ever made.
#include "common.cuh"
#include "obs_fused.cuh"

namespace lrvb {

constexpr int kPrRows = 32;        // rows per warp tile (= lanes = 4 DMMA m-tiles)
constexpr int kPrMaxWarps = 16;
#ifndef LRVB_PR_SLOTS
#define LRVB_PR_SLOTS 1
#endif
// cp.async ring slots per warp.  One: the next tile is requested when the current one is done and the other
// warps cover the copy; it fits twice the warps per SM of two slots and was measured faster at K = 20, 50, 200.
constexpr int kPrSlots = LRVB_PR_SLOTS;
// LR pass with K <= kPrSmemK: a compile-time-K kernel with Bt staged in shared memory (once per CTA).  Measured
// (DESIGN.md 3b): 4.01 against 4.15 ms at K = 20, but 14.9 against 11.6 ms at K = 50, where the 81 KB of staged Bt cost
// the SM 5 of its 14 warps and the L2 serves the re-reads of Bt faster than fewer warps hide their latency.
// (-DLRVB_PR_SMEM_K=0 builds the streamed variant for every K, for A/B timing.)
#ifndef LRVB_PR_SMEM_K
#define LRVB_PR_SMEM_K 24
#endif
constexpr int kPrSmemK = LRVB_PR_SMEM_K;

__host__ __device__ constexpr int pr_kp8(int K) { return (K + 7) / 8 * 8; }
__host__ __device__ constexpr int pr_kp4(int K) { return (K + 3) / 4 * 4; }
// row stride of a staged tile: = 4 (mod 8) doubles makes the DMMA A-fragment reads conflict-free
__host__ __device__ constexpr int pr_stride(int K) { return pr_kp8(K) + 4; }
// row stride of Bt staged in shared memory: = 4 (mod 8) doubles makes the B-fragment reads conflict-free
__host__ __device__ constexpr int pr_bstride(int Kp8) { return Kp8 + 4; }
static inline size_t pr_warp_bytes(int K) { return sizeof(double) * kPrSlots * kPrRows * (size_t)pr_stride(K); }
static inline size_t pr_fixed_bytes(int K, int Q, int KP8) {
  return sizeof(double) * (3 * (size_t)K + 2 * (size_t)Q + (KP8 ? 3 * (size_t)KP8 * pr_bstride(KP8) : 0));
}
static inline int pr_warps(int K, int Q, int KP8) {
  int w = (int)((220 * 1024 - pr_fixed_bytes(K, Q, KP8)) / pr_warp_bytes(K));
  if (w > kPrMaxWarps) w = kPrMaxWarps;
  return w < 1 ? 1 : w;
}

// Bt (3 Kp8, Kp4), n-major: Bt[n][k] = B[k][n] of the K x 3K matrix [P_mm | P'_ms | P'_ss], zero padded.
__global__ void __launch_bounds__(256)
k_predict_pmat(const double* __restrict__ Sinv, const double* __restrict__ vec, double* __restrict__ Bt, int K,
               double beta_lb) {
  const int Kp8 = pr_kp8(K), Kp4 = pr_kp4(K), Dg = 4 + 2 * K;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 3 * (int64_t)Kp8 * Kp4) return;
  const int n = (int)(i / Kp4), k = (int)(i % Kp4);
  const int reg = n / Kp8, c = n % Kp8;
  double v = 0.0;
  if (c < K && k < K) {
    const double ic = vec[4 + K + c];
    const double sc = -(ic - beta_lb) / (ic * ic);
    if (reg == 0) {
      v = Sinv[(size_t)(4 + k) * Dg + 4 + c];
    } else if (reg == 1) {
      v = Sinv[(size_t)(4 + k) * Dg + 4 + K + c] * sc;
    } else {
      const double ik = vec[4 + K + k];
      v = (-(ik - beta_lb) / (ik * ik)) * Sinv[(size_t)(4 + K + k) * Dg + 4 + K + c] * sc;
    }
  }
  Bt[i] = v;
}

// cross (G, 2, 2K): cross[g][r][j] = (H^-1)[beta_j, (u.mean_g, u.info_g)_r] = -(Sinv T_g^T)[beta_j, r],
// T_g = L_g^-1 B_g.  One warp per group; T_g in shared memory, Sinv read along rows (it is symmetric).
__global__ void __launch_bounds__(128)
k_predict_cross(const double* __restrict__ Sinv, const double* __restrict__ B, const double* __restrict__ L,
                double* __restrict__ cross, int K, int G) {
  extern __shared__ __align__(16) double tsm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Dg = 4 + 2 * K;
  double* t0 = tsm + (size_t)warp * 2 * Dg;
  double* t1 = t0 + Dg;
  for (int gi = blockIdx.x * 4 + warp; gi < G; gi += gridDim.x * 4) {
    const double l0 = L[(size_t)gi * 3], l1 = L[(size_t)gi * 3 + 1], l2 = L[(size_t)gi * 3 + 2];
    const double det = l0 * l2 - l1 * l1;
    const double i0 = l2 / det, i1 = -l1 / det, i2 = l0 / det;     // k_linv
    const double* b0 = B + (size_t)gi * 2 * Dg;
    const double* b1 = b0 + Dg;
    __syncwarp();
    for (int c = lane; c < Dg; c += 32) {
      t0[c] = i0 * b0[c] + i1 * b1[c];
      t1[c] = i1 * b0[c] + i2 * b1[c];
    }
    __syncwarp();
    double* out = cross + (size_t)gi * 4 * K;
    for (int j = lane; j < 2 * K; j += 32) {
      double s0 = 0.0, s1 = 0.0;
      for (int c = 0; c < Dg; ++c) {
        const double p = Sinv[(size_t)c * Dg + 4 + j];
        s0 = fma(p, t0[c], s0);
        s1 = fma(p, t1[c], s1);
      }
      out[j] = -s0;
      out[2 * K + j] = -s1;
    }
  }
}

// One warp = one 32-row tile at a time (its own cp.async ring, no block barrier in the loop).
// KP8 > 0 (LR, K <= kPrSmemK, K rounded up to 8 == KP8): compile-time loop bounds, and Bt is copied into shared
// memory once per CTA instead of being re-read from L2 by every tile.
//   phase 1  lane = row: z_m, z_v, the four cross dot products, the quadrature, the MFVB outputs
//   phase 2  (LR) the three quadratic forms of 32 rows on the DMMA units, then the LR variances
// out: (4, M) [eta_mean, eta_var_mfvb, prob, prob_var_mfvb] or, LR, (6, M) + [prob_var_lr, eta_var_lr].
// LOO (implies LR; training rows, order = NULL): phase 1 without its quadrature, then the epilogue above reading y and
// W rows 0-1 (row stride ldw); out (4, M) [lpd, lpd_loo, eta_mean_loo, eta_var_loo].  The LOO arguments come last,
// so the other instantiations keep their parameter layout.
template <bool LR, int KP8, bool LOO = false>
__global__ void __launch_bounds__(32 * kPrMaxWarps, 1)
k_predict(const double* __restrict__ X, const int32_t* __restrict__ g, const int64_t* __restrict__ order, int64_t M,
          const double* __restrict__ vec, const double* __restrict__ freev,
          const double* __restrict__ gh, const double* __restrict__ Bt, const double* __restrict__ Sinv,
          const double* __restrict__ cross, const double* __restrict__ lcov, double* __restrict__ out, int K, int G,
          int Q, lrvb_glmm_bounds bd, const double* __restrict__ yv, const double* __restrict__ Wl, int64_t ldw) {
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int S = pr_stride(K), Kp8 = KP8 ? KP8 : pr_kp8(K), Kp4 = pr_kp4(K), Dg = 4 + 2 * K;
  double* ring = sm + (size_t)warp * kPrSlots * kPrRows * S;
  double* bts = sm + (size_t)nwarp * kPrSlots * kPrRows * S;   // KP8: (3 KP8, pr_bstride(KP8)) staged Bt
  double* bm = bts + (KP8 ? 3 * KP8 * pr_bstride(KP8) : 0);    // K  E[beta]
  double* bv = bm + K;                                  // K  Var[beta]
  double* sk = bv + K;                                  // K  s_k = d Var[beta_k] / d free
  double* ghc = sk + K;                                 // Q
  double* ghw = ghc + Q;                                // Q
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const double ik = freev ? exp(freev[4 + K + k]) + bd.beta_info : vec[4 + K + k];
    bm[k] = freev ? freev[4 + k] : vec[4 + k];
    bv[k] = 1.0 / ik;
    sk[k] = -(ik - bd.beta_info) / (ik * ik);
  }
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    ghc[q] = gh[q];
    ghw[q] = gh[Q + q];
  }
  if (KP8) {   // zero beyond k = Kp4 (the k-steps run to KP8)
    constexpr int BS = pr_bstride(KP8 ? KP8 : 8);
    for (int e = threadIdx.x; e < 3 * KP8 * BS; e += blockDim.x) {
      const int n = e / BS, k = e % BS;
      bts[e] = k < Kp4 ? Bt[(size_t)n * Kp4 + k] : 0.0;
    }
  }
  // padding columns [K, Kp8) of every slot stay zero (the copies never touch them)
  for (int e = lane; e < kPrSlots * kPrRows * (Kp8 - K); e += 32) {
    const int r = e / (Kp8 - K), c = K + e % (Kp8 - K);
    ring[(size_t)r * S + c] = 0.0;
  }
  __syncthreads();

  const int64_t ntiles = (M + kPrRows - 1) / kPrRows;
  const int64_t gw = (int64_t)blockIdx.x * nwarp + warp, tw = (int64_t)gridDim.x * nwarp;
  const bool even = (K & 1) == 0;
  auto issue = [&](int64_t t, int slot) {
    if (t < ntiles) {
      double* dst = ring + (size_t)slot * kPrRows * S;
      const int64_t n0 = t * kPrRows;
      const int rows = (int)((M - n0) < kPrRows ? (M - n0) : kPrRows);
      for (int r = 0; r < kPrRows; ++r) {
        double* d = dst + (size_t)r * S;
        if (r < rows) {
          const double* s = X + (order ? order[n0 + r] : n0 + r) * K;
          if (even) {
            for (int c = 2 * lane; c < K; c += 64) cp_async16(d + c, s + c);
          } else {
            for (int c = lane; c < K; c += 32) cp_async8(d + c, s + c);
          }
        } else {
          for (int c = lane; c < K; c += 32) d[c] = 0.0;
        }
      }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  };

#pragma unroll
  for (int p = 0; p < kPrSlots; ++p) issue(gw + p * tw, p);
  int slot = 0;
  for (int64_t t = gw; t < ntiles; t += tw) {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(kPrSlots - 1) : "memory");
    __syncwarp();
    const double* xs = ring + (size_t)slot * kPrRows * S;
    const int64_t n = t * kPrRows + lane;
    const bool valid = n < M;
    const int64_t o = !valid ? 0 : (order ? order[n] : n);   // the row's place in X, g and out

    // ---- phase 1: lane = row ----
    const int gi = valid ? g[o] : -1;
    const bool bad = gi < -1 || gi >= G;
    const bool pop = gi < 0 || bad;
    const int gs = pop ? 0 : gi;
    // the random effect's mean / info: from the free vector (Parameters.py:53-55) or the cached evaluation
    const int64_t im = pop ? 0 : Dg + gs, ii = pop ? 1 : (int64_t)Dg + G + gs;
    const double em = freev ? freev[im] : vec[im];
    const double info = freev ? exp(freev[ii]) + (pop ? bd.mu_info : bd.u_info) : vec[ii];
    double zm = em, zv = 1.0 / info;
    double cm0 = 0.0, cm1 = 0.0, cs0 = 0.0, cs1 = 0.0;
    const double* xr = xs + (size_t)lane * S;
    if (LR) {
      // C_g: rows of cross, or for mu the rows 0 / 1 of Sinv (its beta columns)
      const double* c0 = pop ? Sinv + 4 : cross + (size_t)gs * 4 * K;
      const double* c1 = pop ? Sinv + Dg + 4 : c0 + 2 * K;
      for (int k = 0; k < K; ++k) {
        const double x = xr[k], xx = x * x, xs2 = xx * sk[k];
        zm = fma(x, bm[k], zm);
        zv = fma(xx, bv[k], zv);
        cm0 = fma(x, c0[k], cm0);
        cm1 = fma(x, c1[k], cm1);
        cs0 = fma(xs2, c0[K + k], cs0);
        cs1 = fma(xs2, c1[K + k], cs1);
      }
    } else {
      for (int k = 0; k < K; ++k) {
        const double x = xr[k];
        zm = fma(x, bm[k], zm);
        zv = fma(x * x, bv[k], zv);
      }
    }
    const double zs = sqrt(zv);
    GHSumsF s = {0, 0, 0, 0, 0, 0, 0};
    if (!LOO) gh_all_nodes_f<3, kOfUnroll>(zm, zs, ghc, ghw, Q, s);
    const double p = s.Am;
    const double a = s.Amm, b = s.Ams * (0.5 / zs);
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (valid && !LOO) {
      out[o] = bad ? nan : zm;
      out[M + o] = bad ? nan : zv;
      out[2 * M + o] = bad ? nan : p;
      out[3 * M + o] = bad ? nan : s.App - p * p;
    }

    if (LR) {
      // ---- phase 2: the three quadratic forms of the warp's 32 rows (4 m-tiles of 8) ----
      double qm[4], qs[4], qq[4];
#pragma unroll
      for (int m = 0; m < 4; ++m) qm[m] = qs[m] = qq[m] = 0.0;
      const int nt_reg = Kp8 / 8;                       // n-tiles per region
      const int ar = lane >> 2, ac = lane & 3;
      const int kend = KP8 ? KP8 : Kp4;
#pragma unroll 1
      for (int nt = 0; nt < 3 * nt_reg; ++nt) {
        const int reg = nt / nt_reg;
        const double* bcol = KP8 ? bts + (nt * 8 + ar) * pr_bstride(KP8 ? KP8 : 8) + ac
                                 : Bt + (size_t)(nt * 8 + ar) * Kp4 + ac;
        double c[4][2];
#pragma unroll
        for (int m = 0; m < 4; ++m) c[m][0] = c[m][1] = 0.0;
#pragma unroll(KP8 ? 2 : 4)
        for (int k0 = 0; k0 < kend; k0 += 4) {
          const double bf = KP8 ? bcol[k0] : __ldg(bcol + k0);
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            double af = xs[(size_t)(8 * m + ar) * S + k0 + ac];
            if (reg == 2) af *= af;
            dmma884(c[m][0], c[m][1], af, bf);
          }
        }
        // row dot products with x (region 0) or x^2 (regions 1, 2)
        const int col = (nt - reg * nt_reg) * 8 + 2 * ac;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const double2 u = *reinterpret_cast<const double2*>(xs + (size_t)(8 * m + ar) * S + col);
          const double u0 = reg == 0 ? u.x : u.x * u.x, u1 = reg == 0 ? u.y : u.y * u.y;
          const double d = fma(c[m][1], u1, c[m][0] * u0);
          if (reg == 0) qm[m] += d;
          else if (reg == 1) qs[m] += d;
          else qq[m] += d;
        }
      }
      // reduce over the 4 lanes of a row, then move row 8m + r to lane 8m + r
      double vm = 0.0, vs = 0.0, vq = 0.0;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        qm[m] += __shfl_xor_sync(0xffffffffu, qm[m], 1);
        qm[m] += __shfl_xor_sync(0xffffffffu, qm[m], 2);
        qs[m] += __shfl_xor_sync(0xffffffffu, qs[m], 1);
        qs[m] += __shfl_xor_sync(0xffffffffu, qs[m], 2);
        qq[m] += __shfl_xor_sync(0xffffffffu, qq[m], 1);
        qq[m] += __shfl_xor_sync(0xffffffffu, qq[m], 2);
        const int src = (lane & 7) * 4;
        const double tm = __shfl_sync(0xffffffffu, qm[m], src);
        const double ts = __shfl_sync(0xffffffffu, qs[m], src);
        const double tq = __shfl_sync(0xffffffffu, qq[m], src);
        if ((lane >> 3) == m) { vm = tm; vs = ts; vq = tq; }
      }
      // the random effect's columns: l = (a, b d), Sigma = its 2 x 2 block of H^-1
      double s00, s01, s11, lbo;
      if (pop) {
        s00 = Sinv[0]; s01 = Sinv[1]; s11 = Sinv[Dg + 1]; lbo = bd.mu_info;
      } else {
        s00 = lcov[(size_t)gs * 3]; s01 = lcov[(size_t)gs * 3 + 1]; s11 = lcov[(size_t)gs * 3 + 2]; lbo = bd.u_info;
      }
      const double dg = -(info - lbo) / (info * info);
      const double l0 = a, l1 = b * dg;
      const double quad = a * a * vm + 2.0 * a * b * vs + b * b * vq;
      const double crs = a * (cm0 * l0 + cm1 * l1) + b * (cs0 * l0 + cs1 * l1);
      const double sig = l0 * l0 * s00 + 2.0 * l0 * l1 * s01 + l1 * l1 * s11;
      if (valid && !LOO) {
        out[4 * M + o] = bad ? nan : quad + 2.0 * crs + sig;
        out[5 * M + o] = bad ? nan : vm + 2.0 * cm0 + s00;
      }
      if (LOO) {
        // Q_n: the forms above with (a, b) = (1, 0), (1, 0) x (0, 1) and (0, 1)
        const double qmm = vm + 2.0 * cm0 + s00;
        const double qmv = vs + dg * cm1 + cs0 + dg * s01;
        const double qvv = vq + 2.0 * dg * cs1 + dg * dg * s11;
        const double wm = valid ? Wl[o] : 0.0, wv = valid ? Wl[ldw + o] : 0.0;
        // w_n = 0: W_m = W_v = 0, the shift is exactly zero and both quadratures see the same (z_m, z_s)
        const double zm1 = zm - fma(qmm, wm, qmv * wv);
        const double zv1 = zv - fma(qmv, wm, qvv * wv);
        const bool ok = zv1 > 0.0;    // outside the linearisation's range: NaN, nothing clamped
        const double sgn = (valid && yv[o] == 0.0) ? -1.0 : 1.0;
        GHSumsF s0 = {0, 0, 0, 0, 0, 0, 0}, s1 = {0, 0, 0, 0, 0, 0, 0};
        gh_all_nodes_f<1, kOfUnroll>(sgn * zm, zs, ghc, ghw, Q, s0);
        gh_all_nodes_f<1, kOfUnroll>(sgn * zm1, ok ? sqrt(zv1) : 1.0, ghc, ghw, Q, s1);
        if (valid) {
          out[o] = log(s0.Am);
          out[M + o] = ok ? log(s1.Am) : nan;
          out[2 * M + o] = zm1;
          out[3 * M + o] = ok ? zv1 : nan;
        }
      }
    }
    __syncwarp();   // every lane is done with this slot before the refill
    issue(t + kPrSlots * tw, slot);
    if (++slot == kPrSlots) slot = 0;
  }
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

template <bool LR, int KP8, bool LOO = false>
static int launch_predict(lrvb_glmm* h, const double* freev, const double* X, const int32_t* g, const int64_t* order, int64_t M,
                          const double* Sinv,
                          const double* cross, const double* lcov, double* out, cudaStream_t st) {
  const int K = h->K, Q = h->Q;
  const int warps = pr_warps(K, Q, KP8);
  const size_t smem = warps * pr_warp_bytes(K) + pr_fixed_bytes(K, Q, KP8);
  LRVB_TRY(raise_smem_limit(k_predict<LR, KP8, LOO>, smem));
  int per_sm = 0;
  LRVB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_predict<LR, KP8, LOO>, 32 * warps, smem));
  if (per_sm < 1) per_sm = 1;
  const int64_t ntiles = (M + kPrRows - 1) / kPrRows;
  int64_t grid = (ntiles + warps - 1) / warps;
  if (grid > (int64_t)kNumSMs * per_sm) grid = (int64_t)kNumSMs * per_sm;
  if (LR) {
    const int64_t nb = 3 * (int64_t)pr_kp8(K) * pr_kp4(K);
    k_predict_pmat<<<cdiv(nb, 256), 256, 0, st>>>(Sinv, h->vec, h->pred_B, K, h->bounds.beta_info);
    LRVB_CHECK_LAUNCH();
  }
  k_predict<LR, KP8, LOO><<<(int)grid, 32 * warps, smem, st>>>(X, g, order, M, h->vec, freev, h->gh, h->pred_B, Sinv, cross, lcov,
                                                         out, K, h->G, Q, h->bounds, LOO ? h->y : nullptr,
                                                         LOO ? h->W : nullptr, h->ldw);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

static int check_rows(lrvb_glmm* h, const char* who, const double* X, int32_t K, const int32_t* g, int64_t M,
                      double* out) {
  LRVB_REQUIRE(h != nullptr, "%s: NULL handle", who);
  LRVB_REQUIRE(K == h->K, "%s: X has %d columns, the model has K = %d", who, K, h->K);
  LRVB_REQUIRE(M >= 0, "%s: M = %lld negative", who, (long long)M);
  LRVB_REQUIRE(M == 0 || (X && g && out), "%s: NULL argument", who);
  LRVB_REQUIRE((((uintptr_t)X) & 15) == 0, "%s: X not 16-byte aligned", who);
  return LRVB_OK;
}

// the (3 Kp8, Kp4) scratch of the LR pass, allocated in the handle on first use
static int ensure_pred_B(lrvb_glmm* h, const char* who) {
  if (h->pred_B) return LRVB_OK;
  const size_t nb = 3 * (size_t)pr_kp8(h->K) * pr_kp4(h->K);
  if (cudaMalloc(&h->pred_B, sizeof(double) * nb) != cudaSuccess) {
    cudaGetLastError();
    h->pred_B = nullptr;
    set_error("%s: out of device memory (%zu bytes of scratch)", who, sizeof(double) * nb);
    return LRVB_ECUDA;
  }
  return LRVB_OK;
}

}  // namespace lrvb

using namespace lrvb;

extern "C" {

int lrvb_glmm_predict(lrvb_glmm* h, const double* free_dev, const double* X_dev, int32_t K, const int32_t* g_dev, const int64_t* order_dev,
                      int64_t M, double* out_dev, void* stream) {
  LRVB_TRY(check_rows(h, "lrvb_glmm_predict", X_dev, K, g_dev, M, out_dev));
  LRVB_REQUIRE_LOGISTIC(h, "lrvb_glmm_predict");
  LRVB_REQUIRE(free_dev != nullptr, "lrvb_glmm_predict: free is NULL");
  if (M == 0) return LRVB_OK;
  return launch_predict<false, 0>(h, free_dev, X_dev, g_dev, order_dev, M, nullptr, nullptr, nullptr, out_dev, (cudaStream_t)stream);
}

int lrvb_glmm_predict_cross(lrvb_glmm* h, const double* Sinv_dev, double* cross_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_predict_cross: NULL handle");
  LRVB_REQUIRE(Sinv_dev && (cross_dev || h->G == 0), "lrvb_glmm_predict_cross: NULL argument");
  if (!h->hess_valid || h->vecmode) {
    set_error("lrvb_glmm_predict_cross: no Hessian in free coordinates cached (call lrvb_glmm_eval with order 2)");
    return LRVB_ESTATE;
  }
  if (h->G == 0) return LRVB_OK;
  const size_t smem = sizeof(double) * 4 * 2 * (size_t)h->Dg;
  LRVB_TRY(raise_smem_limit(k_predict_cross, smem));
  int grid = cdiv(h->G, 4);
  if (grid > 8 * kNumSMs) grid = 8 * kNumSMs;
  k_predict_cross<<<grid, 128, smem, (cudaStream_t)stream>>>(Sinv_dev, h->B, h->L, cross_dev, h->K, h->G);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

int lrvb_glmm_predict_lr(lrvb_glmm* h, const double* Sinv_dev, const double* cross_dev, const double* localcov_dev,
                         const double* X_dev, int32_t K, const int32_t* g_dev, const int64_t* order_dev, int64_t M,
                         double* out_dev, void* stream) {
  LRVB_TRY(check_rows(h, "lrvb_glmm_predict_lr", X_dev, K, g_dev, M, out_dev));
  LRVB_REQUIRE_LOGISTIC(h, "lrvb_glmm_predict_lr");
  if (!h->hess_valid || h->vecmode) {
    set_error("lrvb_glmm_predict_lr: no Hessian in free coordinates cached (call lrvb_glmm_eval with order 2)");
    return LRVB_ESTATE;
  }
  LRVB_REQUIRE(Sinv_dev && ((cross_dev && localcov_dev) || h->G == 0), "lrvb_glmm_predict_lr: NULL argument");
  if (M == 0) return LRVB_OK;
  LRVB_TRY(ensure_pred_B(h, "lrvb_glmm_predict_lr"));
  const cudaStream_t st = (cudaStream_t)stream;
#define LRVB_PR_LR(KP) \
  case KP: return launch_predict<true, KP>(h, nullptr, X_dev, g_dev, order_dev, M, Sinv_dev, cross_dev, localcov_dev, out_dev, st);
  switch (h->K <= kPrSmemK ? pr_kp8(h->K) : 0) {
    LRVB_PR_LR(8) LRVB_PR_LR(16) LRVB_PR_LR(24)
    default: return launch_predict<true, 0>(h, nullptr, X_dev, g_dev, order_dev, M, Sinv_dev, cross_dev, localcov_dev, out_dev, st);
  }
#undef LRVB_PR_LR
}

int lrvb_glmm_loo(lrvb_glmm* h, const double* Sinv_dev, const double* cross_dev, const double* localcov_dev,
                  double* out_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_loo: NULL handle");
  LRVB_REQUIRE_LOGISTIC(h, "lrvb_glmm_loo");
  if (!h->hess_valid || h->vecmode) {
    set_error("lrvb_glmm_loo: no Hessian in free coordinates cached (call lrvb_glmm_eval with order 2)");
    return LRVB_ESTATE;
  }
  const int64_t N = h->N;
  LRVB_REQUIRE(Sinv_dev && ((cross_dev && localcov_dev) || h->G == 0) && (out_dev || N == 0),
               "lrvb_glmm_loo: NULL argument");
  if (N == 0) return LRVB_OK;
  LRVB_REQUIRE((((uintptr_t)h->X) & 15) == 0, "lrvb_glmm_loo: the training X is not 16-byte aligned");
  LRVB_TRY(ensure_pred_B(h, "lrvb_glmm_loo"));
  const cudaStream_t st = (cudaStream_t)stream;
  // the training rows are group-sorted already: visited in place, order = NULL
#define LRVB_PR_LOO(KP) \
  case KP: return launch_predict<true, KP, true>(h, nullptr, h->X, h->g, nullptr, N, Sinv_dev, cross_dev, localcov_dev, out_dev, st);
  switch (h->K <= kPrSmemK ? pr_kp8(h->K) : 0) {
    LRVB_PR_LOO(8) LRVB_PR_LOO(16) LRVB_PR_LOO(24)
    default: return launch_predict<true, 0, true>(h, nullptr, h->X, h->g, nullptr, N, Sinv_dev, cross_dev, localcov_dev, out_dev, st);
  }
#undef LRVB_PR_LOO
}

}  // extern "C"
