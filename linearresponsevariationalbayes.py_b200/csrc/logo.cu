// Approximate leave-one-group-out (LOGO) cross-validation and group influence by the infinitesimal jackknife,
// fp64, sm_100a (lrvb_glmm_logo, DESIGN.md 3d).
//
// Dropping group g is the weight change w_n -> 0 on its rows.  With W_m = w_n l_m, W_v = w_n l_v (rows 0, 1 of the
// handle's W, written by the last evaluation) the data gradient of the group in free coordinates is
//   v_g: sum W_m x on beta.mean, s_k sum W_v x^2 on beta.info (s_k = -(i_k - lb) / i_k^2),
//        sum W_m on u.mean_g, d_g sum W_v on u.info_g (d_g likewise), 0 on mu and tau,
// and the IJ shift of the globals is the global block of -H^-1 v_g; by block elimination on the arrowhead
//   delta_g = -S^-1 V_g,   V_g = v_g,glob - B_g^T L_g^-1 v_g,loc.
// Three passes over the handle's own group-sorted rows, none with atomics (repeated calls are bitwise equal):
//   1. k_logo_grad   one warp per group: V_g (G, Dg) from X and W (not from gsc / BR, which the K > 62
//                    weight-sensitivity pass overwrites)
//   2. k_logo_gemm   Delta = -V S^-1 on the FP64 tensor cores, then Y = Delta_beta P^-1 (P = S^-1 on E[beta])
//                    into the storage of V: Cook's distance is the row dot product Y_g . delta_beta,g / K
//   3. k_logo_rows   one warp per group: the shifted globals mapped exactly to constrained values, q(u_g) at its
//                    closed-form optimum without the group's rows (mean E[mu]', info max(E[tau]', lb_u)), then
//                    lane = row: z_m, z_v and log E_q[p(y_n | z)] by the model's Gauss-Hermite rule (y = 0 as
//                    log E[sigma(-z)]), and the group's sum of them in a fixed order.
#include "common.cuh"
#include "obs_fused.cuh"

namespace lrvb {

// ---- pass 1 ------------------------------------------------------------------------------
// V (G, Dg).  Scalars: lanes over the group's rows, then warp_sum.  Borders: lanes over columns, rows in order
// (the chunk-outer walk of k_group).  An empty group, or one whose rows all have weight 0, gets V_g = 0 exactly.
__global__ void __launch_bounds__(256)
k_logo_grad(const double* __restrict__ X, const double* __restrict__ W, int64_t ldw, const int32_t* __restrict__ gptr,
            const double* __restrict__ vec, const double* __restrict__ B, const double* __restrict__ L,
            double* __restrict__ V, int K, int G, lrvb_glmm_bounds bd) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int Dg = 4 + 2 * K;
  const double* Wm = W;
  const double* Wv = W + ldw;
  for (int gi = blockIdx.x * wpb + (threadIdx.x >> 5); gi < G; gi += gridDim.x * wpb) {
    const int64_t nb = gptr[gi], ne = gptr[gi + 1];
    double sm = 0.0, sv = 0.0;
    for (int64_t n = nb + lane; n < ne; n += 32) {
      sm += Wm[n];
      sv += Wv[n];
    }
    sm = warp_sum(sm);
    sv = warp_sum(sv);
    const double info = vec[(int64_t)Dg + G + gi];
    const double dg = -(info - bd.u_info) / (info * info);
    const double vl0 = sm, vl1 = dg * sv;
    const double l0 = L[(size_t)gi * 3], l1 = L[(size_t)gi * 3 + 1], l2 = L[(size_t)gi * 3 + 2];
    const double det = l0 * l2 - l1 * l1;
    const double t0 = (l2 / det) * vl0 + (-l1 / det) * vl1;     // L_g^-1 v_loc
    const double t1 = (-l1 / det) * vl0 + (l0 / det) * vl1;
    const double* b0 = B + (size_t)gi * 2 * Dg;
    const double* b1 = b0 + Dg;
    double* v = V + (size_t)gi * Dg;
    if (lane < 4) v[lane] = -fma(b0[lane], t0, b1[lane] * t1);
    for (int k = lane; k < K; k += 32) {
      double s0 = 0.0, s1 = 0.0;
      int64_t n = nb;
      for (; n + 4 <= ne; n += 4) {
        double x[4], a[4], c[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          x[u] = X[(n + u) * K + k];
          a[u] = Wm[n + u];
          c[u] = Wv[n + u];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          s0 = fma(a[u], x[u], s0);
          s1 = fma(c[u], x[u] * x[u], s1);
        }
      }
      for (; n < ne; ++n) {
        const double x = X[n * K + k];
        s0 = fma(Wm[n], x, s0);
        s1 = fma(Wv[n], x * x, s1);
      }
      const double ik = vec[4 + K + k];
      const double sk = -(ik - bd.beta_info) / (ik * ik);
      v[4 + k] = s0 - fma(b0[4 + k], t0, b1[4 + k] * t1);
      v[4 + K + k] = sk * s1 - fma(b0[4 + K + k], t0, b1[4 + K + k] * t1);
    }
  }
}

// ---- pass 2 ------------------------------------------------------------------------------
// C (M, N) = alpha A (M, Kd) B (Kd, N), all row-major with leading dimensions lda, ldb, ldc.  A 64 x 64 tile of C
// per CTA, 4 warps of 32 x 32 (4 x 4 DMMA 8x8x4 tiles each), k-steps of 16 staged in shared memory; the next
// k-step is loaded into registers while the current one is multiplied.  Out-of-range entries are read as zero.
constexpr int kLgBM = 64, kLgBN = 64, kLgBK = 16;
constexpr int kLgAS = kLgBK + 4;   // = 4 (mod 8) doubles: conflict-free A-fragment reads
constexpr int kLgBS = kLgBN + 4;   // = 4 (mod 8) doubles: conflict-free B-fragment reads

__global__ void __launch_bounds__(128)
k_logo_gemm(const double* __restrict__ A, int64_t lda, const double* __restrict__ Bm, int64_t ldb,
            double* __restrict__ C, int64_t ldc, int M, int N, int Kd, double alpha) {
  __shared__ __align__(16) double As[kLgBM * kLgAS];
  __shared__ __align__(16) double Bs[kLgBK * kLgBS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wm = warp >> 1, wn = warp & 1, ar = lane >> 2, ac = lane & 3;
  const int64_t m0 = (int64_t)blockIdx.x * kLgBM;
  const int n0 = blockIdx.y * kLgBN;
  double ra[8], rb[8];
  auto load = [&](int k0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = tid + 128 * i;
      const int r = e / kLgBK, c = e % kLgBK;
      ra[i] = (m0 + r < M && k0 + c < Kd) ? A[(m0 + r) * lda + k0 + c] : 0.0;
      const int rr = e / kLgBN, cc = e % kLgBN;
      rb[i] = (k0 + rr < Kd && n0 + cc < N) ? Bm[(int64_t)(k0 + rr) * ldb + n0 + cc] : 0.0;
    }
  };
  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  load(0);
  for (int k0 = 0; k0 < Kd; k0 += kLgBK) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = tid + 128 * i;
      As[(e / kLgBK) * kLgAS + e % kLgBK] = ra[i];
      Bs[(e / kLgBN) * kLgBS + e % kLgBN] = rb[i];
    }
    __syncthreads();
    if (k0 + kLgBK < Kd) load(k0 + kLgBK);
#pragma unroll
    for (int kk = 0; kk < kLgBK; kk += 4) {
      double a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[(wm * 32 + i * 8 + ar) * kLgAS + kk + ac];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[(kk + ac) * kLgBS + wn * 32 + j * 8 + ar];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = m0 + wm * 32 + i * 8 + ar;
    if (r >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = n0 + wn * 32 + j * 8 + 2 * ac;
      if (c < N) C[r * ldc + c] = alpha * acc[i][j][0];
      if (c + 1 < N) C[r * ldc + c + 1] = alpha * acc[i][j][1];
    }
  }
}

static int launch_gemm(const double* A, int64_t lda, const double* Bm, int64_t ldb, double* C, int64_t ldc, int M, int N,
                       int Kd, double alpha, cudaStream_t st) {
  const dim3 grid(cdiv(M, kLgBM), cdiv(N, kLgBN));
  k_logo_gemm<<<grid, 128, 0, st>>>(A, lda, Bm, ldb, C, ldc, M, N, Kd, alpha);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

// ---- pass 3 ------------------------------------------------------------------------------
// One warp per group.  Shared memory per warp: a 32 x 33 tile of X (32 rows x 32 columns, staged with coalesced
// row reads; stride 33 makes the lane = row reads conflict-free) and the group's shifted E[beta]', Var[beta]'.
constexpr int kLgWarps = 4;
constexpr int kLgTS = 33;
__host__ __device__ constexpr size_t logo_warp_doubles(int K) { return 32 * kLgTS + 2 * (size_t)K; }

__global__ void __launch_bounds__(32 * kLgWarps)
k_logo_rows(const double* __restrict__ X, const double* __restrict__ yv, const int32_t* __restrict__ gptr,
            const double* __restrict__ vec, const double* __restrict__ delta, const double* __restrict__ Y,
            const double* __restrict__ gh, double* __restrict__ group_out, double* __restrict__ row_out, int64_t N,
            int K, int G, int Q, lrvb_glmm_bounds bd) {
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Dg = 4 + 2 * K;
  double* ghc = sm;
  double* ghw = ghc + Q;
  double* tile = sm + 2 * Q + (size_t)warp * logo_warp_doubles(K);
  double* bm = tile + 32 * kLgTS;
  double* bv = bm + K;
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    ghc[q] = gh[q];
    ghw[q] = gh[Q + q];
  }
  __syncthreads();
  for (int gi = blockIdx.x * kLgWarps + warp; gi < G; gi += gridDim.x * kLgWarps) {
    const double* dl = delta + (size_t)gi * Dg;
    // the globals at theta + delta_g, mapped to constrained values exactly (info = (i - lb) e^delta + lb)
    double cook = 0.0;
    __syncwarp();   // the previous group's reads of bm / bv are done
    for (int k = lane; k < K; k += 32) {
      const double d = dl[4 + k];
      bm[k] = vec[4 + k] + d;
      bv[k] = 1.0 / fma(vec[4 + K + k] - bd.beta_info, exp(dl[4 + K + k]), bd.beta_info);
      cook = fma(Y[(size_t)gi * K + k], d, cook);
    }
    cook = warp_sum(cook) / K;
    const double emu = vec[0] + dl[0];
    const double shape = fma(vec[2] - bd.tau_shape, exp(dl[2]), bd.tau_shape);
    const double rate = fma(vec[3] - bd.tau_rate, exp(dl[3]), bd.tau_rate);
    const double vu = 1.0 / fmax(shape / rate, bd.u_info);   // q(u_g) without its rows: info max(E[tau]', lb_u)
    __syncwarp();
    const int64_t nb = gptr[gi], ne = gptr[gi + 1];
    double elpd = 0.0;
    for (int64_t r0 = nb; r0 < ne; r0 += 32) {
      const int rows = (int)(ne - r0 < 32 ? ne - r0 : 32);
      double zm = emu, zv = vu;
      for (int c0 = 0; c0 < K; c0 += 32) {
        const int cw = K - c0 < 32 ? K - c0 : 32;
        if (lane < cw)
          for (int r = 0; r < rows; ++r) tile[r * kLgTS + lane] = X[(r0 + r) * K + c0 + lane];
        __syncwarp();
        if (lane < rows)
          for (int c = 0; c < cw; ++c) {
            const double x = tile[lane * kLgTS + c];
            zm = fma(x, bm[c0 + c], zm);
            zv = fma(x * x, bv[c0 + c], zv);
          }
        __syncwarp();
      }
      if (lane < rows) {
        const int64_t n = r0 + lane;
        const double sgn = yv[n] == 0.0 ? -1.0 : 1.0;
        GHSumsF s = {0, 0, 0, 0, 0, 0, 0};
        gh_all_nodes_f<1, kOfUnroll>(sgn * zm, sqrt(zv), ghc, ghw, Q, s);
        const double lpd = log(s.Am);
        row_out[n] = lpd;
        row_out[N + n] = zm;
        row_out[2 * N + n] = zv;
        elpd += lpd;
      }
    }
    elpd = warp_sum(elpd);
    if (lane == 0) {
      group_out[gi] = cook;
      group_out[G + gi] = elpd;
    }
  }
}

// V (G, Dg), allocated in the handle on first use; after pass 2's first product it holds Y (G, K)
static int ensure_logo_V(lrvb_glmm* h) {
  if (h->logo_V) return LRVB_OK;
  const size_t nb = (size_t)h->G * h->Dg;
  if (cudaMalloc(&h->logo_V, sizeof(double) * nb) != cudaSuccess) {
    cudaGetLastError();
    h->logo_V = nullptr;
    set_error("lrvb_glmm_logo: out of device memory (%zu bytes of scratch)", sizeof(double) * nb);
    return LRVB_ECUDA;
  }
  return LRVB_OK;
}

}  // namespace lrvb

using namespace lrvb;

extern "C" {

int lrvb_glmm_logo(lrvb_glmm* h, const double* Sinv_dev, const double* Pinv_dev, double* delta_dev,
                   double* group_out_dev, double* row_out_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_logo: NULL handle");
  if (!h->hess_valid || h->vecmode) {
    set_error("lrvb_glmm_logo: no Hessian in free coordinates cached (call lrvb_glmm_eval with order 2)");
    return LRVB_ESTATE;
  }
  const int K = h->K, G = h->G, Dg = h->Dg, Q = h->Q;
  const int64_t N = h->N;
  LRVB_REQUIRE(Sinv_dev && Pinv_dev && ((delta_dev && group_out_dev) || G == 0) && (row_out_dev || N == 0),
               "lrvb_glmm_logo: NULL argument");
  if (G == 0) return LRVB_OK;
  LRVB_TRY(ensure_logo_V(h));
  const cudaStream_t st = (cudaStream_t)stream;
  k_logo_grad<<<cdiv(G, 8), 256, 0, st>>>(h->X, h->W, h->ldw, h->gptr, h->vec, h->B, h->L, h->logo_V, K, G, h->bounds);
  LRVB_CHECK_LAUNCH();
  // S^-1 is symmetric: Delta = -V S^-1 holds -S^-1 V_g in row g
  LRVB_TRY(launch_gemm(h->logo_V, Dg, Sinv_dev, Dg, delta_dev, Dg, G, Dg, Dg, -1.0, st));
  LRVB_TRY(launch_gemm(delta_dev + 4, Dg, Pinv_dev, K, h->logo_V, K, G, K, K, 1.0, st));
  const size_t smem = sizeof(double) * (2 * (size_t)Q + kLgWarps * logo_warp_doubles(K));
  LRVB_TRY(raise_smem_limit(k_logo_rows, smem));
  k_logo_rows<<<cdiv(G, kLgWarps), 32 * kLgWarps, smem, st>>>(h->X, h->y, h->gptr, h->vec, delta_dev, h->logo_V, h->gh,
                                                              group_out_dev, row_out_dev, N, K, G, Q, h->bounds);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

}  // extern "C"
