// Cross-Hessian of the GLMM objective with the per-observation weights, as an operator.
//
// Replaces, for hyper_par = the observation weights, TwoParameterObjective.fun_hessian_free1_vector2
// as used by ParametricSensitivityLinearApproximation (ModelSensitivity.py:555-612;
// SparseObjectives.py:429-438): the reference forms the dense (D x N) matrix by autodiff, here
//   C = d^2 KL / d free d w ,   column n of C = - grad_free l_n     (KL = -(sum_n w_n l_n + ...))
// is applied without being formed:
//   lrvb_glmm_weight_cross_matvec   out (D) = C dw      one fused observation pass with dw as weights
//   lrvb_glmm_weight_cross_rmatvec  out (N) = C^T v     one quadrature pass, two dot products per row
// both at the point of the last evaluation.  -H^{-1} (C dw) is then the linear response of the
// optimum to a change dw of the weights, and -C^T (H^{-1} v) the influence of every observation on
// the functional v . free (Example.ipynb cells 16-18).
#include "common.cuh"
#include "obs_fused.cuh"

namespace lrvb {

// glmm_eval.cu: the observation and group passes with dw as the weights; the influence pass for K > 62
int launch_weight_pass(lrvb_glmm* h, const double* dw, int* n_gp, cudaStream_t st);
int launch_wide_influence(lrvb_glmm* h, const double* v, double* out, cudaStream_t st);

// out = C dw from the sums of the fused pass run with weights dw (gradpart: X^T l_m, S^T l_v per
// CTA; gsc: per-group sum l_m, sum l_v).  Signs / Jacobians as in k_global / k_local (data terms only).
__global__ void __launch_bounds__(256)
k_wc_finish(const double* __restrict__ vec, const double* __restrict__ gradpart, int n_gp,
            const double* __restrict__ gsc, double* __restrict__ out, int K, int G,
            lrvb_glmm_bounds bd, int vecmode) {
  const int Dg = 4 + 2 * K;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 4) { out[i] = 0.0; return; }          // mu, tau: no data term
  if (i < Dg) {
    const int k = (int)i - 4;                    // 0..K-1 mean, K..2K-1 info
    double s = 0.0;
    for (int p = 0; p < n_gp; ++p) s += gradpart[(size_t)k * n_gp + p];
    if (k < K) {
      out[i] = -s;
    } else {
      const double ik = vec[4 + k];              // beta.info_{k-K} lives at vec[4 + K + (k-K)]
      const double rb = 1.0 / ik;
      out[i] = s * rb * rb * (vecmode ? 1.0 : ik - bd.beta_info);
    }
    return;
  }
  const int64_t j = i - Dg;
  if (j < G) {
    out[i] = -gsc[(size_t)j * 5 + 0];
  } else if (j < 2 * (int64_t)G) {
    const int gi = (int)(j - G);
    const double ui = vec[Dg + G + gi];
    const double r = 1.0 / ui;
    out[i] = gsc[(size_t)gi * 5 + 1] * r * r * (vecmode ? 1.0 : ui - bd.u_info);
  }
}

// out[n] = (C^T v)_n = -(l_m dm_n + l_v dv_n) with unit weight:
//   dm_n = x_n . v_bm + v_um[g_n],   dv_n = x_n^2 . (v_bi dvar/dfree) + v_ui[g_n] dvar_u/dfree.
// Same staging as k_obs_fused (TMA ring per warp, lane = observation, skewed row reads).
__global__ void __launch_bounds__(32 * kOfMaxWarps, 1)
k_obs_influence(const double* __restrict__ X, const double* __restrict__ y, const int32_t* __restrict__ g,
                const double* __restrict__ vec, const double* __restrict__ gh, const double* __restrict__ v,
                double* __restrict__ out, int64_t N, int K, int G, int Q, int64_t rows_per_warp,
                lrvb_glmm_bounds bd, int vecmode) {
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int stage_elems = obs_fused_stage_elems(K);
  const int warp_elems = obs_fused_warp_elems(K);
  double* ring = sm + (size_t)warp * warp_elems;
  double* bm = sm + (size_t)nwarp * warp_elems;   // K   E[beta]
  double* bv = bm + K;                            // K   Var[beta]
  double* ghc = bv + K;                           // Q
  double* ghw = ghc + Q;                          // Q
  double* vm = ghw + Q;                           // K   v on beta.mean
  double* vv = vm + K;                            // K   v on beta.info times d var / d free
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(vv + K + (K & 1)) + warp * kOfStages;
  const unsigned ring_u = smem_u32(ring), bars_u = smem_u32(bars);
  const int Dg = 4 + 2 * K;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const double ik = vec[4 + K + k];
    bm[k] = vec[4 + k];
    bv[k] = 1.0 / ik;
    vm[k] = v[4 + k];
    vv[k] = v[4 + K + k] * (-1.0 / (ik * ik)) * (vecmode ? 1.0 : ik - bd.beta_info);
  }
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    ghc[q] = gh[q];
    ghw[q] = gh[Q + q];
  }
  if (lane == 0) {
#pragma unroll
    for (int p = 0; p < kOfStages; ++p) mbar_init(bars_u + 8 * p, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();

  const int64_t um0 = Dg, ui0 = um0 + G;
  const int64_t gw = (int64_t)blockIdx.x * nwarp + warp;
  const int64_t rs = gw * rows_per_warp;
  const int64_t re = (rs + rows_per_warp < N) ? rs + rows_per_warp : N;
  const int nst = (rs < re) ? (int)((re - rs + kOfRows - 1) / kOfRows) : 0;
  const unsigned xbytes = (unsigned)(kOfRows * K * sizeof(double));
  const unsigned vbytes = (unsigned)(kOfRows * sizeof(double));
  const unsigned gbytes = (unsigned)(kOfRows * sizeof(int32_t));
  auto issue = [&](int st, int slot) {
    const int64_t n0 = rs + (int64_t)st * kOfRows;
    if (st < nst && n0 + kOfRows <= N && lane < 3) {
      const unsigned bar = bars_u + 8 * slot;
      const unsigned dst = ring_u + (unsigned)(slot * stage_elems * sizeof(double));
      if (lane == 0) {
        mbar_arrive_expect_tx(bar, xbytes + vbytes + gbytes);
        bulk_g2s(dst, X + n0 * K, xbytes, bar);
      } else if (lane == 1) {
        bulk_g2s(dst + xbytes, y + n0, vbytes, bar);
      } else {
        bulk_g2s(dst + xbytes + 2 * vbytes, g + n0, gbytes, bar);
      }
    }
  };
  int gcd16 = 1;
  while (gcd16 < 16 && (K % (gcd16 * 2)) == 0) gcd16 *= 2;
  int skew = ((lane & 15) * gcd16) >> 4;
  if (skew >= K) skew = 0;

#pragma unroll
  for (int p = 0; p < kOfStages; ++p) issue(p, p);
  int slot = 0;
  unsigned phase = 0;
  for (int st = 0; st < nst; ++st) {
    const int64_t n0 = rs + (int64_t)st * kOfRows;
    double* xs = ring + (size_t)slot * stage_elems;
    double* ys = xs + kOfRows * K;
    int32_t* gs = reinterpret_cast<int32_t*>(ys + 2 * kOfRows);
    if (n0 + kOfRows <= N) {
      mbar_wait(bars_u + 8 * slot, phase);
    } else {
      const int rows = (int)(N - n0);
      for (int e = lane; e < kOfRows * K; e += 32) xs[e] = (e < rows * K) ? X[n0 * K + e] : 0.0;
      ys[lane] = (lane < rows) ? y[n0 + lane] : 0.0;
      gs[lane] = (lane < rows) ? g[n0 + lane] : 0;
      __syncwarp();
    }
    const int64_t n = n0 + lane;
    const bool valid = n < re;
    const int gi = valid ? gs[lane] : 0;
    const double uinfo = vec[ui0 + gi];
    double zm = vec[um0 + gi];
    double zv = 1.0 / uinfo;
    double dm = v[um0 + gi];
    double dv = v[ui0 + gi] * (-1.0 / (uinfo * uinfo)) * (vecmode ? 1.0 : uinfo - bd.u_info);
    const double* xr = xs + (size_t)lane * K;
    for (int kk = 0; kk < K; ++kk) {
      int k = kk + skew;
      if (k >= K) k -= K;
      const double x = xr[k], xx = x * x;
      zm = fma(x, bm[k], zm);
      zv = fma(xx, bv[k], zv);
      dm = fma(x, vm[k], dm);
      dv = fma(xx, vv[k], dv);
    }
    const double zs = sqrt(zv);
    GHSumsF s = {0, 0, 0, 0, 0, 0}, s2 = {0, 0, 0, 0, 0, 0};
    int q = 0;
    for (; q + 2 <= Q; q += 2) {
      const double c0 = ghc[q], c1 = ghc[q + 1];
      gh_node_f<1>(fma(zs, c0, zm), c0, ghw[q], s);
      gh_node_f<1>(fma(zs, c1, zm), c1, ghw[q + 1], s2);
    }
    if (q < Q) {
      const double c0 = ghc[q];
      gh_node_f<1>(fma(zs, c0, zm), c0, ghw[q], s);
    }
    const double lm = ys[lane] - (s.Am + s2.Am);
    const double lv = -(s.As + s2.As) * (0.5 / zs);
    if (valid) out[n] = -(lm * dm + lv * dv);
    __syncwarp();
    issue(st + kOfStages, slot);
    if (++slot == kOfStages) { slot = 0; phase ^= 1; }
  }
}

}  // namespace lrvb

using namespace lrvb;

extern "C" {

int lrvb_glmm_weight_cross_matvec(lrvb_glmm* h, const double* dw_dev, double* out_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr && out_dev != nullptr && (dw_dev != nullptr || h->N == 0),
               "lrvb_glmm_weight_cross_matvec: NULL argument");
  LRVB_REQUIRE((((uintptr_t)dw_dev) & 15) == 0, "lrvb_glmm_weight_cross_matvec: dw not 16-byte aligned");
  if (!h->point_valid) {
    set_error("lrvb_glmm_weight_cross_matvec: no evaluation cached (call lrvb_glmm_eval first)");
    return LRVB_ESTATE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  int n_gp = 0;
  LRVB_TRY(launch_weight_pass(h, dw_dev, &n_gp, st));
  k_wc_finish<<<cdiv(h->D, 256), 256, 0, st>>>(h->vec, h->gradpart, n_gp, h->gsc, out_dev, h->K, h->G, h->bounds,
                                               h->vecmode);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

int lrvb_glmm_weight_cross_rmatvec(lrvb_glmm* h, const double* v_dev, double* out_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr && v_dev != nullptr && (out_dev != nullptr || h->N == 0),
               "lrvb_glmm_weight_cross_rmatvec: NULL argument");
  if (!h->point_valid) {
    set_error("lrvb_glmm_weight_cross_rmatvec: no evaluation cached (call lrvb_glmm_eval first)");
    return LRVB_ESTATE;
  }
  if (h->N == 0) return LRVB_OK;
  if (!h->obs_fused) return launch_wide_influence(h, v_dev, out_dev, (cudaStream_t)stream);
  const size_t smem = h->of_smem + sizeof(double) * (2 * (size_t)h->K + 2);
  LRVB_TRY(raise_smem_limit(k_obs_influence, smem));
  k_obs_influence<<<h->of_grid, 32 * h->of_warps, smem, (cudaStream_t)stream>>>(
      h->X, h->y, h->g, h->vec, h->gh, v_dev, out_dev, h->N, h->K, h->G, h->Q, h->of_rows_per_warp,
      h->bounds, h->vecmode);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

}  // extern "C"
