// Observation pass of the Poisson log-link GLMM, fp64, sm_100a (DESIGN.md 3g).  Included by glmm_eval.cu only: a
// kernel is compiled in the file that launches it.
//
// Under q, eta_n ~ N(m_n, v_n) with m_n = x_n . E[beta] + E[u_g] + o_n (o = the offset) and v_n = x_n^2 . Var[beta]
// + Var[u_g], so E_q[exp(eta_n)] = e_n = exp(m_n + v_n / 2) exactly: no quadrature.  With the weights folded in,
//   E_q log p(y_n | eta_n) = w (y m - e) - w lgamma(y + 1)
//   l_m = w (y - e),  l_v = -w e / 2,  l_mm = -w e,  l_mv = -w e / 2,  l_vv = -w e / 4.
// The constant c = sum_n w_n lgamma(y_n + 1) is computed once at creation (lrvb_glmm_create_poisson) and subtracted
// by CTA 0.  Everything after this pass reads only W (lrvb_glmm_obs_weights), as for the logistic model.
//
// Layout: a CTA of 256 threads walks tiles of R = 256 / S consecutive rows, S = a power of two >= K / 8 (at most 32)
// lanes per row, so every lane of every warp has a row to work on at any K (the logistic k_obs puts lane = column and
// idles 31 of 32 lanes at K = 1).  A lane owns at most 8 columns, the same ones in every tile: x, the E[beta], Var[beta]
// factors of its columns and its share of the gradient partials X^T l_m, S^T l_v stay in registers, so X is read
// once from shared memory and the gradient needs no second pass.  Row r's lanes start at column chunk r mod (K / S)
// (rows of one warp hit different banks).  A full tile is one set of TMA bulk copies (X, y, g and, when given, w and
// the offset) on the stage's mbarrier, kPoStages deep; the last, partial tile of the grid is read with plain loads.
// Fixed-order reductions at the end, no atomics: repeated evaluations are bitwise equal.
#pragma once
#include "common.cuh"
#include "gram_small.cuh"

namespace lrvb {

constexpr int kPoThreads = 256;
constexpr int kPoStages = 4;
constexpr int kPoMaxCols = 8;   // columns per lane

// lanes per row: the smallest power of two with at most kPoMaxCols columns per lane
__host__ __device__ inline int pois_lanes(int K) {
  int s = 1;
  while (s < 32 && s * kPoMaxCols < K) s *= 2;
  return s;
}
__host__ __device__ inline int pois_rows(int K) { return kPoThreads / pois_lanes(K); }
// doubles of one stage: X (R, K) | y (R) | w (R) | offset (R) | g (R int32)
__host__ __device__ inline int pois_stage_elems(int K) {
  const int R = pois_rows(K);
  return R * K + 3 * R + R / 2;
}
inline size_t pois_smem(int K) {
  return sizeof(double) * ((size_t)kPoStages * pois_stage_elems(K) + 32) + 8 * kPoStages;
}

struct PoisArgs {
  const double* X; const double* y; const int32_t* g; const double* w; const double* off;
  const double* vec; int64_t N; int K; int G;
};

// The tile walk shared by the observation and the influence kernels.  NV = 2 (m, v) or 4 (+ the directional
// derivatives dm, dv of the influence pass) dot products per row; coef (NV, K) the per-column factors; per row,
// row(n, valid, dots, x, yn, wn, gi) is called by every lane of the row's group after the dots are complete.
template <int NV, typename RowFn>
__device__ __forceinline__ void pois_walk(const PoisArgs& a, double* sm, const double (&coef)[NV][kPoMaxCols],
                                          int (&col)[kPoMaxCols], RowFn row) {
  const int tid = threadIdx.x, K = a.K;
  const int S = pois_lanes(K), R = kPoThreads / S, NI = (K + S - 1) / S;
  const int r = tid / S, s = tid % S;
  const int se = pois_stage_elems(K);
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(sm + (size_t)kPoStages * se + 32);
  const unsigned bars_u = smem_u32(bars), sm_u = smem_u32(sm);
  const int64_t N = a.N, ntiles = (N + R - 1) / R;
  const unsigned xb = (unsigned)(R * K * sizeof(double)), vb = (unsigned)(R * sizeof(double));
  auto issue = [&](int64_t j) {
    const int64_t t = blockIdx.x + j * gridDim.x;
    if (tid != 0 || t >= ntiles || (t + 1) * R > N) return;
    const int slot = (int)(j % kPoStages);
    const unsigned bar = bars_u + 8 * slot, dst = sm_u + (unsigned)(slot * se * sizeof(double));
    const int64_t n0 = t * R;
    mbar_arrive_expect_tx(bar, xb + vb + vb / 2 + (a.w ? vb : 0) + (a.off ? vb : 0));
    bulk_g2s(dst, a.X + n0 * K, xb, bar);
    bulk_g2s(dst + xb, a.y + n0, vb, bar);
    if (a.w) bulk_g2s(dst + xb + vb, a.w + n0, vb, bar);
    if (a.off) bulk_g2s(dst + xb + 2 * vb, a.off + n0, vb, bar);
    bulk_g2s(dst + xb + 3 * vb, a.g + n0, vb / 2, bar);
  };
  if (tid == 0) {
    for (int p = 0; p < kPoStages; ++p) mbar_init(bars_u + 8 * p, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  for (int j = 0; j < kPoStages; ++j) issue(j);
  for (int64_t j = 0;; ++j) {
    const int64_t t = blockIdx.x + j * gridDim.x;
    if (t >= ntiles) break;
    const int slot = (int)(j % kPoStages);
    double* xs = sm + (size_t)slot * se;
    double* ys = xs + R * K;
    double* ws = ys + R;
    double* os = ws + R;
    int32_t* gs = reinterpret_cast<int32_t*>(os + R);
    const int64_t n0 = t * R;
    const int rows = (int)(N - n0 < R ? N - n0 : R);
    if (rows == R) {
      mbar_wait(bars_u + 8 * slot, (unsigned)(j / kPoStages) & 1u);
    } else {         // the last tile of the grid
      for (int e = tid; e < rows * K; e += kPoThreads) xs[e] = a.X[n0 * K + e];
      for (int e = tid; e < rows; e += kPoThreads) {
        ys[e] = a.y[n0 + e];
        if (a.w) ws[e] = a.w[n0 + e];
        if (a.off) os[e] = a.off[n0 + e];
        gs[e] = a.g[n0 + e];
      }
      __syncthreads();
    }
    const bool valid = r < rows;
    const int gi = valid ? gs[r] : 0;
    double d[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) d[v] = 0.0;
    double x[kPoMaxCols];
    const double* xr = xs + (size_t)r * K;
#pragma unroll
    for (int i = 0; i < kPoMaxCols; ++i) {
      x[i] = 0.0;
      if (i < NI && col[i] < K) {
        x[i] = xr[col[i]];
        const double xx = x[i] * x[i];
#pragma unroll
        for (int v = 0; v < NV; ++v) d[v] = fma((v & 1) ? xx : x[i], coef[v][i], d[v]);
      }
    }
    for (int o = S >> 1; o > 0; o >>= 1) {
#pragma unroll
      for (int v = 0; v < NV; ++v) d[v] += __shfl_xor_sync(0xffffffffu, d[v], o);
    }
    row(n0 + r, valid, d, x, valid ? ys[r] : 0.0, (valid && a.w) ? ws[r] : 1.0, (valid && a.off) ? os[r] : 0.0, gi,
        s);
    __syncthreads();     // the slot is refilled next
    issue(j + kPoStages);
  }
}

// the columns a lane owns (the same in every tile) and their factors E[beta], Var[beta]
__device__ __forceinline__ void pois_columns(const double* __restrict__ vec, int K, int (&col)[kPoMaxCols],
                                             double (&bm)[kPoMaxCols], double (&bv)[kPoMaxCols]) {
  const int S = pois_lanes(K), NI = (K + S - 1) / S;
  const int r = threadIdx.x / S, s = threadIdx.x % S, rot = r % NI;
#pragma unroll
  for (int i = 0; i < kPoMaxCols; ++i) {
    const int c = i + rot < NI ? i + rot : i + rot - NI;
    col[i] = (i < NI) ? S * c + s : K;
    const bool in = col[i] < K;
    bm[i] = in ? vec[4 + col[i]] : 0.0;
    bv[i] = in ? 1.0 / vec[4 + K + col[i]] : 0.0;
  }
}

// Writes W (rows 0-1 at order 1, 0-4 at order 2; ldw the row stride), klpart (n_cta) = per-CTA sums of w (y m - e),
// CTA 0 minus *lgc, and (order >= 1) gradpart (2K, n_cta) = per-CTA X^T l_m, S^T l_v: k_obs's layout.
template <int ORDER>
__global__ void __launch_bounds__(kPoThreads, 2)
k_obs_pois(PoisArgs a, const double* __restrict__ lgc, double* __restrict__ W, int64_t ldw,
           double* __restrict__ klpart, double* __restrict__ gradpart) {
  extern __shared__ __align__(16) double sm[];
  const int K = a.K;
  const int64_t um0 = 4 + 2 * (int64_t)K, ui0 = um0 + a.G;
  int col[kPoMaxCols];
  double coef[2][kPoMaxCols], gm[kPoMaxCols], gv[kPoMaxCols];
  pois_columns(a.vec, K, col, coef[0], coef[1]);
#pragma unroll
  for (int i = 0; i < kPoMaxCols; ++i) gm[i] = gv[i] = 0.0;
  double klacc = 0.0;
  pois_walk<2>(a, sm, coef, col, [&](int64_t n, bool valid, const double (&d)[2], const double (&x)[kPoMaxCols],
                                     double yn, double wn, double on, int gi, int s) {
    const double m = d[0] + a.vec[um0 + gi] + on;
    const double v = d[1] + 1.0 / a.vec[ui0 + gi];
    const double e = exp(fma(0.5, v, m));
    if (!valid) return;
    if (s == 0) klacc += wn * (yn * m - e);
    if (ORDER >= 1) {
      const double lm = wn * (yn - e), we = wn * e, lv = -0.5 * we;
      if (s == 0) {
        W[n] = lm;
        W[ldw + n] = lv;
        if (ORDER >= 2) {
          W[2 * ldw + n] = -we;
          W[3 * ldw + n] = lv;
          W[4 * ldw + n] = -0.25 * we;
        }
      }
#pragma unroll
      for (int i = 0; i < kPoMaxCols; ++i) {
        gm[i] = fma(x[i], lm, gm[i]);
        gv[i] = fma(x[i] * x[i], lv, gv[i]);
      }
    }
  });
  double* red = sm + (size_t)kPoStages * pois_stage_elems(K);
  const double kl = block_sum(klacc, red);
  if (threadIdx.x == 0) klpart[blockIdx.x] = blockIdx.x == 0 ? kl - *lgc : kl;
  if (ORDER >= 1) {
    // per-row-slot partials -> shared memory (the stage buffers: 2 R K <= 2 stages) -> fixed-order sum over the slots
    const int R = pois_rows(K), r = threadIdx.x / pois_lanes(K);
    double* buf = sm;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kPoMaxCols; ++i)
      if (col[i] < K) {
        buf[(size_t)r * 2 * K + col[i]] = gm[i];
        buf[(size_t)r * 2 * K + K + col[i]] = gv[i];
      }
    __syncthreads();
    const size_t gs = gridDim.x;
    for (int k = threadIdx.x; k < 2 * K; k += kPoThreads) {
      double t = 0.0;
      for (int p = 0; p < R; ++p) t += buf[(size_t)p * 2 * K + k];
      gradpart[(size_t)k * gs + blockIdx.x] = t;
    }
  }
}

// Influence of every observation (lrvb_glmm_weight_cross_rmatvec): out[n] = (C^T v)_n = -(l_m dm_n + l_v dv_n) with
// unit weight, dm_n = x_n . v_bm + v_um[g_n], dv_n = x_n^2 . (v_bi dvar/dfree) + v_ui[g_n] dvar_u/dfree.  e_n is
// recomputed from x_n rather than read back from W: dm_n, dv_n need the pass over x_n anyway (two more FMAs per
// element), W holds w_n l_m, which cannot be divided back at a zero weight, and the call then needs only an
// evaluation of order 0.
__global__ void __launch_bounds__(kPoThreads, 2)
k_pois_influence(PoisArgs a, const double* __restrict__ v, double* __restrict__ out, lrvb_glmm_bounds bd,
                 int vecmode) {
  extern __shared__ __align__(16) double sm[];
  const int K = a.K;
  const int64_t um0 = 4 + 2 * (int64_t)K, ui0 = um0 + a.G;
  int col[kPoMaxCols];
  double coef[4][kPoMaxCols];
  pois_columns(a.vec, K, col, coef[0], coef[1]);
#pragma unroll
  for (int i = 0; i < kPoMaxCols; ++i) {
    const bool in = col[i] < K;
    const double ik = in ? a.vec[4 + K + col[i]] : 1.0;
    coef[2][i] = in ? v[4 + col[i]] : 0.0;
    coef[3][i] = in ? v[4 + K + col[i]] * (-1.0 / (ik * ik)) * (vecmode ? 1.0 : ik - bd.beta_info) : 0.0;
  }
  pois_walk<4>(a, sm, coef, col, [&](int64_t n, bool valid, const double (&d)[4], const double (&)[kPoMaxCols],
                                     double yn, double, double on, int gi, int s) {
    const double uinfo = a.vec[ui0 + gi];
    const double m = d[0] + a.vec[um0 + gi] + on;
    const double e = exp(fma(0.5, d[1] + 1.0 / uinfo, m));
    const double dm = d[2] + v[um0 + gi];
    const double dv = d[3] + v[ui0 + gi] * (-1.0 / (uinfo * uinfo)) * (vecmode ? 1.0 : uinfo - bd.u_info);
    if (valid && s == 0) out[n] = -((yn - e) * dm - 0.5 * e * dv);
  });
}

}  // namespace lrvb
