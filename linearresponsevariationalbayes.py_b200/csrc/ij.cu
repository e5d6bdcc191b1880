// The "meat" of the infinitesimal-jackknife (IJ) bootstrap covariance of the global parameters, rows or whole groups
// resampled, fp64, sm_100a (lrvb_glmm_ij_meat, DESIGN.md 3f).
//
// The IJ (Giordano et al., "A Swiss Army Infinitesimal Jackknife") approximates the bootstrap covariance of the
// optimum by S^-1 (sum_u V_u V_u^T - s s^T / U) S^-1, s = sum_u V_u, where S^-1 V_u is the global block of H^-1 psi_u
// and psi_u the weighted score of unit u.  For row n of group g, with W_m = W[0, n], W_v = W[1, n] (w_n-weighted):
//   h_n (Dg) = 0 on mu, tau; W_m x on beta.mean; s (.) W_v x^2 on beta.info (s_k = -(i_k - lb) / i_k^2)
//   r_n (2)  = (W_m, d_g W_v) on (u.mean_g, u.info_g) (d_g likewise)
//   V_n = h_n - B_g^T L_g^-1 r_n
// Groups: V_g = sum_{n in g} V_n is k_logo_grad's V (logo.cu), and the meat is V^T V.  Rows: per group,
//   sum_n V_n V_n^T = sum_n h_n h_n^T - B_g^T L_g^-1 E_g - E_g^T L_g^-1 B_g + B_g^T L_g^-1 F_g L_g^-1 B_g
// with E_g = sum_{n in g} r_n h_n^T (2, Dg) and F_g = sum_{n in g} r_n r_n^T (2, 2).  Passes (no atomics, fixed
// reduction orders: repeated calls are bitwise equal; only the handle's IJ scratch and the outputs are written):
//   k_ij_weights      (5, ldw) = (W_m, W_v, W_m^2, W_m W_v, W_v^2)
//   launch_ij_gram    (glmm_eval.cu) rows: the evaluation's Gram kernel on (a, b, c) = rows 2..4 and its finish,
//                     giving -sum_n h_n h_n^T in the meat; k_group<2> on the same rows, giving F_g and the four
//                     sums of E_g before the s / d_g factors
//   k_ij_group_prep   rows: E_g and the per-group 4 x 4 middle [[L^-1 F L^-1, -L^-1], [-L^-1, 0]] of [B_g; E_g]
//   launch_logo_grad  (logo.cu) V (G, Dg)
//   k_ij_colsum_*     s = the column sums of V, in a fixed order
//   k_ij_corr         sum_u Y_u^T M_u Y_u on the FP64 tensor cores (DMMA 8x8x4, one unit's four rows per k-step):
//                     rows: Y_g = [B_g; E_g] with the middle above; groups: four consecutive rows of V, M = I
//   k_ij_corr_finish  fixed-order sum of the k-chunks; meat = corr - (what the meat held)
#include "common.cuh"

namespace lrvb {

size_t ij_gram_parts(const lrvb_glmm* h);
int launch_ij_gram(lrvb_glmm* h, const double* W5, double* part, double* gsc, double* BR, double* A, cudaStream_t st);
int launch_logo_grad(lrvb_glmm* h, double* V, cudaStream_t st);

__global__ void __launch_bounds__(256)
k_ij_weights(const double* __restrict__ W, double* __restrict__ W5, int64_t N, int64_t ldw) {
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
    const double m = W[n], v = W[ldw + n];
    W5[n] = m;
    W5[ldw + n] = v;
    W5[2 * ldw + n] = m * m;
    W5[3 * ldw + n] = m * v;
    W5[4 * ldw + n] = v * v;
  }
}

// One warp per group.  gsc (G, 5) = sums of (W_m, W_v, W_m^2, W_m W_v, W_v^2); BR (G, 4, K) = sums of
// (W_m^2 x, W_m W_v x, W_m W_v x^2, W_v^2 x^2).  Writes E (G, 2, Dg) and mid (G, 6) = (P00, P01, P11, Li00, Li01,
// Li11) with Li = L_g^-1, P = Li F_g Li.
__global__ void __launch_bounds__(256)
k_ij_group_prep(const double* __restrict__ gsc, const double* __restrict__ BR, const double* __restrict__ vec,
                const double* __restrict__ L, double* __restrict__ E, double* __restrict__ mid, int K, int G,
                lrvb_glmm_bounds bd) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int Dg = 4 + 2 * K;
  for (int gi = blockIdx.x * wpb + (threadIdx.x >> 5); gi < G; gi += gridDim.x * wpb) {
    const double info = vec[(int64_t)Dg + G + gi];
    const double dg = -(info - bd.u_info) / (info * info);
    const double l0 = L[(size_t)gi * 3], l1 = L[(size_t)gi * 3 + 1], l2 = L[(size_t)gi * 3 + 2];
    const double det = l0 * l2 - l1 * l1;
    const double i00 = l2 / det, i01 = -l1 / det, i11 = l0 / det;
    const double* gs = gsc + (size_t)gi * 5;
    const double f00 = gs[2], f01 = dg * gs[3], f11 = dg * dg * gs[4];
    if (lane == 0) {
      const double t00 = fma(i00, f00, i01 * f01), t01 = fma(i00, f01, i01 * f11);
      const double t10 = fma(i01, f00, i11 * f01), t11 = fma(i01, f01, i11 * f11);
      double* m = mid + (size_t)gi * 6;
      m[0] = fma(t00, i00, t01 * i01);
      m[1] = fma(t00, i01, t01 * i11);
      m[2] = fma(t10, i01, t11 * i11);
      m[3] = i00;
      m[4] = i01;
      m[5] = i11;
    }
    double* e0 = E + (size_t)gi * 2 * Dg;
    double* e1 = e0 + Dg;
    if (lane < 4) e0[lane] = e1[lane] = 0.0;
    const double* br = BR + (size_t)gi * 4 * K;
    for (int k = lane; k < K; k += 32) {
      const double ik = vec[4 + K + k];
      const double sk = -(ik - bd.beta_info) / (ik * ik);
      e0[4 + k] = br[k];
      e0[4 + K + k] = sk * br[2 * K + k];
      e1[4 + k] = dg * br[K + k];
      e1[4 + K + k] = dg * (sk * br[3 * K + k]);
    }
  }
}

// ---- column sums of V (G, Dg): s ---------------------------------------------------------------
// Block (column block of 32, row chunk): 8 row lanes in a fixed order, then the chunks in order.
__global__ void __launch_bounds__(256, 1)
k_ij_colsum_part(const double* __restrict__ V, double* __restrict__ part, int Dg, int G, int per) {
  __shared__ double red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const int r0 = blockIdx.y * per, r1 = (r0 + per < G) ? r0 + per : G;
  double s = 0.0;
  if (c < Dg)
    for (int g = r0 + ty; g < r1; g += 8) s += V[(size_t)g * Dg + c];
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && c < Dg) {
    double t = red[0][tx];
#pragma unroll
    for (int i = 1; i < 8; ++i) t += red[i][tx];
    part[(size_t)blockIdx.y * Dg + c] = t;
  }
}

__global__ void __launch_bounds__(256)
k_ij_colsum_fin(const double* __restrict__ part, double* __restrict__ sum, int Dg, int nrc) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Dg) return;
  double s = 0.0;
  for (int i = 0; i < nrc; ++i) s += part[(size_t)i * Dg + c];
  sum[c] = s;
}

// ---- sum_u Y_u^T M_u Y_u on DMMA ----------------------------------------------------------------
// Row r of unit p is (r < 2 ? y0 : y1) + p ldp + (r & 1) Dg, read as zero when 4 p + r >= nrows.
struct IjRows {
  const double* y0;
  const double* y1;
  int64_t ldp;
  int64_t nrows;
};

// The k-steps [k0, k1) of one warp job (k_schur's, solve.cu): lane (lc, lr) holds A = Y_p[lr, cola] and
// B = (M_p Y_p)[lr, colb]; with IDENT, M_p = I and B = Y_p[lr, colb].
template <int NI, int NJ, bool TRI, bool IDENT>
__device__ __forceinline__ void ij_ksteps(double (&acc)[kRT][kRT][2], const IjRows Y, const double* __restrict__ mid,
                                          int Dg, const int (&cola)[kRT], const int (&colb)[kRT], int k0, int k1,
                                          int lr) {
  for (int p = k0; p < k1; ++p) {
    const double* base = Y.y0 + (int64_t)p * Y.ldp;
    const double* base1 = Y.y1 + (int64_t)p * Y.ldp;
    const double* mine = (lr < 2 ? base : base1) + (lr & 1) * Dg;
    const bool ok = 4 * (int64_t)p + lr < Y.nrows;
    double fa[kRT], fb[kRT];
#pragma unroll
    for (int i = 0; i < kRT; ++i)
      if (i < NI) fa[i] = (ok && cola[i] < Dg) ? mine[cola[i]] : 0.0;
    if constexpr (IDENT) {
#pragma unroll
      for (int j = 0; j < kRT; ++j)
        if (j < NJ) fb[j] = (ok && colb[j] < Dg) ? mine[colb[j]] : 0.0;
    } else {
      // row lr of [[P, -Li], [-Li, 0]]
      const double* m = mid + (size_t)p * 6;
      const double p00 = m[0], p01 = m[1], p11 = m[2], l00 = m[3], l01 = m[4], l11 = m[5];
      const double c0 = lr == 0 ? p00 : lr == 1 ? p01 : lr == 2 ? -l00 : -l01;
      const double c1 = lr == 0 ? p01 : lr == 1 ? p11 : lr == 2 ? -l01 : -l11;
      const double c2 = lr == 0 ? -l00 : lr == 1 ? -l01 : 0.0;
      const double c3 = lr == 0 ? -l01 : lr == 1 ? -l11 : 0.0;
#pragma unroll
      for (int j = 0; j < kRT; ++j)
        if (j < NJ) {
          const int c = colb[j];
          fb[j] = c < Dg ? fma(c0, base[c], fma(c1, base[Dg + c], fma(c2, base1[c], c3 * base1[Dg + c]))) : 0.0;
        }
    }
#pragma unroll
    for (int i = 0; i < kRT; ++i)
#pragma unroll
      for (int j = 0; j < kRT; ++j)
        if (i < NI && j < NJ && (!TRI || i <= j)) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
  }
}

// A warp per (job, chunk): job = a kRT x kRT rectangle of 8 x 8 output tiles of the upper triangle, chunk = a
// contiguous range of units.  part (n_chunk, n_jobs, kRT^2, 64), live tiles only.
template <bool IDENT>
__global__ void __launch_bounds__(256, 1)
k_ij_corr(IjRows Y, const double* __restrict__ mid, double* __restrict__ part, int Dg, int units, int R, int n_jobs,
          int n_chunk) {
  const int lane = threadIdx.x & 31;
  const int wg = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int job = wg % n_jobs, chunk = wg / n_jobs;
  if (chunk >= n_chunk) return;
  int ri = 0, rem = job;
  while (rem >= R - ri) { rem -= R - ri; ++ri; }
  const int rj = ri + rem;
  const int DT = (Dg + 7) / 8;
  const int lr = lane & 3, lc = lane >> 2;
  double acc[kRT][kRT][2];
#pragma unroll
  for (int i = 0; i < kRT; ++i)
#pragma unroll
    for (int j = 0; j < kRT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  unsigned tmask = 0;
  int cola[kRT], colb[kRT];
#pragma unroll
  for (int i = 0; i < kRT; ++i) {
    cola[i] = 8 * (kRT * ri + i) + lc;
    colb[i] = 8 * (kRT * rj + i) + lc;
#pragma unroll
    for (int j = 0; j < kRT; ++j) {
      const int it = kRT * ri + i, jt = kRT * rj + j;
      if (it < DT && jt < DT && it <= jt) tmask |= 1u << (i * kRT + j);
    }
  }
  const int per = (units + n_chunk - 1) / n_chunk;
  const int k0 = chunk * per, k1 = (k0 + per < units) ? k0 + per : units;
  int ni = DT - kRT * ri, nj = DT - kRT * rj;
  ni = ni > kRT ? kRT : ni;
  nj = nj > kRT ? kRT : nj;
#define LRVB_S(NI, NJ, T) ij_ksteps<NI, NJ, T, IDENT>(acc, Y, mid, Dg, cola, colb, k0, k1, lr)
  if (ri == rj) {
    switch (ni) {
      case 1: LRVB_S(1, 1, true); break;
      case 2: LRVB_S(2, 2, true); break;
      case 3: LRVB_S(3, 3, true); break;
      default: LRVB_S(4, 4, true); break;
    }
  } else {
    switch (nj) {
      case 1: LRVB_S(4, 1, false); break;
      case 2: LRVB_S(4, 2, false); break;
      case 3: LRVB_S(4, 3, false); break;
      default: LRVB_S(4, 4, false); break;
    }
  }
#undef LRVB_S
  double* out = part + ((size_t)chunk * n_jobs + job) * (kRT * kRT * 64);
  const int crow = lane >> 2, ccol = 2 * (lane & 3);
#pragma unroll
  for (int i = 0; i < kRT; ++i)
#pragma unroll
    for (int j = 0; j < kRT; ++j)
      if (tmask & (1u << (i * kRT + j)))
        *reinterpret_cast<double2*>(out + (i * kRT + j) * 64 + crow * 8 + ccol) = make_double2(acc[i][j][0], acc[i][j][1]);
}

// meat[p][q] = meat[q][p] = (sum of the chunks) - meat[p][q], for p <= q: exactly symmetric.  Each (p, q) of the
// upper triangle belongs to one thread, which reads and writes only its own pair.
__global__ void __launch_bounds__(256)
k_ij_corr_finish(const double* __restrict__ part, double* __restrict__ meat, int Dg, int R, int n_jobs, int n_chunk) {
  __shared__ double red[4][64];
  const int job = blockIdx.x / (kRT * kRT), t = blockIdx.x % (kRT * kRT);
  int ri = 0, rem = job;
  while (rem >= R - ri) { rem -= R - ri; ++ri; }
  const int rj = ri + rem;
  const int DT = (Dg + 7) / 8;
  const int it = kRT * ri + t / kRT, jt = kRT * rj + t % kRT;
  if (it >= DT || jt >= DT || it > jt) return;
  const int e = threadIdx.x & 63, ps = threadIdx.x >> 6;
  const double* src = part + ((size_t)job * kRT * kRT + t) * 64 + e;
  const size_t stride = (size_t)n_jobs * kRT * kRT * 64;
  double s = 0.0;
#pragma unroll 8
  for (int c = ps; c < n_chunk; c += 4) s += src[(size_t)c * stride];
  red[ps][e] = s;
  __syncthreads();
  if (ps != 0) return;
  s = (red[0][e] + red[1][e]) + (red[2][e] + red[3][e]);
  const int p = 8 * it + (e >> 3), q = 8 * jt + (e & 7);
  if (p >= Dg || q >= Dg || (it == jt && p > q)) return;
  const double v = s - meat[(size_t)p * Dg + q];
  meat[(size_t)p * Dg + q] = v;
  meat[(size_t)q * Dg + p] = v;
}

// ---- scratch and plan ---------------------------------------------------------------------------
struct IjCorrPlan {
  int R, n_jobs, n_chunk;
};
// k_schur's split: about 16 warps per SM over the jobs and chunks of units
static IjCorrPlan ij_corr_plan(int Dg, int units) {
  IjCorrPlan p;
  const int DT = (Dg + 7) / 8;
  p.R = (DT + kRT - 1) / kRT;
  p.n_jobs = p.R * (p.R + 1) / 2;
  p.n_chunk = (8 * 2 * kNumSMs) / p.n_jobs;
  if (p.n_chunk > units) p.n_chunk = units;
  if (p.n_chunk > 512) p.n_chunk = 512;
  if (p.n_chunk < 1) p.n_chunk = 1;
  return p;
}

// ij_work (doubles, every piece a multiple of 8): W5 (5, ldw) | gsc (G, 5) | BR (G, 4, K) | E (G, 2, Dg) |
// mid (G, 6) | V (G, Dg) | Gram partials | correction partials | column-sum partials (nrc, Dg)
struct IjLayout {
  size_t w5, gsc, br, e, mid, v, gram, corr, colp, total;
  int nrc, per;
};
static size_t up8(size_t n) { return (n + 7) / 8 * 8; }
static IjLayout ij_layout(const lrvb_glmm* h) {
  const size_t G = (size_t)h->G, K = (size_t)h->K, Dg = (size_t)h->Dg;
  IjLayout l;
  l.per = h->G > 0 ? cdiv(h->G, cdiv(h->G, 512) < 64 ? cdiv(h->G, 512) : 64) : 1;
  l.nrc = h->G > 0 ? cdiv(h->G, l.per) : 1;
  const IjCorrPlan pr = ij_corr_plan(h->Dg, h->G), pg = ij_corr_plan(h->Dg, cdiv(h->G, 4));
  const size_t nc = (size_t)(pr.n_chunk > pg.n_chunk ? pr.n_chunk : pg.n_chunk) * pr.n_jobs;
  size_t o = 0;
  l.w5 = o;   o += up8(5 * (size_t)h->ldw);
  l.gsc = o;  o += up8(5 * G);
  l.br = o;   o += up8(4 * K * G);
  l.e = o;    o += up8(2 * Dg * G);
  l.mid = o;  o += up8(6 * G);
  l.v = o;    o += up8(Dg * G);
  l.gram = o; o += up8(ij_gram_parts(h));
  l.corr = o; o += up8(nc * kRT * kRT * 64);
  l.colp = o; o += up8((size_t)l.nrc * Dg);
  l.total = o;
  return l;
}

// allocated and cleared on first use (the Gram kernels leave partial slots they never own untouched, and their
// finish reads them as zero, as with the evaluation's own partial buffer)
static int ensure_ij_work(lrvb_glmm* h, const IjLayout& l, cudaStream_t st) {
  if (h->ij_work) return LRVB_OK;
  if (cudaMalloc(&h->ij_work, sizeof(double) * l.total) != cudaSuccess) {
    cudaGetLastError();
    h->ij_work = nullptr;
    set_error("lrvb_glmm_ij_meat: out of device memory (%zu bytes of scratch)", sizeof(double) * l.total);
    return LRVB_ECUDA;
  }
  LRVB_CUDA(cudaMemsetAsync(h->ij_work, 0, sizeof(double) * l.total, st));
  return LRVB_OK;
}

static int launch_corr(const IjRows& Y, const double* mid, double* part, double* meat, int Dg, int units,
                       cudaStream_t st) {
  if (units == 0) return LRVB_OK;
  const IjCorrPlan p = ij_corr_plan(Dg, units);
  if (mid) k_ij_corr<false><<<cdiv((int64_t)p.n_jobs * p.n_chunk, 8), 256, 0, st>>>(Y, mid, part, Dg, units, p.R,
                                                                                    p.n_jobs, p.n_chunk);
  else k_ij_corr<true><<<cdiv((int64_t)p.n_jobs * p.n_chunk, 8), 256, 0, st>>>(Y, mid, part, Dg, units, p.R,
                                                                               p.n_jobs, p.n_chunk);
  LRVB_CHECK_LAUNCH();
  k_ij_corr_finish<<<p.n_jobs * kRT * kRT, 256, 0, st>>>(part, meat, Dg, p.R, p.n_jobs, p.n_chunk);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

}  // namespace lrvb

using namespace lrvb;

extern "C" {

int lrvb_glmm_ij_meat(lrvb_glmm* h, int32_t unit, double* meat_dev, double* sum_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_ij_meat: NULL handle");
  LRVB_REQUIRE(unit == 0 || unit == 1, "lrvb_glmm_ij_meat: unit must be 0 (rows) or 1 (groups), got %d", (int)unit);
  if (!h->hess_valid || h->vecmode) {
    set_error("lrvb_glmm_ij_meat: no Hessian in free coordinates cached (call lrvb_glmm_eval with order 2)");
    return LRVB_ESTATE;
  }
  LRVB_REQUIRE(meat_dev && sum_dev, "lrvb_glmm_ij_meat: NULL argument");
  const int K = h->K, G = h->G, Dg = h->Dg;
  const int64_t N = h->N;
  const cudaStream_t st = (cudaStream_t)stream;
  if (G == 0) {
    LRVB_CUDA(cudaMemsetAsync(meat_dev, 0, sizeof(double) * Dg * Dg, st));
    LRVB_CUDA(cudaMemsetAsync(sum_dev, 0, sizeof(double) * Dg, st));
    return LRVB_OK;
  }
  const IjLayout l = ij_layout(h);
  LRVB_TRY(ensure_ij_work(h, l, st));
  double* w = h->ij_work;
  double* V = w + l.v;
  LRVB_TRY(launch_logo_grad(h, V, st));
  k_ij_colsum_part<<<dim3(cdiv(Dg, 32), l.nrc), 256, 0, st>>>(V, w + l.colp, Dg, G, l.per);
  LRVB_CHECK_LAUNCH();
  k_ij_colsum_fin<<<cdiv(Dg, 256), 256, 0, st>>>(w + l.colp, sum_dev, Dg, l.nrc);
  LRVB_CHECK_LAUNCH();
  if (unit == 0) {
    if (N > 0) {
      k_ij_weights<<<cdiv(N, 256) < 8 * kNumSMs ? cdiv(N, 256) : 8 * kNumSMs, 256, 0, st>>>(h->W, w + l.w5, N, h->ldw);
      LRVB_CHECK_LAUNCH();
    }
    LRVB_TRY(launch_ij_gram(h, w + l.w5, w + l.gram, w + l.gsc, w + l.br, meat_dev, st));
    k_ij_group_prep<<<cdiv(G, 8), 256, 0, st>>>(w + l.gsc, w + l.br, h->vec, h->L, w + l.e, w + l.mid, K, G, h->bounds);
    LRVB_CHECK_LAUNCH();
    const IjRows Y{h->B, w + l.e, 2 * (int64_t)Dg, 4 * (int64_t)G};
    LRVB_TRY(launch_corr(Y, w + l.mid, w + l.corr, meat_dev, Dg, G, st));
  } else {
    LRVB_CUDA(cudaMemsetAsync(meat_dev, 0, sizeof(double) * Dg * Dg, st));
    const IjRows Y{V, V + 2 * Dg, 4 * (int64_t)Dg, (int64_t)G};
    LRVB_TRY(launch_corr(Y, nullptr, w + l.corr, meat_dev, Dg, cdiv(G, 4), st));
  }
  return LRVB_OK;
}

}  // extern "C"
