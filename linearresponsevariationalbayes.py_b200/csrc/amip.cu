// The third derivative of the GLMM KL along one direction, t = D^3 KL[a, a, .] (D), and the per-row quadratic forms
// q_n = a^T (grad^2 l_n) a, fp64, sm_100a (lrvb_glmm_third_contract, DESIGN.md 3e).  With a = H^-1 c they give how
// the LRVB variance c^T H^-1 c moves with the observation weights (the approximate maximum influence perturbation).
//
// Data part: -sum_n w_n D^3 l_n[a, a, .] with l_n = l(z_m, z_v).  z_m is linear in the free parameters; z_v sees
// the exp + lb transform through r(f) = 1 / (e^f + lb) (r', r'', r''' = s, s', s'' on beta.info, d, d', d'' on
// u.info), so its Hessian and third derivative are diagonal.  Per row, the moments along a
//   alpha = j_m.a,  beta1 = j_v.a,  beta2 = a^T grad^2 z_v a = sum_k s'_k x_k^2 a_k^2 + d'_g a_g^2
// and the Gauss-Hermite derivatives of A(z_m, z_v) to third order (the sum differentiated node by node, every node
// function from one exp) give
//   q  = -(A_mm alpha^2 + 2 A_mv alpha beta1 + A_vv beta1^2 + A_v beta2)
//   Cm =   A_mmm alpha^2 + 2 A_mmv alpha beta1 + A_mvv beta1^2 + A_mv beta2
//   Cv =   A_mmv alpha^2 + 2 A_mvv alpha beta1 + A_vvv beta1^2 + A_vv beta2,   Ch = 2 (A_mv alpha + A_vv beta1)
// and t gets  w Cm x_k (beta.mean), w x_k^2 (Cv s_k + Ch s'_k a_k + A_v s''_k a_k^2) (beta.info), w Cm (u.mean_g),
// w (Cv d_g + Ch d'_g a_g + A_v d''_g a_g^2) (u.info_g).
// Non-data part: E[tau] (S / 2 + rate0) with S = sum_g ((mu - u_g)^2 + 1/mu_i + 1/u_i,g), by the product rule, plus
// one-variable terms (entropies, priors, E log tau: psi', psi'', psi''').
// Three kernels, no atomics (repeated calls are bitwise equal):
//   1. k_amip_rows    contiguous row ranges per warp: q, the two per-row group coefficients, and per-CTA partials of
//                     the beta entries (warps summed in order)
//   2. k_amip_group   one warp per group: the u entries of t and five per-group sums of the random-effect term
//   3. k_amip_finish  one CTA: fixed-order sums of the partials, the beta and the four mu / tau entries
#include "common.cuh"
#include "obs_fused.cuh"   // exp_nonpos

namespace lrvb {

struct RDer {
  double d1, d2, d3;
};
// r', r'', r''' of r = 1 / info in the free coordinate f = log(info - lb)
__device__ __forceinline__ RDer r_derivs(double info, double lb) {
  const double e = info - lb, ri = 1.0 / info, r2 = ri * ri;
  RDer o;
  o.d1 = -e * r2;
  o.d2 = e * (e - lb) * r2 * ri;
  o.d3 = e * fma(e, 4.0 * lb - e, -lb * lb) * r2 * r2;
  return o;
}
// d^3/df^3 h(e^f + lb) from h', h'', h''' (e = e^f)
__device__ __forceinline__ double chain3(double h1, double h2, double h3, double e) {
  return e * fma(e, fma(e, h3, 3.0 * h2), h1);
}

// E[tau] = shape / rate and its first two directional derivatives along (a_shape, a_rate) in free coordinates
struct TauE {
  double E, E1, E2;
};
__device__ __forceinline__ TauE tau_e(const double* vec, const double* a, lrvb_glmm_bounds bd) {
  const double sh = vec[2], ra = vec[3], ea = sh - bd.tau_shape, eb = ra - bd.tau_rate, aa = a[2], ab = a[3];
  const double ir = 1.0 / ra;
  const double Ea = ea * ir, Eb = -sh * eb * ir * ir, Eab = -ea * eb * ir * ir;
  const double Ebb = -sh * eb * (ra - 2.0 * eb) * ir * ir * ir;
  TauE o;
  o.E = sh * ir;
  o.E1 = Ea * aa + Eb * ab;
  o.E2 = Ea * aa * aa + 2.0 * Eab * aa * ab + Ebb * ab * ab;
  return o;
}

struct GH3 {
  double S1, P0, P1, P2, R0, R1, R2, R3;   // sum what f(t_q) c_q^p: f = sigma (S), sigma' (P), sigma'' (R)
};
__device__ __forceinline__ void gh3_node(double t, double c, double wq, GH3& s) {
  const double e = exp_nonpos(-fabs(t));
  const double p = 1.0 / (1.0 + e), ep = e * p;
  const double sg = t >= 0.0 ? p : ep, sb = t >= 0.0 ? ep : p;   // sigma(t), 1 - sigma(t)
  const double d1 = sg * sb, d2 = d1 * (sb - sg);
  const double wc = wq * c;
  s.S1 = fma(wc, sg, s.S1);
  s.P0 = fma(wq, d1, s.P0);
  s.P1 = fma(wc, d1, s.P1);
  s.P2 = fma(wc * c, d1, s.P2);
  s.R0 = fma(wq, d2, s.R0);
  s.R1 = fma(wc, d2, s.R1);
  s.R2 = fma(wc * c, d2, s.R2);
  s.R3 = fma(wc * c * c, d2, s.R3);
}

// ---- pass 1 ------------------------------------------------------------------------------
// Shared memory: 8 K-vectors (E[beta], Var[beta], a_beta.mean, s a_bi, s' a_bi^2, s, s' a_bi, s'' a_bi^2), the
// rule, then per warp a 32 x 33 tile of X (coalesced row reads; stride 33: lane = row and lane = column reads
// are both conflict-free), its 2K accumulators and the 4 x 32 row coefficients of the current stage.
constexpr int kAmWarps = 8;
constexpr int kAmTS = 33;
__host__ __device__ constexpr size_t amip_warp_doubles(int K) { return 32 * kAmTS + 2 * (size_t)K + 4 * 32; }
static size_t amip_rows_smem(int K, int Q) {
  return sizeof(double) * (8 * (size_t)K + 2 * (size_t)Q + kAmWarps * amip_warp_doubles(K));
}

__global__ void __launch_bounds__(32 * kAmWarps)
k_amip_rows(const double* __restrict__ X, const int32_t* __restrict__ gid, const double* __restrict__ w,
            const double* __restrict__ vec, const double* __restrict__ a, const double* __restrict__ gh,
            double* __restrict__ q_out, double* __restrict__ rowc, double* __restrict__ part, int64_t N, int K,
            int G, int Q, int64_t rows_per_warp, lrvb_glmm_bounds bd) {
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Dg = 4 + 2 * K;
  double* km = sm;            // E[beta]
  double* kv = km + K;        // Var[beta]
  double* ka = kv + K;        // a on beta.mean
  double* kb = ka + K;        // s a_bi
  double* kc = kb + K;        // s' a_bi^2
  double* kd = kc + K;        // s
  double* ke = kd + K;        // s' a_bi
  double* kf = ke + K;        // s'' a_bi^2
  double* ghc = kf + K;
  double* ghw = ghc + Q;
  double* tile = ghw + Q + (size_t)warp * amip_warp_doubles(K);
  double* acc = tile + 32 * kAmTS;    // 2K: beta.mean | beta.info
  double* coef = acc + 2 * K;         // 4 x 32
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const double bi = vec[4 + K + k], abi = a[4 + K + k];
    const RDer s = r_derivs(bi, bd.beta_info);
    km[k] = vec[4 + k];
    kv[k] = 1.0 / bi;
    ka[k] = a[4 + k];
    kb[k] = s.d1 * abi;
    kc[k] = s.d2 * abi * abi;
    kd[k] = s.d1;
    ke[k] = s.d2 * abi;
    kf[k] = s.d3 * abi * abi;
  }
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    ghc[q] = gh[q];
    ghw[q] = gh[Q + q];
  }
  for (int k = lane; k < 2 * K; k += 32) acc[k] = 0.0;
  __syncthreads();

  const int nch = (K + 31) >> 5;
  const int64_t gw = (int64_t)blockIdx.x * kAmWarps + warp;
  const int64_t rs = gw * rows_per_warp;
  const int64_t re = rs + rows_per_warp < N ? rs + rows_per_warp : N;
  for (int64_t r0 = rs; r0 < re; r0 += 32) {
    const int rows = (int)(re - r0 < 32 ? re - r0 : 32);
    double zm = 0.0, zv = 0.0, al = 0.0, b1 = 0.0, b2 = 0.0;
    for (int c0 = 0; c0 < K; c0 += 32) {
      const int cw = K - c0 < 32 ? K - c0 : 32;
      __syncwarp();
      if (lane < cw)
        for (int r = 0; r < rows; ++r) tile[r * kAmTS + lane] = X[(r0 + r) * K + c0 + lane];
      __syncwarp();
      if (lane < rows)
        for (int c = 0; c < cw; ++c) {
          const double x = tile[lane * kAmTS + c], xx = x * x;
          zm = fma(x, km[c0 + c], zm);
          zv = fma(xx, kv[c0 + c], zv);
          al = fma(x, ka[c0 + c], al);
          b1 = fma(xx, kb[c0 + c], b1);
          b2 = fma(xx, kc[c0 + c], b2);
        }
    }
    double c1 = 0.0, c2 = 0.0, c3 = 0.0, c4 = 0.0;
    if (lane < rows) {
      const int64_t n = r0 + lane;
      const int g = gid[n];
      const double ui = vec[(int64_t)Dg + G + g], aum = a[(int64_t)Dg + g], aui = a[(int64_t)Dg + G + g];
      const RDer d = r_derivs(ui, bd.u_info);
      zm += vec[(int64_t)Dg + g];
      zv += 1.0 / ui;
      al += aum;
      b1 = fma(d.d1, aui, b1);
      b2 = fma(d.d2 * aui, aui, b2);
      const double zs = sqrt(zv);
      GH3 s = {0, 0, 0, 0, 0, 0, 0, 0};
      for (int q = 0; q < Q; ++q) gh3_node(fma(zs, ghc[q], zm), ghc[q], ghw[q], s);
      const double iv = 1.0 / zv, is = 1.0 / zs;
      const double A_v = 0.5 * s.S1 * is;
      const double A_mm = s.P0, A_mv = 0.5 * s.P1 * is, A_vv = 0.25 * (s.P2 - s.S1 * is) * iv;
      const double A_mmm = s.R0, A_mmv = 0.5 * s.R1 * is, A_mvv = 0.25 * (s.R2 - s.P1 * is) * iv;
      const double A_vvv = (0.125 * s.R3 * is - 0.375 * (s.P2 - s.S1 * is) * iv) * iv;
      const double aa = al * al, ab = 2.0 * al * b1, bb = b1 * b1;
      q_out[n] = -(A_mm * aa + A_mv * ab + A_vv * bb + A_v * b2);
      const double wn = w ? w[n] : 1.0;
      c1 = wn * (A_mmm * aa + A_mmv * ab + A_mvv * bb + A_mv * b2);
      c2 = wn * (A_mmv * aa + A_mvv * ab + A_vvv * bb + A_vv * b2);
      c3 = wn * 2.0 * (A_mv * al + A_vv * b1);
      c4 = wn * A_v;
      rowc[n] = c1;
      rowc[N + n] = fma(c2, d.d1, fma(c3 * d.d2, aui, c4 * d.d3 * aui * aui));
    }
    coef[lane] = c1;
    coef[32 + lane] = c2;
    coef[64 + lane] = c3;
    coef[96 + lane] = c4;
    for (int c0 = 0; c0 < K; c0 += 32) {
      const int cw = K - c0 < 32 ? K - c0 : 32;
      __syncwarp();
      if (nch > 1 && lane < cw)   // with one column chunk the tile still holds it
        for (int r = 0; r < rows; ++r) tile[r * kAmTS + lane] = X[(r0 + r) * K + c0 + lane];
      __syncwarp();
      if (lane < cw) {
        const int k = c0 + lane;
        const double fd = kd[k], fe = ke[k], ff = kf[k];
        double sm_ = acc[k], si = acc[K + k];
        for (int r = 0; r < rows; ++r) {
          const double x = tile[r * kAmTS + lane];
          sm_ = fma(coef[r], x, sm_);
          si = fma(x * x, fma(coef[32 + r], fd, fma(coef[64 + r], fe, coef[96 + r] * ff)), si);
        }
        acc[k] = sm_;
        acc[K + k] = si;
      }
    }
  }
  __syncthreads();
  const double* acc0 = ghw + Q + 32 * kAmTS;
  for (int k = threadIdx.x; k < 2 * K; k += blockDim.x) {
    double s = 0.0;
    for (int wi = 0; wi < kAmWarps; ++wi) s += acc0[(size_t)wi * amip_warp_doubles(K) + k];
    part[(size_t)blockIdx.x * 2 * K + k] = s;
  }
}

// ---- pass 2 ------------------------------------------------------------------------------
// One warp per group: the row coefficients summed lane-strided then by warp_sum, plus the non-data terms of u_g.
// gs (5, G): the group's parts of S, S'[a], S''[a, a] and of the mu_m derivatives, (mu - u_g) and (a_mu - a_u,g).
__global__ void __launch_bounds__(256)
k_amip_group(const double* __restrict__ rowc, const int32_t* __restrict__ gptr, const double* __restrict__ vec,
             const double* __restrict__ a, double* __restrict__ t, double* __restrict__ gs, int64_t N, int K, int G,
             lrvb_glmm_bounds bd) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  const int Dg = 4 + 2 * K;
  const TauE te = tau_e(vec, a, bd);
  for (int gi = blockIdx.x * wpb + (threadIdx.x >> 5); gi < G; gi += gridDim.x * wpb) {
    const int64_t nb = gptr[gi], ne = gptr[gi + 1];
    double sm_ = 0.0, si = 0.0;
    for (int64_t n = nb + lane; n < ne; n += 32) {
      sm_ += rowc[n];
      si += rowc[N + n];
    }
    sm_ = warp_sum(sm_);
    si = warp_sum(si);
    if (lane == 0) {
      const double um = vec[Dg + gi], ui = vec[Dg + G + gi], aui = a[Dg + G + gi];
      const double dm = vec[0] - um, da = a[0] - a[Dg + gi];
      const RDer d = r_derivs(ui, bd.u_info);
      const double iu = 1.0 / ui;
      t[Dg + gi] = sm_ - te.E2 * dm - 2.0 * te.E1 * da;
      t[Dg + G + gi] = si + 0.5 * (te.E2 * d.d1 + 2.0 * te.E1 * d.d2 * aui + te.E * d.d3 * aui * aui) +
                       chain3(0.5 * iu, -0.5 * iu * iu, iu * iu * iu, ui - bd.u_info) * aui * aui;
      gs[gi] = dm * dm + iu;
      gs[G + gi] = 2.0 * dm * da + d.d1 * aui;
      gs[2 * G + gi] = 2.0 * da * da + d.d2 * aui * aui;
      gs[3 * G + gi] = dm;
      gs[4 * G + gi] = da;
    }
  }
}

// ---- pass 3 ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_amip_finish(const double* __restrict__ part, int n_part, const double* __restrict__ gs,
              const double* __restrict__ vec, const double* __restrict__ a, double* __restrict__ t, int K, int G,
              lrvb_glmm_prior pr, lrvb_glmm_bounds bd, int include_global) {
  __shared__ double red[32];
  __shared__ double sh[5];
  const int tid = threadIdx.x;
  for (int k = tid; k < K; k += blockDim.x) {
    double sm_ = 0.0, si = 0.0;
    for (int p = 0; p < n_part; ++p) {
      sm_ += part[(size_t)p * 2 * K + k];
      si += part[(size_t)p * 2 * K + K + k];
    }
    if (include_global) {   // entropy + prior of beta_k: (1/2) log i + (beta_info / 2) / i
      const double bi = vec[4 + K + k], ib = 1.0 / bi, abi = a[4 + K + k];
      si += chain3(0.5 * ib - 0.5 * pr.beta_info * ib * ib, -0.5 * ib * ib + pr.beta_info * ib * ib * ib,
                   ib * ib * ib - 3.0 * pr.beta_info * ib * ib * ib * ib, bi - bd.beta_info) * abi * abi;
    }
    t[4 + k] = sm_;
    t[4 + K + k] = si;
  }
  for (int j = 0; j < 5; ++j) {
    double s = 0.0;
    for (int i = tid; i < G; i += blockDim.x) s += gs[(size_t)j * G + i];
    s = block_sum(s, red);
    if (tid == 0) sh[j] = s;
  }
  if (tid != 0) return;
  const double Gl = (double)G, inc = include_global ? 1.0 : 0.0;
  const double mu_i = vec[1], shp = vec[2], ra = vec[3], ai = a[1], aa = a[2], ab = a[3];
  const RDer m = r_derivs(mu_i, bd.mu_info);
  const double S = sh[0] + Gl / mu_i, S_a = sh[1] + Gl * m.d1 * ai, S_aa = sh[2] + Gl * m.d2 * ai * ai;
  const double ea = shp - bd.tau_shape, eb = ra - bd.tau_rate, ir = 1.0 / ra;
  const double Ea = ea * ir, Eb = -shp * eb * ir * ir, Eab = -ea * eb * ir * ir;
  const double Ebb = -shp * eb * (ra - 2.0 * eb) * ir * ir * ir;
  const double Eabb = -ea * eb * (ra - 2.0 * eb) * ir * ir * ir;
  const double Ebbb = -shp * eb * (ra * ra - 6.0 * eb * ra + 6.0 * eb * eb) * ir * ir * ir * ir;
  const TauE te = tau_e(vec, a, bd);
  // E[tau] (S / 2 + rate0): the product rule on (shape, rate) x (mu, u)
  const double St = 0.5 * S + inc * pr.tau_rate, St_a = 0.5 * S_a, St_aa = 0.5 * S_aa;
  double t2 = (Ea * aa * aa + 2.0 * Eab * aa * ab + Eabb * ab * ab) * St + 2.0 * (Ea * aa + Eab * ab) * St_a +
              Ea * St_aa;
  double t3 = (Eab * aa * aa + 2.0 * Eabb * aa * ab + Ebbb * ab * ab) * St + 2.0 * (Eab * aa + Ebb * ab) * St_a +
              Eb * St_aa;
  const double t0 = te.E2 * sh[3] + 2.0 * te.E1 * sh[4];
  double t1 = 0.5 * Gl * (te.E2 * m.d1 + 2.0 * te.E1 * m.d2 * ai + te.E * m.d3 * ai * ai);
  // one-variable terms of shape: -shape - lgamma - (1 - shape) psi (entropy), -cg psi (E log tau of the random
  // effect and the prior); of rate: kb log(rate); of mu_i: (1/2) log i + (mu_info / 2) / i
  const Psi123 ps = polygamma123_pos(shp);
  const double cg = 0.5 * Gl + inc * (pr.tau_shape - 1.0);
  const double g1 = inc * (-1.0 + (shp - 1.0) * ps.p1) - cg * ps.p1;
  const double g2 = inc * (ps.p1 + (shp - 1.0) * ps.p2) - cg * ps.p2;
  const double g3 = inc * (2.0 * ps.p2 + (shp - 1.0) * ps.p3) - cg * ps.p3;
  t2 += chain3(g1, g2, g3, ea) * aa * aa;
  const double kb = 0.5 * Gl + inc * pr.tau_shape;
  t3 += chain3(kb * ir, -kb * ir * ir, 2.0 * kb * ir * ir * ir, eb) * ab * ab;
  if (include_global) {
    const double im = 1.0 / mu_i;
    t1 += chain3(0.5 * im - 0.5 * pr.mu_info * im * im, -0.5 * im * im + pr.mu_info * im * im * im,
                 im * im * im - 3.0 * pr.mu_info * im * im * im * im, mu_i - bd.mu_info) * ai * ai;
  }
  t[0] = t0;
  t[1] = t1;
  t[2] = t2;
  t[3] = t3;
}

// Geometry of pass 1 for N rows: contiguous ranges of a multiple of 32 rows per warp, as many CTAs as fit on the
// chip at once (fewer for small N).  Fixed by (N, K, Q): the order of every sum is too.
struct AmipPlan {
  int grid;
  int64_t rows_per_warp;
  size_t smem;
};
static AmipPlan amip_plan(int64_t N, int K, int Q) {
  AmipPlan p;
  p.smem = amip_rows_smem(K, Q);
  int per_sm = (int)((227 * 1024) / p.smem);
  if (per_sm > 8) per_sm = 8;
  if (per_sm < 1) per_sm = 1;
  const int64_t warps = (int64_t)kNumSMs * per_sm * kAmWarps;
  p.rows_per_warp = 32 * (int64_t)cdiv(cdiv(N, warps), 32);
  if (p.rows_per_warp < 32) p.rows_per_warp = 32;
  p.grid = N > 0 ? cdiv(N, p.rows_per_warp * kAmWarps) : 0;
  return p;
}

// amip_work: rowc (2, N) | part (grid, 2K) | gs (5, G), allocated in the handle on first use
static int ensure_amip_work(lrvb_glmm* h, const AmipPlan& p) {
  if (h->amip_work) return LRVB_OK;
  const size_t nb = sizeof(double) * (2 * (size_t)h->N + (size_t)p.grid * 2 * h->K + 5 * (size_t)h->G + 1);
  if (cudaMalloc(&h->amip_work, nb) != cudaSuccess) {
    cudaGetLastError();
    h->amip_work = nullptr;
    set_error("lrvb_glmm_third_contract: out of device memory (%zu bytes of scratch)", nb);
    return LRVB_ECUDA;
  }
  return LRVB_OK;
}

}  // namespace lrvb

using namespace lrvb;

extern "C" {

int lrvb_glmm_third_contract(lrvb_glmm* h, const double* a_dev, double* t_dev, double* q_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_third_contract: NULL handle");
  LRVB_REQUIRE(a_dev && t_dev && (q_dev || h->N == 0), "lrvb_glmm_third_contract: NULL argument");
  if (!h->point_valid || h->vecmode) {
    set_error("lrvb_glmm_third_contract: no evaluation in free coordinates cached (call lrvb_glmm_eval first)");
    return LRVB_ESTATE;
  }
  const int K = h->K, G = h->G, Q = h->Q;
  const int64_t N = h->N;
  const AmipPlan p = amip_plan(N, K, Q);
  LRVB_TRY(ensure_amip_work(h, p));
  double* rowc = h->amip_work;
  double* part = rowc + 2 * N;
  double* gs = part + (size_t)p.grid * 2 * K;
  const cudaStream_t st = (cudaStream_t)stream;
  if (p.grid > 0) {
    LRVB_TRY(raise_smem_limit(k_amip_rows, p.smem));
    k_amip_rows<<<p.grid, 32 * kAmWarps, p.smem, st>>>(h->X, h->g, h->w, h->vec, a_dev, h->gh, q_dev, rowc, part, N,
                                                       K, G, Q, p.rows_per_warp, h->bounds);
    LRVB_CHECK_LAUNCH();
  }
  if (G > 0) {
    k_amip_group<<<cdiv(G, 8), 256, 0, st>>>(rowc, h->gptr, h->vec, a_dev, t_dev, gs, N, K, G, h->bounds);
    LRVB_CHECK_LAUNCH();
  }
  k_amip_finish<<<1, 256, 0, st>>>(part, p.grid, gs, h->vec, a_dev, t_dev, K, G, h->prior, h->bounds,
                                   h->include_global);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

}  // extern "C"
