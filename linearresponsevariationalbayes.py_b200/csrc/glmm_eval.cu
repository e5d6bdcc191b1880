// ELBO (KL) value, gradient and arrowhead Hessian blocks of the logistic GLMM, fp64, sm_100a.
//
// Replaces, for the composed GLMM objective (SURVEY.md A.1/A.2), what the reference obtains by
// running autograd over Modeling.py:35-52 (get_e_logistic_term_guass_hermite),
// ExponentialFamilies.py:23-35,111-112,186-195 and the constraining transforms of
// Parameters.py:47-61, i.e. Objective.fun_free / fun_free_grad / fun_free_hessian
// (SparseObjectives.py:120-158) plus convert_vector_to_free_hessian (Parameters.py:397-424).
//
// Pipeline of one evaluation (all on one stream, no atomics, fixed reduction orders so the
// result is bitwise reproducible for a given launch geometry):
//   k_prep          free -> constrained vector
//   observation pass: z_mean/z_var, Gauss-Hermite softplus / sigma / sigma', analytic l, dl, d2l; per-CTA
//                   partials of KL and of X^T l_m, S^T l_v; per-group segmented sums (observations are
//                   group-sorted): scalars + borders
//     K <= 24, order 2   k_fused_eval (fused.cuh) also computes the Gram: one pass over X
//     K <= 62            k_obs_fused (obs_fused.cuh), one-slot rings
//     K > 62             k_obs, then k_group
//   Gram            X^T diag(a) X, X^T diag(b) S, S^T diag(c) S on the FP64 tensor cores (DMMA), order 2:
//                   k_gram_mid (K <= 104), k_gram_wide (gram_wide_eligible), k_gram_big (the rest)
//   k_finish, k_global_post   straddling-group fix-up, chain rule to free coordinates, non-data terms
#include <stdlib.h>
#include "common.cuh"
#include "gram_small.cuh"
#include "obs_fused.cuh"
#include "gram_mid.cuh"
#define LRVB_GRAM_BIG_KERNELS
#include "gram_big.cuh"
#define LRVB_GRAM_WIDE_KERNELS
#include "gram_wide.cuh"
#include "fused.cuh"

namespace lrvb {

// ------------------------------------------------------------------------------------------
// shard_G > 0: free_v is the full flat vector of a sharded job with shard_G groups of which this
// handle owns [shard_g0, shard_g0 + G); the gather into the local layout happens here.
__global__ void k_prep(const double* __restrict__ free_v, double* __restrict__ vec, int K, int G,
                       lrvb_glmm_bounds bd, int vecmode, double* __restrict__ zero, int64_t nzero,
                       int64_t shard_g0, int64_t shard_G) {
  pdl_sync();
  const int64_t D = 4 + 2 * (int64_t)K + 2 * (int64_t)G;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // the global Hessian block starts from zero (order 2): cleared here instead of by a memset node,
  // which would cut the chain of programmatic launches
  for (int64_t j = i; j < nzero; j += (int64_t)gridDim.x * blockDim.x) zero[j] = 0.0;
  if (i >= D) return;
  int64_t si = i;
  if (shard_G > 0 && i >= 4 + 2 * K) si = (i < 4 + 2 * K + G) ? i + shard_g0 : i - G + shard_G + shard_g0;
  const double f = free_v[si];
  double lb = 0.0;
  bool con = true;
  if (i == 0) con = false;
  else if (i == 1) lb = bd.mu_info;
  else if (i == 2) lb = bd.tau_shape;
  else if (i == 3) lb = bd.tau_rate;
  else if (i < 4 + K) con = false;
  else if (i < 4 + 2 * K) lb = bd.beta_info;
  else if (i < 4 + 2 * K + G) con = false;
  else lb = bd.u_info;
  const double v = (con && !vecmode) ? exp(f) + lb : f;   // Parameters.py:53-55
  vec[i] = v;
  // factors the finishing pass would otherwise re-derive with an fp64 division per (group, column):
  // aux = vec + D: [E tau = a/b, 1/b, a/b^2, -, -, -, -, - | -1/beta.info_k^2 (K) | 1/u.info_g^2 (G)]
  double* aux = vec + D;
  if (i == 3) {
    const double a = vecmode ? free_v[2] : exp(free_v[2]) + bd.tau_shape;
    const double ib = 1.0 / v;
    aux[0] = a / v;
    aux[1] = ib;
    aux[2] = a / (v * v);
  } else if (i >= 4 + K && i < 4 + 2 * K) {
    aux[8 + (i - 4 - K)] = -1.0 / (v * v);
  } else if (i >= 4 + 2 * K + G) {
    aux[8 + K + (i - 4 - 2 * K - G)] = 1.0 / (v * v);
  }
}

// Observation pass for K > 62 (the fused kernels of obs_fused.cuh / fused.cuh cover K <= 62).  A CTA of 8
// warps walks 64-row tiles of X, double-buffered in shared memory (TMA bulk copies on an mbarrier per buffer, cp.async
// for odd K; tile t + 1 is in flight while tile t is computed; one buffer when two do not fit, K > 214).  Per tile every warp owns 8 rows:
//   A. z_mean / z_var dot products with lane = column (coalesced, conflict-free), then ONE transposing
//      butterfly (16 exchanges instead of 16 x 5) that leaves row rr's two sums in lanes 4 rr .. 4 rr + 3;
//   B. quadrature with lane = (row, node slot): the 4 lanes of a row split the Q nodes (branch-free exp /
//      log1p / reciprocal of obs_fused.cuh), two exchanges combine the six sums; lane 4 rr writes the row's
//      weights l_m, l_v, l_mm, l_mv, l_vv;
//   C. gradient partials X^T l_m, S^T l_v with lane = column again (weights broadcast by shuffle), kept in
//      registers across tiles; per-CTA fixed-order reduction at the end (no atomics).
// The first version (one thread per row, 64-thread CTAs, synchronous tile loads) ran at 1.5 TB/s with 4
// warps per SM; profiles/r02_launches_c4.md.
constexpr int kObsTile = 64;       // rows per tile
constexpr int kObsRows = 8;        // rows per warp and tile
constexpr int kObsMaxChunks = 8;   // 32-column chunks (K <= 256)

template <int ORDER>
__global__ void __launch_bounds__(256, 1)
k_obs(const double* __restrict__ X, const double* __restrict__ y, const int32_t* __restrict__ g,
      const double* __restrict__ w, const double* __restrict__ vec, const double* __restrict__ gh,
      double* __restrict__ W, double* __restrict__ klpart, double* __restrict__ gradpart,
      int64_t N, int64_t ldw, int K, int G, int Q, int nbuf) {
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t tile_elems = (size_t)kObsTile * K;
  double* xs = sm;                          // nbuf x 64 x K
  double* ghc = xs + nbuf * tile_elems;     // Q   sqrt(2) x_q
  double* ghw = ghc + 4 * ((Q + 3) >> 2);   //     w_q / sqrt(pi)
  double* red = ghw + 4 * ((Q + 3) >> 2);   // 32
  // nodes permuted so that the nodes ns, ns + 4, ... of node slot ns are contiguous: slot ns starts at ns * npl
  const int npl = (Q + 3) >> 2;              // nodes per slot (the last slots may have one fewer)
  for (int q = tid; q < Q; q += blockDim.x) {
    const int at = (q & 3) * npl + (q >> 2);
    ghc[at] = gh[q];
    ghw[at] = gh[Q + q];
  }
  const int nch = (K + 31) >> 5;
  double bmr[kObsMaxChunks], bvr[kObsMaxChunks];     // E[beta], Var[beta] of this lane's columns
  double gm[kObsMaxChunks], gv[kObsMaxChunks];
#pragma unroll
  for (int c = 0; c < kObsMaxChunks; ++c) {
    const int k = 32 * c + lane;
    bmr[c] = (c < nch && k < K) ? vec[4 + k] : 0.0;
    bvr[c] = (c < nch && k < K) ? 1.0 / vec[4 + K + k] : 0.0;
    gm[c] = gv[c] = 0.0;
  }
  const int64_t um0 = 4 + 2 * (int64_t)K, ui0 = um0 + G;
  double klacc = 0.0;
  const int rr = lane >> 2, ns = lane & 3;          // quadrature role: row of the warp, node slot

  const int64_t ntiles = (N + kObsTile - 1) / kObsTile;
  // A tile is contiguous in global and in shared memory: with K even thread 0 requests it as 8 bulk async
  // copies (TMA) on the buffer's mbarrier; odd K (rows not 16-byte multiples) takes the cp.async path.
  const bool tma = (K & 1) == 0;
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(red + 32);
  const unsigned bars_u = smem_u32(bars);
  if (tid == 0) {
    mbar_init(bars_u, 1);
    mbar_init(bars_u + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  auto load_tile = [&](int64_t tile, int buf) {
    const int64_t n0 = tile * kObsTile;
    const int rows = (int)((N - n0 < kObsTile) ? (N - n0) : kObsTile);
    if (tma) {
      if (tid == 0) {
        const unsigned bar = bars_u + 8 * buf;
        const unsigned total = (unsigned)(rows * K * sizeof(double));
        mbar_arrive_expect_tx(bar, total);
        const unsigned piece = (unsigned)(8 * K * sizeof(double));
        const unsigned dst = smem_u32(xs + buf * tile_elems);
        const char* src = reinterpret_cast<const char*>(X + n0 * K);
        for (unsigned off = 0; off < total; off += piece)
          bulk_g2s(dst + off, src + off, total - off < piece ? total - off : piece, bar);
      }
    } else {
      tile_load_async(xs + buf * tile_elems, X + n0 * K, (int64_t)rows * K);
    }
  };
  // per-row scalars of the quadrature phase, two tiles deep: the group index of tile t + 2 and, with the index
  // fetched one iteration earlier, the random effect / weight / response of tile t + 1 are requested while
  // tile t is computed (the second load depends on the first: in one step it would stall the warp)
  double nu_m = 0.0, nu_i = 1.0, nwn = 0.0, nyn = 0.0;
  int ngi = 0;
  const int64_t rowoff = warp * kObsRows + rr, tstride = (int64_t)gridDim.x * kObsTile;
  auto fetch_scalars = [&](int64_t n) {     // uses ngi = g[n] fetched earlier
    if (n < N) {
      nu_m = vec[um0 + ngi];
      nu_i = vec[ui0 + ngi];
      nwn = w ? w[n] : 1.0;
      nyn = y[n];
    }
  };
  auto fetch_group = [&](int64_t n) { if (n < N) ngi = g[n]; };
  int64_t tile = blockIdx.x;
  fetch_group(tile * kObsTile + rowoff);
  fetch_scalars(tile * kObsTile + rowoff);
  fetch_group(tile * kObsTile + rowoff + tstride);
  if (tile < ntiles) load_tile(tile, 0);
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  for (int it = 0; tile < ntiles; tile += gridDim.x, ++it) {
    const int buf = (nbuf == 2) ? (it & 1) : 0;
    const int64_t n0 = tile * kObsTile;
    const int rows = (int)((N - n0 < kObsTile) ? (N - n0) : kObsTile);
    // this lane's row of the quadrature phase: its group's random effect, response and weight were requested
    // one tile ahead (two dependent global round trips), the next tile's are requested now
    const int64_t nq = n0 + warp * kObsRows + rr;
    const bool rvalid = warp * kObsRows + rr < rows;
    const double u_m = nu_m, u_i = nu_i, wn = nwn, yn = nyn;
    fetch_scalars(n0 + rowoff + tstride);
    fetch_group(n0 + rowoff + 2 * tstride);
    if (nbuf == 2) {
      if (tile + gridDim.x < ntiles) load_tile(tile + gridDim.x, buf ^ 1);
      asm volatile("cp.async.commit_group;\ncp.async.wait_group 1;\n" ::: "memory");
    } else {
      if (it > 0) load_tile(tile, 0);      // the end-of-tile barrier of the previous iteration freed the buffer
      asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
    }
    if (tma) mbar_wait(bars_u + 8 * buf, (unsigned)(nbuf == 2 ? (it >> 1) : it) & 1u);
    __syncthreads();
    const double* xb = xs + buf * tile_elems + (size_t)(warp * kObsRows) * K;
    const int wrows = rows - warp * kObsRows;       // valid rows of this warp (may be <= 0)

    // A. partial dot products of 8 rows; v[2 r] = z_mean part, v[2 r + 1] = z_var part
    double v[2 * kObsRows];
#pragma unroll
    for (int r = 0; r < kObsRows; ++r) {
      double am = 0.0, av = 0.0;
      if (r < wrows) {
        const double* xr = xb + (size_t)r * K + lane;
#pragma unroll
        for (int c = 0; c < kObsMaxChunks; ++c)
          if (c < nch && 32 * c + lane < K) {
            const double x = xr[32 * c];
            am = fma(x, bmr[c], am);
            av = fma(x * x, bvr[c], av);
          }
      }
      v[2 * r] = am;
      v[2 * r + 1] = av;
    }
    // transposing butterfly: after the step with mask m a lane keeps the half of its values selected by
    // (lane & m); value index bits 3..0 follow lane bits 4..1, so lane L ends with value (L >> 1) & 15
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const bool hi = lane & 16;
      const double send = hi ? v[i] : v[i + 8], keep = hi ? v[i + 8] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const bool hi = lane & 8;
      const double send = hi ? v[i] : v[i + 4], keep = hi ? v[i + 4] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const bool hi = lane & 4;
      const double send = hi ? v[i] : v[i + 2], keep = hi ? v[i + 2] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    {
      const bool hi = lane & 2;
      const double send = hi ? v[0] : v[1], keep = hi ? v[1] : v[0];
      v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
    // lanes with ns < 2 hold row rr's z_mean sum, the others its z_var sum: swap across the pair
    const double other = __shfl_xor_sync(0xffffffffu, v[0], 2);
    double zm = (ns < 2) ? v[0] : other, zv = (ns < 2) ? other : v[0];

    // B. quadrature: lane (rr, ns) takes nodes ns, ns + 4, ...
    double lm = 0.0, lv = 0.0;
    {
      const int64_t n = nq;
      GHSumsF s = {0, 0, 0, 0, 0, 0};
      double zs = 1.0;
      if (rvalid) {
        zm += u_m;
        zv += 1.0 / u_i;
        zs = sqrt(zv);
        // this slot's nodes, two at a time with their chains interleaved step by step (obs_fused.cuh)
        gh_all_nodes_f<ORDER, 2>(zm, zs, ghc + ns * npl, ghw + ns * npl, (Q - ns + 3) >> 2, s);
      }
#pragma unroll
      for (int m = 1; m <= 2; m <<= 1) {
        s.A += __shfl_xor_sync(0xffffffffu, s.A, m);
        if (ORDER >= 1) {
          s.Am += __shfl_xor_sync(0xffffffffu, s.Am, m);
          s.As += __shfl_xor_sync(0xffffffffu, s.As, m);
        }
        if (ORDER >= 2) {
          s.Amm += __shfl_xor_sync(0xffffffffu, s.Amm, m);
          s.Ams += __shfl_xor_sync(0xffffffffu, s.Ams, m);
          s.Ass += __shfl_xor_sync(0xffffffffu, s.Ass, m);
        }
      }
      if (rvalid) {
        if (ns == 0) klacc += wn * (yn * zm - s.A);
        if (ORDER >= 1) {
          const double h = 0.5 / zs;
          lm = wn * (yn - s.Am);
          lv = -wn * s.As * h;
          if (ns == 0) {
            W[n] = lm;
            W[ldw + n] = lv;
            if (ORDER >= 2) {
              W[2 * ldw + n] = -wn * s.Amm;
              W[3 * ldw + n] = -wn * s.Ams * h;
              // l_vv = -(A_ss / (4 z_v) - A_s / (4 z_s^3))
              W[4 * ldw + n] = -wn * (s.Ass - s.As / zs) / (4.0 * zv);
            }
          }
        }
      }
    }
    // C. gradient partials, lane = column
    if (ORDER >= 1) {
#pragma unroll
      for (int r = 0; r < kObsRows; ++r) {
        const double lmr = __shfl_sync(0xffffffffu, lm, 4 * r), lvr = __shfl_sync(0xffffffffu, lv, 4 * r);
        if (r < wrows) {
          const double* xr = xb + (size_t)r * K + lane;
#pragma unroll
          for (int c = 0; c < kObsMaxChunks; ++c)
            if (c < nch && 32 * c + lane < K) {
              const double x = xr[32 * c];
              gm[c] = fma(x, lmr, gm[c]);
              gv[c] = fma(x * x, lvr, gv[c]);
            }
        }
      }
    }
    __syncthreads();   // the buffer is refilled by the next iteration's load
  }
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");

  const double kl = block_sum(klacc, red);
  if (tid == 0) klpart[blockIdx.x] = kl;
  if (ORDER >= 1) {
    // per-warp partials -> shared memory -> fixed-order sum over the 8 warps; layout (2K, n_cta)
    __syncthreads();
    double* buf = xs;      // 8 x 2K <= 64 x K
#pragma unroll
    for (int c = 0; c < kObsMaxChunks; ++c) {
      const int k = 32 * c + lane;
      if (c < nch && k < K) {
        buf[(size_t)warp * 2 * K + k] = gm[c];
        buf[(size_t)warp * 2 * K + K + k] = gv[c];
      }
    }
    __syncthreads();
    const size_t gs = gridDim.x;
    for (int k = tid; k < 2 * K; k += blockDim.x) {
      double s = 0.0;
#pragma unroll
      for (int p = 0; p < 8; ++p) s += buf[(size_t)p * 2 * K + k];
      gradpart[(size_t)k * gs + blockIdx.x] = s;
    }
  }
}

// Influence of every observation for wide models (K > 62): out[n] = (C^T v)_n = -(l_m dm_n + l_v dv_n) with unit
// weight (sensitivity.cu: lrvb_glmm_weight_cross_rmatvec), dm_n = x_n . v_bm + v_um[g_n], dv_n = x_n^2 . (v_bi
// dvar/dfree) + v_ui[g_n] dvar_u/dfree.  The tile walk of k_obs with FOUR dot products per row: the transposing
// butterfly takes 8 rows x 4 sums = 32 values to one per lane (31 exchanges), lane 4 rr + i ends with sum i of
// row rr, and the four lanes of a row share them by three shuffles; then the order-1 quadrature of k_obs.
__global__ void __launch_bounds__(256, 1)
k_obs_influence_wide(const double* __restrict__ X, const double* __restrict__ y, const int32_t* __restrict__ g,
                     const double* __restrict__ vec, const double* __restrict__ gh, const double* __restrict__ v,
                     double* __restrict__ out, int64_t N, int K, int G, int Q, int nbuf,
                     lrvb_glmm_bounds bd, int vecmode) {
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t tile_elems = (size_t)kObsTile * K;
  double* xs = sm;
  double* ghc = xs + nbuf * tile_elems;
  double* ghw = ghc + 4 * ((Q + 3) >> 2);
  const int npl = (Q + 3) >> 2;
  for (int q = tid; q < Q; q += blockDim.x) {
    const int at = (q & 3) * npl + (q >> 2);
    ghc[at] = gh[q];
    ghw[at] = gh[Q + q];
  }
  const int nch = (K + 31) >> 5;
  double bmr[kObsMaxChunks], bvr[kObsMaxChunks], vmr[kObsMaxChunks], vvr[kObsMaxChunks];
#pragma unroll
  for (int c = 0; c < kObsMaxChunks; ++c) {
    const int k = 32 * c + lane;
    const bool in = c < nch && k < K;
    const double ik = in ? vec[4 + K + k] : 1.0;
    bmr[c] = in ? vec[4 + k] : 0.0;
    bvr[c] = in ? 1.0 / ik : 0.0;
    vmr[c] = in ? v[4 + k] : 0.0;
    vvr[c] = in ? v[4 + K + k] * (-1.0 / (ik * ik)) * (vecmode ? 1.0 : ik - bd.beta_info) : 0.0;
  }
  const int64_t um0 = 4 + 2 * (int64_t)K, ui0 = um0 + G;
  const int rr = lane >> 2, ns = lane & 3;
  const int64_t ntiles = (N + kObsTile - 1) / kObsTile;
  auto load_tile = [&](int64_t tile, int buf) {
    const int64_t n0 = tile * kObsTile;
    const int rows = (int)((N - n0 < kObsTile) ? (N - n0) : kObsTile);
    tile_load_async(xs + buf * tile_elems, X + n0 * K, (int64_t)rows * K);
  };
  int64_t tile = blockIdx.x;
  if (tile < ntiles) load_tile(tile, 0);
  asm volatile("cp.async.commit_group;\n" ::: "memory");
  __syncthreads();
  for (int it = 0; tile < ntiles; tile += gridDim.x, ++it) {
    const int buf = (nbuf == 2) ? (it & 1) : 0;
    const int64_t n0 = tile * kObsTile;
    const int rows = (int)((N - n0 < kObsTile) ? (N - n0) : kObsTile);
    if (nbuf == 2) {
      if (tile + gridDim.x < ntiles) load_tile(tile + gridDim.x, buf ^ 1);
      asm volatile("cp.async.commit_group;\ncp.async.wait_group 1;\n" ::: "memory");
    } else {
      if (it > 0) load_tile(tile, 0);
      asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
    }
    __syncthreads();
    const double* xb = xs + buf * tile_elems + (size_t)(warp * kObsRows) * K;
    const int wrows = rows - warp * kObsRows;
    double t[4 * kObsRows];
#pragma unroll
    for (int r = 0; r < kObsRows; ++r) {
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      if (r < wrows) {
        const double* xr = xb + (size_t)r * K + lane;
#pragma unroll
        for (int c = 0; c < kObsMaxChunks; ++c)
          if (c < nch && 32 * c + lane < K) {
            const double x = xr[32 * c], xx = x * x;
            a0 = fma(x, bmr[c], a0);
            a1 = fma(xx, bvr[c], a1);
            a2 = fma(x, vmr[c], a2);
            a3 = fma(xx, vvr[c], a3);
          }
      }
      t[4 * r] = a0; t[4 * r + 1] = a1; t[4 * r + 2] = a2; t[4 * r + 3] = a3;
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
      const bool hi = lane & m;
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (i < m) {
          const double send = hi ? t[i] : t[i + m], keep = hi ? t[i + m] : t[i];
          t[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
        }
    }
    // lane 4 rr + i holds sum i of row rr
    const int base = lane & ~3;
    double zm = __shfl_sync(0xffffffffu, t[0], base), zv = __shfl_sync(0xffffffffu, t[0], base + 1);
    double dm = __shfl_sync(0xffffffffu, t[0], base + 2), dv = __shfl_sync(0xffffffffu, t[0], base + 3);
    const int64_t n = n0 + warp * kObsRows + rr;
    const bool rvalid = rr < wrows;
    GHSumsF s = {0, 0, 0, 0, 0, 0};
    double zs = 1.0, yn = 0.0;
    if (rvalid) {
      const int gi = g[n];
      const double uinfo = vec[ui0 + gi];
      zm += vec[um0 + gi];
      zv += 1.0 / uinfo;
      dm += v[um0 + gi];
      dv += v[ui0 + gi] * (-1.0 / (uinfo * uinfo)) * (vecmode ? 1.0 : uinfo - bd.u_info);
      zs = sqrt(zv);
      yn = y[n];
      gh_all_nodes_f<1, 2>(zm, zs, ghc + ns * npl, ghw + ns * npl, (Q - ns + 3) >> 2, s);
    }
#pragma unroll
    for (int m = 1; m <= 2; m <<= 1) {
      s.Am += __shfl_xor_sync(0xffffffffu, s.Am, m);
      s.As += __shfl_xor_sync(0xffffffffu, s.As, m);
    }
    if (rvalid && ns == 0) {
      const double lm = yn - s.Am, lv = -s.As * (0.5 / zs);
      out[n] = -(lm * dm + lv * dv);
    }
    __syncthreads();
  }
  asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

// ------------------------------------------------------------------------------------------
// Per-group segmented sums.  One warp per group (grid-stride); observations of a group are
// the contiguous range [gptr[g], gptr[g+1]) so no atomics are needed and the summation order
// is fixed.  gsc (G,5): sums of l_m, l_v, a, b, c.  BR (G,4,K): sum a x, sum b x, sum b s, sum c s.
// (Rows outer / the lane's column chunks inner -- every row read once, 32 accumulators per lane -- was measured
// at K = 200: 0.70 ms against 0.24 ms per 500k rows; the chunk-outer walk below keeps 33 warps per SM in flight
// and its re-reads are L2 hits.)
template <int ORDER>
__global__ void __launch_bounds__(256)
k_group(const double* __restrict__ X, const double* __restrict__ W,
        const int32_t* __restrict__ gptr, double* __restrict__ gsc, double* __restrict__ BR,
        int64_t ldw, int K, int G) {
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const int nrow = (ORDER >= 2) ? 5 : 2;
  for (int gi = blockIdx.x * wpb + (threadIdx.x >> 5); gi < G; gi += gridDim.x * wpb) {
    const int64_t nb = gptr[gi], ne = gptr[gi + 1];
    double s[5] = {0, 0, 0, 0, 0};
    for (int64_t n = nb + lane; n < ne; n += 32) {
#pragma unroll
      for (int r = 0; r < 5; ++r)
        if (r < nrow) s[r] += W[r * ldw + n];
    }
#pragma unroll
    for (int r = 0; r < 5; ++r)
      if (r < nrow) s[r] = warp_sum(s[r]);
    if (lane == 0) {
#pragma unroll
      for (int r = 0; r < 5; ++r) gsc[(size_t)gi * 5 + r] = (r < nrow) ? s[r] : 0.0;
    }
    if (ORDER >= 2) {
      const double* Wa = W + 2 * ldw;
      const double* Wb = W + 3 * ldw;
      const double* Wc = W + 4 * ldw;
      for (int k = lane; k < K; k += 32) {
        double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
        int64_t n = nb;
        for (; n + 4 <= ne; n += 4) {
          double x[4], a[4], b[4], c[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            x[u] = X[(n + u) * K + k];
            a[u] = Wa[n + u];
            b[u] = Wb[n + u];
            c[u] = Wc[n + u];
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const double xx = x[u] * x[u];
            s0 = fma(a[u], x[u], s0);
            s1 = fma(b[u], x[u], s1);
            s2 = fma(b[u], xx, s2);
            s3 = fma(c[u], xx, s3);
          }
        }
        for (; n < ne; ++n) {
          const double x = X[n * K + k], xx = x * x;
          s0 = fma(Wa[n], x, s0);
          s1 = fma(Wb[n], x, s1);
          s2 = fma(Wb[n], xx, s2);
          s3 = fma(Wc[n], xx, s3);
        }
        double* br = BR + (size_t)gi * 4 * K;
        br[k] = s0;
        br[K + k] = s1;
        br[2 * K + k] = s2;
        br[3 * K + k] = s3;
      }
    }
  }
}

// The data terms of the gradient with dw as the weights, for lrvb_glmm_weight_cross_matvec (sensitivity.cu):
// the per-CTA partials of X^T l_m, S^T l_v go to gradpart (*n_gp of them), the per-group sums to gsc and BR.  The
// cached evaluation's W (lrvb_glmm_obs_weights) stays intact.  K <= 62: the two-slot fused observation pass,
// which writes no W, then k_obs_fixup<1>; K > 62: k_obs<1>, writing l_m, l_v into a scratch block, then k_group<1>.
int launch_weight_pass(lrvb_glmm* h, const double* dw, int* n_gp, cudaStream_t st) {
  const int K = h->K, G = h->G, Q = h->Q;
  const int64_t N = h->N;
  *n_gp = 0;
  if (h->obs_fused) {
    if (N > 0) {
      auto kern = (K + 1 + 31) / 32 == 1 ? k_obs_fused<1, 1> : k_obs_fused<1, 2>;
      LRVB_TRY(raise_smem_limit(kern, h->of_smem));
      kern<<<h->of_grid, 32 * h->of_warps, h->of_smem, st>>>(h->X, h->y, h->g, dw, h->vec, h->gh, h->gptr, nullptr,
                                                             h->ldw, h->klpart, h->gradpart, h->gsc, h->BR, h->bval,
                                                             N, K, G, Q, h->of_rows_per_warp);
      LRVB_CHECK_LAUNCH();
      *n_gp = h->of_grid;
    }
    if (G > 0) {
      k_obs_fixup<1><<<cdiv(G, 8), 256, 0, st>>>(h->gptr, h->bval, h->gsc, h->BR, K, G,
                                                 h->of_rows_per_warp > 0 ? h->of_rows_per_warp : 32);
      LRVB_CHECK_LAUNCH();
    }
    return LRVB_OK;
  }
  if (N > 0) {
    if (!h->wc_scratch && cudaMalloc(&h->wc_scratch, sizeof(double) * 2 * (size_t)h->ldw) != cudaSuccess) {
      cudaGetLastError();
      set_error("lrvb_glmm_weight_cross_matvec: out of device memory (%zu bytes of scratch)",
                sizeof(double) * 2 * (size_t)h->ldw);
      return LRVB_ECUDA;
    }
    k_obs<1><<<h->obs_grid, 256, h->obs_smem, st>>>(h->X, h->y, h->g, dw, h->vec, h->gh, h->wc_scratch, h->klpart,
                                                    h->gradpart, N, h->ldw, K, G, Q, h->obs_nbuf);
    LRVB_CHECK_LAUNCH();
    *n_gp = h->obs_grid;
  }
  if (G > 0) {
    const int ggrid = (int)((G + 7) / 8 < 148 * 8 ? (G + 7) / 8 : 148 * 8);
    k_group<1><<<ggrid, 256, 0, st>>>(h->X, h->wc_scratch, h->gptr, h->gsc, h->BR, h->ldw, K, G);
    LRVB_CHECK_LAUNCH();
  }
  return LRVB_OK;
}
// The influence pass for K > 62 (lrvb_glmm_weight_cross_rmatvec) on the k_obs tile walk
int launch_wide_influence(lrvb_glmm* h, const double* v, double* out, cudaStream_t st) {
  LRVB_TRY(raise_smem_limit(k_obs_influence_wide, h->obs_smem));
  k_obs_influence_wide<<<h->obs_grid, 256, h->obs_smem, st>>>(h->X, h->y, h->g, h->vec, h->gh, v, out, h->N, h->K,
                                                             h->G, h->Q, h->obs_nbuf, h->bounds, h->vecmode);
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

// Finish of the packed Gram (layout of gram_small.cuh, written by the one-pass, mid and wide kernels):
// fixed-order sum of the per-CTA partials of one packed tile, then the same chain rule as k_gram_finish.
// Packed column p < K is x_p, p >= K is s_{p-K}; only the upper triangle of the packed matrix was computed.
__device__ __forceinline__ void gram_small_finish_body(int bid, const double* __restrict__ part, const double* __restrict__ vec,
                    double* __restrict__ A, int K, int Dg, int NT, int n_cta, lrvb_glmm_bounds bd,
                    int vecmode) {
  __shared__ double red[4][64];
  const int t = bid;
  int jt = 0;
  while ((jt + 1) * (jt + 2) / 2 <= t) ++jt;
  const int it = t - jt * (jt + 1) / 2;
  const int e = threadIdx.x & 63, ps = threadIdx.x >> 6;
  const double* src = part + (size_t)t * 64 + e;
  const size_t stride = (size_t)NT * 64;
  double s = 0.0;
#pragma unroll 8
  for (int c = ps; c < n_cta; c += 4) s += src[(size_t)c * stride];
  red[ps][e] = s;
  __syncthreads();
  if (ps != 0) return;
  s = (red[0][e] + red[1][e]) + (red[2][e] + red[3][e]);
  const int p = 8 * it + (e >> 3), q = 8 * jt + (e & 7);
  if (p > q || q >= 2 * K) return;
  const int bm0 = 4, bi0 = 4 + K;
  if (q < K) {                       // (x, x): beta.mean is unconstrained, j = 1
    const double v = -s;
    A[(size_t)(bm0 + p) * Dg + bm0 + q] = v;
    A[(size_t)(bm0 + q) * Dg + bm0 + p] = v;
  } else if (p < K) {                // (x, s)
    const int k2 = q - K;
    const double iq = vec[bi0 + k2];
    const double v = -s * (-1.0 / (iq * iq)) * (vecmode ? 1.0 : iq - bd.beta_info);
    A[(size_t)(bm0 + p) * Dg + bi0 + k2] = v;
    A[(size_t)(bi0 + k2) * Dg + bm0 + p] = v;
  } else {                           // (s, s)
    const int k1 = p - K, k2 = q - K;
    const double ip = vec[bi0 + k1], iq = vec[bi0 + k2];
    const double v = -s * (1.0 / (ip * ip * iq * iq)) *
                     (vecmode ? 1.0 : (ip - bd.beta_info) * (iq - bd.beta_info));
    A[(size_t)(bi0 + k1) * Dg + bi0 + k2] = v;
    A[(size_t)(bi0 + k2) * Dg + bi0 + k1] = v;
  }
}

// ------------------------------------------------------------------------------------------
// Per-group sums as the finishing pass sees them.  The fused observation kernels write a group's sums
// (gsc: 5 scalars, BR: 4 x K) directly when the group lies inside one warp's row range; a group that
// straddles ranges has its pieces in bval (head / tail records per warp, layout [5 | 4K]) and they are
// added here in row order -- the separate k_obs_fixup launch of round 1 folded into the consumer.
// rpw = rows per warp of the producing kernel (0: gsc / BR are complete, e.g. the K > 62 path).
struct GroupFix {
  const int32_t* gptr;
  const double* bval;
  unsigned rpw;    // rows per warp (N < 2^31)
  int nb;          // 5 + 4K
  double inv_rpw;  // 1 / rpw: the quotient comes from one multiplication and an exact correction step
};
__device__ __forceinline__ unsigned div_rpw(unsigned n, const GroupFix& fx) {
  unsigned q = __double2uint_rz((double)n * fx.inv_rpw);      // floor(n / rpw) or one off
  if ((unsigned long long)(q + 1) * fx.rpw <= n) ++q;
  else if ((unsigned long long)q * fx.rpw > n) --q;
  return q;
}
struct GroupSpan {
  unsigned wf, wl;     // first / last producing warp; wf > wl: empty group; wf == wl: the sums were written directly
};
__device__ __forceinline__ GroupSpan group_span(const GroupFix& fx, int gi) {
  GroupSpan sp;
  sp.wf = sp.wl = 0;
  if (fx.rpw == 0) return sp;
  const unsigned gb = (unsigned)fx.gptr[gi], ge = (unsigned)fx.gptr[gi + 1];
  if (gb == ge) { sp.wf = 1; sp.wl = 0; return sp; }        // empty group: nobody wrote its sums
  sp.wf = div_rpw(gb, fx);
  sp.wl = div_rpw(ge - 1, fx);
  return sp;
}
__device__ __forceinline__ double group_val(const GroupFix& fx, const GroupSpan& sp, const double* __restrict__ direct,
                                            size_t di, int e) {
  if (sp.wf == sp.wl) return direct[di];
  if (sp.wf > sp.wl) return 0.0;
  double s = fx.bval[((size_t)sp.wf * 2 + 1) * fx.nb + e];     // tail of the first warp
  for (unsigned wi = sp.wf + 1; wi <= sp.wl; ++wi) s += fx.bval[((size_t)wi * 2) * fx.nb + e];   // heads, row order
  return s;
}

// ------------------------------------------------------------------------------------------
// Group-level chain rule: local gradient, local 2x2 blocks, and partial sums of the
// random-effect term  sum_g [-1/2 E[tau]((E mu - E u_g)^2 + Var mu + Var u_g) + 1/2 E log tau]
// (SURVEY.md A.1; GammaParams.py:9-13, NormalParams.py:58-63).
template <int ORDER>
__device__ __forceinline__ void local_body(int bid, int nblk, const double* __restrict__ vec, const double* __restrict__ gsc,
        double* __restrict__ gradl, double* __restrict__ L, double* __restrict__ locpart,
        int K, int G, lrvb_glmm_bounds bd, int vecmode, const GroupFix& fx) {
  __shared__ double red[32];
  const int Dg = 4 + 2 * K;
  const double mu_m = vec[0], mu_i = vec[1], a = vec[2], b = vec[3];
  const double E = a / b;
  double dsum = 0.0, ssum = 0.0, lsum = 0.0;
  for (int gi = bid * blockDim.x + threadIdx.x; gi < G; gi += nblk * blockDim.x) {
    const double um = vec[Dg + gi], ui = vec[Dg + G + gi];
    const double dm = mu_m - um;
    const double r = 1.0 / ui;
    dsum += dm;
    ssum += dm * dm + 1.0 / mu_i + r;
    lsum += log(ui);
    if (ORDER >= 1) {
      double s[5];
      const GroupSpan sp = group_span(fx, gi);
      // the five sums of a group: written directly, or the pieces of a straddling group added in row order
      // (all five of a record are loaded before they are added: independent loads, one chain of additions)
      if (sp.wf == sp.wl) {
#pragma unroll
        for (int e = 0; e < 5; ++e) s[e] = (ORDER >= 2 || e < 2) ? gsc[(size_t)gi * 5 + e] : 0.0;
      } else if (sp.wf > sp.wl) {
#pragma unroll
        for (int e = 0; e < 5; ++e) s[e] = 0.0;
      } else {
        const double* t = fx.bval + ((size_t)sp.wf * 2 + 1) * fx.nb;
#pragma unroll
        for (int e = 0; e < 5; ++e) s[e] = (ORDER >= 2 || e < 2) ? t[e] : 0.0;
        for (unsigned wi = sp.wf + 1; wi <= sp.wl; ++wi) {
          const double* hd = fx.bval + ((size_t)wi * 2) * fx.nb;
          double q[5];
#pragma unroll
          for (int e = 0; e < 5; ++e) q[e] = (ORDER >= 2 || e < 2) ? hd[e] : 0.0;
#pragma unroll
          for (int e = 0; e < 5; ++e) s[e] += q[e];
        }
      }
      const double r2 = r * r;
      const double gF_um = s[0] + E * dm;
      const double gF_ui = -s[1] * r2 + 0.5 * E * r2 - 0.5 * r;
      // d info / d free = d2 info / d free2 = info - lb (Parameters.py:55); identity in vector mode
      const double ji = vecmode ? 1.0 : ui - bd.u_info;
      const double ji2 = vecmode ? 0.0 : ji;
      const double gv_ui = -gF_ui;
      gradl[gi] = -gF_um;
      gradl[G + gi] = gv_ui * ji;
      if (ORDER >= 2) {
        const double dr = -r2;
        const double L0 = s[2] - E;
        const double L1 = s[3] * dr;
        const double L2 = s[4] * dr * dr + s[1] * 2.0 * r2 * r - E * r2 * r + 0.5 * r2;
        L[(size_t)gi * 3 + 0] = -L0;
        L[(size_t)gi * 3 + 1] = -L1 * ji;
        L[(size_t)gi * 3 + 2] = -L2 * ji * ji + gv_ui * ji2;
      }
    }
  }
  dsum = block_sum(dsum, red);
  ssum = block_sum(ssum, red);
  lsum = block_sum(lsum, red);
  if (threadIdx.x == 0) {
    locpart[bid * 4 + 0] = dsum;
    locpart[bid * 4 + 1] = ssum;
    locpart[bid * 4 + 2] = lsum;
    locpart[bid * 4 + 3] = 0.0;
  }
}

// Border rows B (G,2,Dg) in free coordinates: row 0 = (u.mean_g, globals), row 1 = (u.info_g, .).
// A block covers 8 x gpw consecutive groups: their per-group scalars and producer spans are fetched
// cooperatively once (one round trip for the block), then every warp streams its gpw groups with lanes over
// the K fixed effects: a lane reads its four sums (a x, b x, b s, c s) of all its groups before it writes
// anything (the pass is a pure stream and needs the memory-level parallelism).  No fp64 division here:
// -1/beta.info^2, 1/u.info^2 and the tau ratios come from k_prep (one division per parameter instead of one
// per (group, column)).  A group whose sums were written by one producer warp is read from BR; one that
// straddles two producer ranges (every sixth group at C2, where a warp's range holds six groups) is the sum
// of two records of bval, read as two more coalesced streams; more pieces (rare: a group longer than a
// warp's range) go through group_val.
constexpr int kBorderBigG = 32768;
__host__ __device__ inline int border_groups_per_warp(int G) { return G >= kBorderBigG ? 2 : 1; }

struct BorderSrc {
  const double* pa;     // first (or only) source record, element (e, k) at pa[e * K + k]
  const double* pb;     // second record or nullptr
};
template <int NG>
__device__ __forceinline__ void border_stream(const double* __restrict__ vec, double* __restrict__ B,
         const double* __restrict__ adv, int K, int Dg, int g0, int lane, const BorderSrc (&src)[2],
         const double (&r2)[2], const double (&ji)[2], bool two, lrvb_glmm_bounds bd, int vecmode) {
  double* __restrict__ o0 = B + (size_t)g0 * 2 * Dg + 4 + lane;        // (group, 2, Dg)
  const double* __restrict__ pj = vec + 4 + K + lane;
  const double* __restrict__ pd = adv + lane;
  const int K2 = 2 * K, K3 = 3 * K, D2 = 2 * Dg;
#pragma unroll 2
  for (int k = lane; k < K; k += 32, o0 += 32, pj += 32, pd += 32) {
    double v[NG][4];
#pragma unroll
    for (int r = 0; r < NG; ++r) {
      const double* p = src[r].pa + k;
      v[r][0] = p[0]; v[r][1] = p[K]; v[r][2] = p[K2]; v[r][3] = p[K3];
    }
    if (two) {
#pragma unroll
      for (int r = 0; r < NG; ++r) {
        if (src[r].pb) {
          const double* p = src[r].pb + k;
          v[r][0] += p[0]; v[r][1] += p[K]; v[r][2] += p[K2]; v[r][3] += p[K3];
        }
      }
    }
    const double dv = *pd;
    const double jg = vecmode ? 1.0 : *pj - bd.beta_info;
#pragma unroll
    for (int r = 0; r < NG; ++r) {
      const double dr = -r2[r];
      double* o = o0 + r * D2;
      o[0] = -v[r][0];
      o[Dg] = -(v[r][1] * dr) * ji[r];
      o[K] = -(v[r][2] * dv) * jg;
      o[Dg + K] = -(v[r][3] * dv * dr) * jg * ji[r];
    }
  }
}

__device__ __forceinline__ void border_body(int bid, const double* __restrict__ vec, const double* __restrict__ BR, double* __restrict__ B,
         int K, int G, lrvb_glmm_bounds bd, int vecmode, const GroupFix& fx) {
  __shared__ double s_um[16], s_ji[16], s_r2[16];
  __shared__ unsigned s_wf[16], s_wl[16];
  const int Dg = 4 + 2 * K;
  const int lane = threadIdx.x & 31;
  const int gpw = border_groups_per_warp(G);
  const int gb = bid * 8 * gpw;                    // first group of the block
  const double* __restrict__ aux = vec + Dg + 2 * (size_t)G;
  const double* __restrict__ adv = aux + 8;
  if ((int)threadIdx.x < 8 * gpw && gb + (int)threadIdx.x < G) {
    const int gi = gb + threadIdx.x;
    s_um[threadIdx.x] = vec[Dg + gi];
    s_ji[threadIdx.x] = vecmode ? 1.0 : vec[Dg + G + gi] - bd.u_info;
    s_r2[threadIdx.x] = aux[8 + K + gi];
    const GroupSpan sp = group_span(fx, gi);
    s_wf[threadIdx.x] = sp.wf;
    s_wl[threadIdx.x] = sp.wl;
  }
  __syncthreads();
  const int l0 = (threadIdx.x >> 5) * gpw;         // first group of the warp, block-local
  const int g0 = gb + l0;
  if (g0 >= G) return;
  const int ng = (gpw == 2 && g0 + 1 < G) ? 2 : 1;
  double um[2], r2[2], ji[2];
  GroupSpan sp[2];
  BorderSrc src[2];
  bool two = false, many = false;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int l = (r < ng) ? l0 + r : l0;
    um[r] = s_um[l]; ji[r] = s_ji[l]; r2[r] = s_r2[l];
    sp[r].wf = s_wf[l]; sp[r].wl = s_wl[l];
    src[r].pb = nullptr;
    if (sp[r].wf == sp[r].wl) {
      src[r].pa = BR + (size_t)(gb + l) * 4 * K;
    } else if (sp[r].wf + 1 == sp[r].wl) {
      src[r].pa = fx.bval + ((size_t)sp[r].wf * 2 + 1) * fx.nb + 5;     // tail record of the first warp
      src[r].pb = fx.bval + ((size_t)sp[r].wl * 2) * fx.nb + 5;         // head record of the second
      two = true;
    } else {
      src[r].pa = BR;          // empty group (wf > wl: zeros) or more than two pieces: generic path below
      many = true;
    }
  }
  if (lane < 4) {
    const double mu_m = vec[0], a = vec[2], b = vec[3];
    const double E = aux[0], ib = aux[1], aib2 = aux[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (r >= ng) break;
      double b0, b1, jg = 1.0;
      if (lane == 0) { b0 = E; b1 = 0.0; }
      else if (lane == 1) { b0 = 0.0; b1 = 0.0; jg = vec[1] - bd.mu_info; }
      else if (lane == 2) { b0 = (mu_m - um[r]) * ib; b1 = 0.5 * r2[r] * ib; jg = a - bd.tau_shape; }
      else { b0 = -(mu_m - um[r]) * aib2; b1 = -0.5 * r2[r] * aib2; jg = b - bd.tau_rate; }
      if (vecmode) jg = 1.0;
      double* out = B + (size_t)(g0 + r) * 2 * Dg;
      out[lane] = -b0 * jg;
      out[Dg + lane] = -b1 * jg * ji[r];
    }
  }
  if (!many) {
    if (ng == 2) border_stream<2>(vec, B, adv, K, Dg, g0, lane, src, r2, ji, two, bd, vecmode);
    else border_stream<1>(vec, B, adv, K, Dg, g0, lane, src, r2, ji, two, bd, vecmode);
    return;
  }
  for (int r = 0; r < ng; ++r) {
    const size_t br = (size_t)(g0 + r) * 4 * K;
    const double dr = -r2[r];
    double* out = B + (size_t)(g0 + r) * 2 * Dg;
    for (int k = lane; k < K; k += 32) {
      const double v0 = group_val(fx, sp[r], BR, br + k, 5 + k);
      const double v1 = group_val(fx, sp[r], BR, br + K + k, 5 + K + k);
      const double v2 = group_val(fx, sp[r], BR, br + 2 * (size_t)K + k, 5 + 2 * K + k);
      const double v3 = group_val(fx, sp[r], BR, br + 3 * (size_t)K + k, 5 + 3 * K + k);
      const double dv = adv[k];
      const double jg = vecmode ? 1.0 : vec[4 + K + k] - bd.beta_info;
      out[4 + k] = -v0;
      out[Dg + 4 + k] = -(v1 * dr) * ji[r];
      out[4 + K + k] = -(v2 * dv) * jg;
      out[Dg + 4 + K + k] = -(v3 * dv * dr) * jg * ji[r];
    }
  }
}

// ------------------------------------------------------------------------------------------
// Single-CTA finish: fixed-order sums of the per-CTA partials, the non-data terms
// (ExponentialFamilies.py:23-25 uvn entropy, :33-35 gamma entropy, :111-112 E log tau,
// :191-195 priors), the global gradient and the 4x4 corner / diagonal extras of A,
// then the vector->free chain rule (Parameters.py:397-424 for diagonal transforms).
// out = [KL, grad_g (Dg), A (Dg*Dg)].
struct GlobalArgs {
  const double* klpart; int n_kl; const double* gradpart; int n_gp; int n_lp; double* out;
  lrvb_glmm_prior pr; int include_global; unsigned int* counter;
  double* pre;      // scratch [data_ll, psi, psi1, psi2, lgamma | gsum (2K)] from block 0 for the last block
};
// Block 0 of k_finish: what needs only the kernels BEFORE k_finish -- the special functions of tau.shape
// (long serial chains: one lane of four different warps each) and the fixed-order sums of the observation
// pass's partials -- computed while the other blocks do the group-level work.
template <int ORDER>
__device__ __forceinline__ void global_pre(const double* __restrict__ vec, const GlobalArgs& ga, int K) {
  __shared__ double red[32];
  const int tid = threadIdx.x;
  double* pre = ga.pre;
  if (tid == 32) pre[1] = digamma_pos(vec[2]);
  else if (tid == 64) pre[2] = trigamma_pos(vec[2]);
  else if (tid == 96) pre[3] = tetragamma_pos(vec[2]);
  else if (tid == 128) pre[4] = lgamma(vec[2]);
  double v = 0.0;
  for (int i = tid; i < ga.n_kl; i += blockDim.x) v += ga.klpart[i];
  const double data_ll = block_sum(v, red);
  if (tid == 0) pre[0] = data_ll;
  if (ORDER >= 1) {
    // one warp per column, lanes over the per-CTA partials (fixed order: deterministic)
    for (int k = tid >> 5; k < 2 * K; k += blockDim.x >> 5) {
      double s = 0.0;
      for (int p = tid & 31; p < ga.n_gp; p += 32) s += ga.gradpart[(size_t)k * ga.n_gp + p];
      s = warp_sum(s);
      if ((tid & 31) == 0) pre[8 + k] = s;
    }
  }
}
// k_global_post (one CTA, after k_finish): fixed-order sums of
// the group-level partials, the non-data terms (ExponentialFamilies.py:23-25 uvn entropy, :33-35 gamma
// entropy, :111-112 E log tau, :191-195 priors), the global gradient, the 4x4 corner / diagonal extras of
// A and the vector->free chain rule (Parameters.py:397-424).
template <int ORDER>
__device__ __forceinline__ void global_post(const double* __restrict__ vec, const GlobalArgs& ga, const double* locpart,
                                            int K, int G, lrvb_glmm_bounds bd, int vecmode) {
  const int n_lp = ga.n_lp, include_global = ga.include_global;
  double* out = ga.out;
  const lrvb_glmm_prior pr = ga.pr;
  __shared__ double red[32];
  __shared__ double sh[8];
  __shared__ double spec[4];
  extern __shared__ double gsum[];  // 2K
  const int tid = threadIdx.x;
  const int Dg = 4 + 2 * K;
  if (tid < 4) spec[tid] = __ldcg(ga.pre + 1 + tid);
  if (ORDER >= 1)
    for (int k = tid; k < 2 * K; k += blockDim.x) gsum[k] = __ldcg(ga.pre + 8 + k);
  const double data_ll = __ldcg(ga.pre);
  double d0 = 0, d1 = 0, d2 = 0;
  for (int i = tid; i < n_lp; i += blockDim.x) {      // written by other CTAs of this grid: L2 loads
    d0 += __ldcg(locpart + i * 4 + 0);
    d1 += __ldcg(locpart + i * 4 + 1);
    d2 += __ldcg(locpart + i * 4 + 2);
  }
  d0 = block_sum(d0, red);
  d1 = block_sum(d1, red);
  d2 = block_sum(d2, red);
  if (tid == 0) { sh[0] = data_ll; sh[1] = d0; sh[2] = d1; sh[3] = d2; }
  __syncthreads();
  const double ll = sh[0], dsum = sh[1], Ssum = sh[2], logsum = sh[3];
  const double mu_m = vec[0], mu_i = vec[1], a = vec[2], b = vec[3];
  const double Gl = (double)G;
  const double E = a / b;
  const double l2pi = 1.8378770664093454836;  // log(2 pi)
  double* grad = out + 1;
  double* A = out + 1 + Dg;

  if (tid == 0) {
    const double psi = spec[0], psi1 = spec[1], psi2 = spec[2];
    const double elt = psi - log(b);
    double F = ll - 0.5 * E * Ssum + 0.5 * Gl * elt + 0.5 * (-logsum + Gl * (1.0 + l2pi));
    double g0 = -E * dsum;
    double g1 = 0.5 * E * Gl / (mu_i * mu_i);
    double g2 = -0.5 * Ssum / b + 0.5 * Gl * psi1;
    double g3 = 0.5 * a * Ssum / (b * b) - 0.5 * Gl / b;
    double a00 = -E * Gl, a02 = -dsum / b, a03 = a * dsum / (b * b);
    double a11 = -E * Gl / (mu_i * mu_i * mu_i);
    double a12 = 0.5 * Gl / (b * mu_i * mu_i), a13 = -0.5 * a * Gl / (b * b * mu_i * mu_i);
    double a22 = 0.5 * Gl * psi2, a23 = 0.5 * Ssum / (b * b);
    double a33 = -a * Ssum / (b * b * b) + 0.5 * Gl / (b * b);
    if (include_global) {
      F += 0.5 * (-log(mu_i) + 1.0 + l2pi) + a - log(b) + spec[3] + (1.0 - a) * psi;
      F += -0.5 * pr.mu_info * ((mu_m - pr.mu_mean) * (mu_m - pr.mu_mean) + 1.0 / mu_i);
      F += (pr.tau_shape - 1.0) * elt - pr.tau_rate * E;
      g0 += -pr.mu_info * (mu_m - pr.mu_mean);
      g1 += -0.5 / mu_i + 0.5 * pr.mu_info / (mu_i * mu_i);
      g2 += 1.0 + (1.0 - a) * psi1 + (pr.tau_shape - 1.0) * psi1 - pr.tau_rate / b;
      g3 += -1.0 / b - (pr.tau_shape - 1.0) / b + pr.tau_rate * a / (b * b);
      a00 += -pr.mu_info;
      a11 += 0.5 / (mu_i * mu_i) - pr.mu_info / (mu_i * mu_i * mu_i);
      a22 += -psi1 + (1.0 - a) * psi2 + (pr.tau_shape - 1.0) * psi2;
      a23 += pr.tau_rate / (b * b);
      a33 += 1.0 / (b * b) + (pr.tau_shape - 1.0) / (b * b) - 2.0 * pr.tau_rate * a / (b * b * b);
    }
    sh[4] = F;
    if (ORDER >= 1) {
      const double j1 = vecmode ? 1.0 : mu_i - bd.mu_info, j2 = vecmode ? 1.0 : a - bd.tau_shape,
                   j3 = vecmode ? 1.0 : b - bd.tau_rate;
      grad[0] = -g0;
      grad[1] = -g1 * j1;
      grad[2] = -g2 * j2;
      grad[3] = -g3 * j3;
      if (ORDER >= 2) {
        const double jj[4] = {1.0, j1, j2, j3};
        const double gvv[4] = {-g0, -g1, -g2, -g3};
        const double m[4][4] = {{a00, 0.0, a02, a03}, {0.0, a11, a12, a13},
                                {a02, a12, a22, a23}, {a03, a13, a23, a33}};
        for (int r = 0; r < 4; ++r)
          for (int c = r; c < 4; ++c) {   // upper triangle, mirrored: exactly symmetric
            double h = -m[r][c] * jj[r] * jj[c];
            if (r == c && r > 0 && !vecmode) h += gvv[r] * jj[r];
            A[(size_t)r * Dg + c] = h;
            A[(size_t)c * Dg + r] = h;
          }
      }
    }
  }
  // beta entries: entropy + prior + data gradient, diagonal extras of A
  double fpart = 0.0;
  for (int k = tid; k < K; k += blockDim.x) {
    const double bmk = vec[4 + k], bik = vec[4 + K + k];
    const double rb = 1.0 / bik;
    if (include_global) {
      fpart += 0.5 * (-log(bik) + 1.0 + l2pi)
             - 0.5 * pr.beta_info * ((bmk - pr.beta_mean) * (bmk - pr.beta_mean) + rb);
    }
    if (ORDER >= 1) {
      double gbm = gsum[k];
      double gbi = -gsum[K + k] * rb * rb;
      if (include_global) {
        gbm += -pr.beta_info * (bmk - pr.beta_mean);
        gbi += -0.5 * rb + 0.5 * pr.beta_info * rb * rb;
      }
      const double jb = vecmode ? 1.0 : bik - bd.beta_info;
      grad[4 + k] = -gbm;
      grad[4 + K + k] = -gbi * jb;
      if (ORDER >= 2) {
        double emm = 0.0;
        double eii = gsum[K + k] * 2.0 * rb * rb * rb;
        if (include_global) {
          emm += -pr.beta_info;
          eii += 0.5 * rb * rb - pr.beta_info * rb * rb * rb;
        }
        double* a0 = A + (size_t)(4 + k) * Dg + 4 + k;
        double* a1 = A + (size_t)(4 + K + k) * Dg + 4 + K + k;
        *a0 = __ldcg(a0) - emm;
        *a1 = __ldcg(a1) - eii * jb * jb + (vecmode ? 0.0 : (-gbi) * jb);
      }
    }
  }
  fpart = block_sum(fpart, red);
  if (tid == 0) out[0] = -(sh[4] + fpart);
}

// ------------------------------------------------------------------------------------------
// One launch for the finishing passes (round 1: k_obs_fixup, k_finish and the first half of k_global):
// block 0 runs global_pre; the next n_gf blocks the Gram finish, the next n_loc the group-level chain rule,
// the last n_bor the border rows (block-uniform roles).
template <int ORDER>
__global__ void __launch_bounds__(256, 4)
k_finish(const double* __restrict__ vec, const double* __restrict__ gsc, const double* __restrict__ BR,
         double* __restrict__ gradl, double* __restrict__ L, double* __restrict__ B,
         double* locpart, const double* __restrict__ grampart, const GbJob* __restrict__ jobs,
         const GbSlot* __restrict__ slots, double* A, int K, int G, int n_loc, int n_bor, int n_gf,
         int gram_small, int NT, int gram_groups, int gram_chunks, lrvb_glmm_bounds bd, int vecmode,
         GroupFix fx, GlobalArgs ga) {
  // wait first: the dependent (k_global_post) signals ITS dependents after its own wait, so whoever follows
  // it may read B and L ahead of its wait (the CSR refill does)
  pdl_wait();
  pdl_launch_dependents();
  const int Dg = 4 + 2 * K;
  // the few blocks with long serial chains (special functions, the sums over the per-CTA Gram partials)
  // come first, so that they run under the stream of border blocks instead of after it
  const int bid = (int)blockIdx.x - 1;
  if (bid < 0) {
    global_pre<ORDER>(vec, ga, K);
  } else if (bid < n_gf) {
    if (gram_small) gram_small_finish_body(bid, grampart, vec, A, K, Dg, NT, gram_chunks, bd, vecmode);
    else gram_big_finish_body(bid, grampart, jobs, slots, vec, A, K, Dg, gram_groups, gram_chunks, bd, vecmode);
  } else if (bid < n_gf + n_loc) {
    local_body<ORDER>(bid - n_gf, n_loc, vec, gsc, gradl, L, locpart, K, G, bd, vecmode, fx);
  } else {
    border_body(bid - n_gf - n_loc, vec, BR, B, K, G, bd, vecmode, fx);
  }
}

// Single-CTA end of the evaluation: global_post on the results of k_finish.  Signals its dependents only
// after its own wait: when the next kernel's CTAs start, k_finish has completed (B, L and the Gram part
// of A are final); only what this kernel writes (KL, global gradient, corner and diagonal of A) needs
// the next kernel's own wait.
template <int ORDER>
__global__ void __launch_bounds__(256)
k_global_post(const double* __restrict__ vec, const double* locpart, int K, int G, lrvb_glmm_bounds bd, int vecmode,
              GlobalArgs ga) {
  pdl_wait();
  pdl_launch_dependents();
  global_post<ORDER>(vec, ga, locpart, K, G, bd, vecmode);
}

// ------------------------------------------------------------------------------------------
int plan_eval(lrvb_glmm* h, cudaStream_t st) {
  const int K = h->K, G = h->G, Q = h->Q;
  const int64_t N = h->N;
  // observation pass geometry (k_obs, K > 62: 64-row tiles; obs_nbuf = tile buffers, two when they fit)
  {
    const size_t tile = sizeof(double) * 64 * (size_t)K, extra = sizeof(double) * (2 * (size_t)(Q + 3) + 32 + 2);
    h->obs_nbuf = (2 * tile + extra <= 220 * 1024) ? 2 : 1;
    h->obs_smem = h->obs_nbuf * tile + extra;
    int64_t nt = (N + 63) / 64;
    h->obs_grid = (int)(nt < kNumSMs ? nt : kNumSMs);
    if (h->obs_grid < 1) h->obs_grid = 1;
  }
  if (K <= kOfMaxK) {
    // fused observation + group pass: every warp owns a contiguous multiple-of-32 range of rows.  The two-slot
    // geometry (of_*) serves the weight-cross pass (launch_weight_pass) and the influence pass (k_obs_influence).
    h->obs_fused = 1;
    h->of_warps = obs_fused_warps(K);
    const int64_t nst = (N + kOfRows - 1) / kOfRows;
    int64_t grid = (nst + h->of_warps - 1) / h->of_warps;
    if (grid > kNumSMs) grid = kNumSMs;
    if (grid < 1) grid = 1;
    h->of_grid = (int)grid;
    const int64_t tw = grid * h->of_warps;
    h->of_rows_per_warp = ((nst + tw - 1) / tw) * kOfRows;
    h->of_smem = obs_fused_smem(K, Q, h->of_warps);
    int64_t nrec = tw;
    {
      // the evaluation runs one-slot rings: they fit 16 down to 12 warps per SM where two slots fit 12 down to 6
      const int w1 = obs_fused_warps(K, 1);
      int64_t g1 = (nst + w1 - 1) / w1;
      if (g1 > kNumSMs) g1 = kNumSMs;
      if (g1 < 1) g1 = 1;
      const int64_t tw1 = g1 * w1;
      h->of1_grid = (int)g1;
      h->of1_warps = w1;
      h->of1_rows_per_warp = ((nst + tw1 - 1) / tw1) * kOfRows;
      h->of1_smem = obs_fused_smem(K, Q, w1, 1);
      if (tw1 > nrec) nrec = tw1;
      if (h->obs_grid < h->of1_grid) h->obs_grid = h->of1_grid;
      if ((K + 1 + 31) / 32 == 1) {
        LRVB_TRY(raise_smem_limit(k_obs_fused<0, 1, 1>, h->of1_smem));
        LRVB_TRY(raise_smem_limit(k_obs_fused<1, 1, 1>, h->of1_smem));
        LRVB_TRY(raise_smem_limit(k_obs_fused<2, 1, 1>, h->of1_smem));
      } else {
        LRVB_TRY(raise_smem_limit(k_obs_fused<0, 2, 1>, h->of1_smem));
        LRVB_TRY(raise_smem_limit(k_obs_fused<1, 2, 1>, h->of1_smem));
        LRVB_TRY(raise_smem_limit(k_obs_fused<2, 2, 1>, h->of1_smem));
      }
    }
    if (K <= kFuMaxK) {
      // order 2 in one pass (fused.cuh): teams of NQ quadrature warps + P DMMA warps, one CTA per SM; every
      // Q warp owns a contiguous multiple-of-32 range of rows.  Only for K <= 24, where quadrature and Gram
      // need about the same pipe time and the one-pass kernel is ~10 % faster than the two kernels; for larger
      // K the Gram dominates, the D warps of the one-pass kernel (128 registers, 4 warps per triangle) are
      // slower than gram_mid's (255 registers, 2 warps) and the two-kernel path wins
      // (profiles/r02_onepass_attempts.md).
      const int nqw = kFuGeom.teams * kFuGeom.NQ;
      int64_t fgrid = (nst + nqw - 1) / nqw;
      if (fgrid > kNumSMs) fgrid = kNumSMs;
      if (fgrid < 1) fgrid = 1;
      const int64_t tt = fgrid * nqw;
      h->fused2 = 1;
      h->fu_grid = (int)fgrid;
      h->fu_teams = nqw;
      h->fu_warps = kFuGeom.warps;
      h->fu_rows_per_team = ((nst + tt - 1) / tt) * kFuRows;
      h->fu_kernel = fused_eval_kernel(K);
      h->fu_smem = fused_smem(K, Q, gram_small_shape(K).T2);
      LRVB_TRY(raise_smem_limit(h->fu_kernel, h->fu_smem));
      if (tt > nrec) nrec = tt;
    }
    LRVB_TRY(dev_alloc(&h->bval, (size_t)nrec * 2 * (5 + 4 * (size_t)K)));
    if (h->obs_grid < h->of_grid) h->obs_grid = h->of_grid;
    if (h->obs_grid < h->fu_grid) h->obs_grid = h->fu_grid;     // klpart / gradpart are sized by obs_grid
  } else {
    LRVB_TRY(raise_smem_limit(k_obs<0>, h->obs_smem));
    LRVB_TRY(raise_smem_limit(k_obs<1>, h->obs_smem));
    LRVB_TRY(raise_smem_limit(k_obs<2>, h->obs_smem));
  }
  LRVB_TRY(dev_alloc(&h->klpart, (size_t)h->obs_grid));
  LRVB_TRY(dev_alloc(&h->gradpart, (size_t)h->obs_grid * 2 * K));

  LRVB_TRY(dev_alloc(&h->gsc, (size_t)G * 5));
  LRVB_TRY(dev_alloc(&h->BR, (size_t)G * 4 * K));
  h->loc_grid = cdiv(G, 256);
  if (h->loc_grid > 2 * kNumSMs) h->loc_grid = 2 * kNumSMs;
  if (h->loc_grid < 1) h->loc_grid = 1;
  LRVB_TRY(dev_alloc(&h->locpart, (size_t)h->loc_grid * 4));
  LRVB_TRY(dev_alloc(&h->fin_counter, 1));
  LRVB_TRY(dev_alloc(&h->fin_pre, 8 + 2 * (size_t)K));
  LRVB_CUDA(cudaMemsetAsync(h->fin_counter, 0, sizeof(unsigned int), st));

  // Gram geometry
  size_t npart;
  if (h->fused2) {
    // no Gram kernel: the one-pass kernel (fused.cuh) writes the packed partials, one slab per CTA
    npart = (size_t)h->fu_grid * gram_small_shape(K).NT * 64;
  } else if (K <= kGmMaxK) {
    // 24 < K <= 104: one warp or a team of warps = the whole packed triangle (gram_mid.cuh)
    const GramMidKernel gk = gram_mid_kernel(K);
    h->gram_mid = 1;
    h->gm_kernel = gk.fn;
    h->gm_warps = gk.warps;
    h->gram_smem = gram_mid_smem(K, gram_small_shape(K).T2);
    LRVB_TRY(raise_smem_limit(h->gm_kernel, h->gram_smem));
    h->gram_grid_x = kNumSMs;
    h->gram_grid_y = 1;
    npart = (size_t)h->gram_grid_x * gram_small_shape(K).NT * 64;
  } else if (gram_wide_eligible(K)) {
    // large K, no straddle tile: block-against-block jobs (16 - 25 tiles per warp), 8 warps per SM, only the
    // column blocks of a job group staged (gram_wide.cuh)
    const GwPlan pl = gram_wide_plan(K);
    h->gram_wide = 1;
    if (getenv("LRVB_GROUP_OVERLAP") && getenv("LRVB_GROUP_OVERLAP")[0] == '0') h->group_overlap = 0;
    h->gram_grid_x = (int)pl.ctas.size();
    h->gram_grid_y = (int)pl.groups.size();
    h->gram_smem = pl.smem;
    LRVB_TRY(raise_smem_limit(k_gram_wide, h->gram_smem));
    LRVB_TRY(dev_alloc((char**)&h->jobs, sizeof(GwGroup) * pl.groups.size()));
    LRVB_TRY(dev_alloc((char**)&h->gslots, sizeof(GwCta) * pl.ctas.size()));
    LRVB_CUDA(cudaMemcpyAsync(h->jobs, pl.groups.data(), sizeof(GwGroup) * pl.groups.size(),
                              cudaMemcpyHostToDevice, st));
    LRVB_CUDA(cudaMemcpyAsync(h->gslots, pl.ctas.data(), sizeof(GwCta) * pl.ctas.size(),
                              cudaMemcpyHostToDevice, st));
    LRVB_CUDA(cudaStreamSynchronize(st));   // pl goes out of scope
    npart = (size_t)h->gram_grid_x * gram_small_shape(K).NT * 64;
  } else {
    // rectangles of the packed triangle dealt to 16-warp CTAs (gram_big.cuh)
    const GbPlan pl = gram_big_plan(K);
    h->gram_jobs = (int)pl.jobs.size();
    h->gram_grid_y = pl.n_groups;
    h->gram_tn = pl.TN;
    h->gram_smem = pl.smem;
    LRVB_TRY(raise_smem_limit(k_gram_big, h->gram_smem));
    int64_t nst = (N + pl.TN - 1) / pl.TN;
    int64_t nchunk = (kNumSMs * kGbCtasPerSM) / pl.n_groups;
    if (nchunk > nst) nchunk = nst;
    if (nchunk < 1) nchunk = 1;
    h->gram_grid_x = (int)nchunk * pl.n_groups;
    LRVB_TRY(dev_alloc((char**)&h->jobs, sizeof(GbJob) * pl.jobs.size()));
    LRVB_TRY(dev_alloc((char**)&h->gslots, sizeof(GbSlot) * pl.slots.size()));
    LRVB_CUDA(cudaMemcpyAsync(h->jobs, pl.jobs.data(), sizeof(GbJob) * pl.jobs.size(),
                              cudaMemcpyHostToDevice, st));
    LRVB_CUDA(cudaMemcpyAsync(h->gslots, pl.slots.data(), sizeof(GbSlot) * pl.slots.size(),
                              cudaMemcpyHostToDevice, st));
    LRVB_CUDA(cudaStreamSynchronize(st));   // pl goes out of scope
    npart = (size_t)nchunk * pl.n_groups * kGbWarps * 16 * 64;
  }
  LRVB_TRY(dev_alloc(&h->grampart, npart));
  LRVB_CUDA(cudaMemsetAsync(h->grampart, 0, sizeof(double) * npart, st));
  return LRVB_OK;
}

// ------------------------------------------------------------------------------------------
int launch_eval(lrvb_glmm* h, const double* free_dev, int order, double* out_global,
                double* grad_local, cudaStream_t st) {
  const int K = h->K, G = h->G, Q = h->Q, Dg = h->Dg;
  const int64_t N = h->N;
  h->hess_valid = 0;
  h->grad_valid = 0;
  if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[4], st));
  double* outp = out_global ? out_global : h->outg;
  LRVB_CUDA(launch_pdl(k_prep, dim3(cdiv(h->D, 256)), dim3(256), 0, st, free_dev, h->vec, K, G, h->bounds,
                       h->vecmode, outp + 1 + Dg, (int64_t)(order >= 2 ? (int64_t)Dg * Dg : 0), h->shard_g0,
                       h->shard_G));
  LRVB_CHECK_LAUNCH();

  int n_obs_cta = 0;
  bool group_overlap = false;
  int64_t fix_rpw = 0;       // rows per warp of the fused producer whose straddling-group pieces sit in bval
  const bool one_pass = h->fused2 && order >= 2 && N > 0;
  h->ev_gram = 0;
  if (one_pass) {
    // order 2, K <= 24: quadrature, per-group sums and the packed Gram in ONE pass over X (fused.cuh)
    if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[0], st));
    FusedArgs fa;
    fa.X = h->X; fa.y = h->y; fa.g = h->g; fa.w = h->w; fa.vec = h->vec; fa.gh = h->gh; fa.gptr = h->gptr;
    fa.W = h->W; fa.ldw = h->ldw; fa.klpart = h->klpart; fa.gradpart = h->gradpart; fa.gsc = h->gsc; fa.BR = h->BR;
    fa.bval = h->bval; fa.grampart = h->grampart; fa.N = N; fa.K = K; fa.G = G; fa.Q = Q;
    fa.rows_per_q = h->fu_rows_per_team;
    LRVB_CUDA(launch_pdl(h->fu_kernel, dim3(h->fu_grid), dim3(32 * h->fu_warps), h->fu_smem, st, fa));
    LRVB_CHECK_LAUNCH();
    if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[1], st));
    n_obs_cta = h->fu_grid;
    fix_rpw = h->fu_rows_per_team;       // pieces of straddling groups are added by k_finish's readers
  } else if (h->obs_fused) {
    // K <= 62: observation pass and per-group sums in one kernel (obs_fused.cuh)
    if (N > 0) {
      if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[0], st));
      const int nch = (K + 1 + 31) / 32;
#define LRVB_OF(O, C)                                                                          \
  LRVB_CUDA(launch_pdl(k_obs_fused<O, C, 1>, dim3(h->of1_grid), dim3(32 * h->of1_warps), h->of1_smem, st, \
                       h->X, h->y, h->g, h->w, h->vec, h->gh, h->gptr, h->W, h->ldw, h->klpart, h->gradpart, \
                       h->gsc, h->BR, h->bval, N, K, G, Q, h->of1_rows_per_warp))
      if (nch == 1) {
        if (order == 0) LRVB_OF(0, 1);
        else if (order == 1) LRVB_OF(1, 1);
        else LRVB_OF(2, 1);
      } else {
        if (order == 0) LRVB_OF(0, 2);
        else if (order == 1) LRVB_OF(1, 2);
        else LRVB_OF(2, 2);
      }
#undef LRVB_OF
      LRVB_CHECK_LAUNCH();
      if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[1], st));
      n_obs_cta = h->of1_grid;
      fix_rpw = h->of1_rows_per_warp > 0 ? h->of1_rows_per_warp : 32;
    }
  } else {
  if (N > 0) {
    if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[0], st));
#define LRVB_OBS(O)                                                                          \
  k_obs<O><<<h->obs_grid, 256, h->obs_smem, st>>>(h->X, h->y, h->g, h->w, h->vec, h->gh, \
                                                   h->W, h->klpart, h->gradpart, N, h->ldw, K, G, Q, h->obs_nbuf)
    if (order == 0) LRVB_OBS(0);
    else if (order == 1) LRVB_OBS(1);
    else LRVB_OBS(2);
#undef LRVB_OBS
    LRVB_CHECK_LAUNCH();
    if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[1], st));
  }
  n_obs_cta = (N > 0) ? h->obs_grid : 0;

  // The per-group pass runs before the Gram kernel on the same stream -- except under k_gram_wide: its CTA (256
  // threads x 200 registers, one per SM) leaves room for exactly one k_group CTA (48 registers, no shared
  // memory) per SM, and the two kernels want different things (DMMA pipe at 22 % of the issue slots against
  // L2 / HBM latency), so k_group goes to the handle's side stream, is launched AFTER the Gram kernel and hides
  // behind it (C4: 4.8 ms of the step; LRVB_GROUP_OVERLAP=0 restores the serial order)
  group_overlap = h->gram_wide && order >= 2 && N > 0 && G > 0 && h->group_overlap;
  if (group_overlap) {
    LRVB_CUDA(cudaEventRecord(h->ev_fork, st));       // k_obs has written W
  } else if (order >= 1 && G > 0) {
    const int ggrid = (int)((G + 7) / 8 < 148 * 8 ? (G + 7) / 8 : 148 * 8);
    cudaStream_t gs = st;
    if (order == 1) k_group<1><<<ggrid, 256, 0, gs>>>(h->X, h->W, h->gptr, h->gsc, h->BR, h->ldw, K, G);
    else k_group<2><<<ggrid, 256, 0, gs>>>(h->X, h->W, h->gptr, h->gsc, h->BR, h->ldw, K, G);
    LRVB_CHECK_LAUNCH();
  }
  }
  if (order >= 2 && !one_pass) {
    if (N > 0) {
      h->ev_gram = 1;
      if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[2], st));
      if (h->gram_mid) {
        LRVB_CUDA(launch_pdl(h->gm_kernel, dim3(h->gram_grid_x), dim3(32 * h->gm_warps), h->gram_smem, st,
                             h->X, h->W + 2 * h->ldw, h->grampart, N, h->ldw, K));
      } else if (h->gram_wide) {
        LRVB_CUDA(launch_pdl(k_gram_wide, dim3(h->gram_grid_x), dim3(32 * kGwWarps), h->gram_smem, st,
            h->X, h->W + 2 * h->ldw, h->ldw, (const GwGroup*)h->jobs, (const GwCta*)h->gslots,
            h->grampart, N, K, gram_small_shape(K).NT));
      } else {
        LRVB_CUDA(launch_pdl(k_gram_big, dim3(h->gram_grid_x), dim3(32 * kGbWarps), h->gram_smem, st,
            h->X, h->W + 2 * h->ldw, h->ldw, (const GbJob*)h->jobs, (const GbSlot*)h->gslots,
            h->grampart, N, K, h->gram_tn, h->gram_grid_y, h->gram_grid_x / h->gram_grid_y));
      }
      LRVB_CHECK_LAUNCH();
      if (group_overlap) {
        const int ggrid = (int)((G + 7) / 8 < 148 * 8 ? (G + 7) / 8 : 148 * 8);
        LRVB_CUDA(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
        k_group<2><<<ggrid, 256, 0, h->side>>>(h->X, h->W, h->gptr, h->gsc, h->BR, h->ldw, K, G);
        LRVB_CHECK_LAUNCH();
        LRVB_CUDA(cudaEventRecord(h->ev_join, h->side));
        LRVB_CUDA(cudaStreamWaitEvent(st, h->ev_join, 0));
      }
      if (h->timing) LRVB_CUDA(cudaEventRecord(h->ev[3], st));
    }
  }
  double* gl = grad_local ? grad_local : h->gradl;
  {
    const int n_loc = h->loc_grid;
    int n_bor = 0, n_gf = 0, NT = 0;
    const int packed_gram = (h->gram_mid || h->gram_wide || one_pass) ? 1 : 0;   // partial layout (n_cta, NT, 64)
    const int packed_ctas = one_pass ? h->fu_grid : h->gram_grid_x;
    if (order >= 2) {
      if (G > 0) n_bor = cdiv(G, 8 * border_groups_per_warp(G));
      if (N > 0) {
        if (packed_gram) { NT = gram_small_shape(K).NT; n_gf = NT; }
        else n_gf = h->gram_jobs * 16;
      }
    }
    const int n_work = n_loc + n_bor + n_gf;
    GroupFix fx;
    fx.gptr = h->gptr; fx.bval = h->bval; fx.rpw = (N > 0) ? (unsigned)fix_rpw : 0u; fx.nb = 5 + 4 * K;
    if (N == 0 && h->obs_fused) {
      // no observation kernel ran: every group is empty, which the readers must see as zeros
      fx.rpw = 32;
    }
    fx.inv_rpw = fx.rpw ? 1.0 / (double)fx.rpw : 0.0;
    GlobalArgs ga;
    ga.klpart = h->klpart; ga.n_kl = n_obs_cta; ga.gradpart = h->gradpart; ga.n_gp = n_obs_cta;
    ga.n_lp = h->loc_grid; ga.out = outp; ga.pr = h->prior; ga.include_global = h->include_global;
    ga.counter = h->fin_counter;
    ga.pre = h->fin_pre;
    const size_t gsm = sizeof(double) * 2 * (size_t)K;
#define LRVB_FIN(O)                                                                              \
  LRVB_CUDA(launch_pdl(k_finish<O>, dim3(n_work + 1), dim3(256), 0, st, h->vec, h->gsc, h->BR, gl, h->L, h->B, \
                       h->locpart, h->grampart, (const GbJob*)h->jobs, (const GbSlot*)h->gslots,   \
                       outp + 1 + Dg, K, G, n_loc, n_bor, n_gf, packed_gram, NT, h->gram_grid_y,         \
                       packed_gram ? packed_ctas : h->gram_grid_x / (h->gram_grid_y > 0 ? h->gram_grid_y : 1), \
                       h->bounds, h->vecmode, fx, ga));                                            \
  LRVB_CHECK_LAUNCH();                                                                           \
  LRVB_CUDA(launch_pdl(k_global_post<O>, dim3(1), dim3(256), gsm, st, h->vec, h->locpart, K, G, h->bounds, \
                       h->vecmode, ga))
    if (order == 0) { LRVB_FIN(0); }
    else if (order == 1) { LRVB_FIN(1); }
    else { LRVB_FIN(2); }
#undef LRVB_FIN
    LRVB_CHECK_LAUNCH();
  }
  if (outp != h->outg) {
    const size_t nout = 1 + (order >= 1 ? Dg : 0) + (order >= 2 ? (size_t)Dg * Dg : 0);
    LRVB_CUDA(cudaMemcpyAsync(h->outg, outp, sizeof(double) * nout, cudaMemcpyDeviceToDevice, st));
  }
  if (gl != h->gradl && order >= 1)
    LRVB_CUDA(cudaMemcpyAsync(h->gradl, gl, sizeof(double) * 2 * (size_t)G, cudaMemcpyDeviceToDevice, st));
  if (order >= 2) {
    // the handle's own copy of the global block (A) lives inside outg
    h->A = h->outg + 1 + Dg;
    h->hess_valid = 1;
  }
  if (order >= 1) h->grad_valid = 1;
  h->point_valid = 1;
  if (h->timing) {
    LRVB_CUDA(cudaEventRecord(h->ev[5], st));
    h->ev_order = order;
  }
  return LRVB_OK;
}

}  // namespace lrvb
