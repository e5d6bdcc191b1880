// Per-observation pass fused with the per-group segmented sums (K <= 62), fp64, sm_100a.
//
// One kernel computes, for every observation n (SURVEY.md A.1/A.2; Modeling.py:35-52):
//   z_mean = E[u_g] + x.E[beta], z_var = Var[u_g] + x^2.Var[beta], the Q-node Gauss-Hermite
//   softplus / sigma / sigma' sums from ONE exp per node, and the analytic l, l_m, l_v, l_mm,
//   l_mv, l_vv  ->  W (5, ldw) and the KL partial,
// and, over the group-sorted rows, for every group g
//   gsc[g] = sum (l_m, l_v, a, b, c)          BR[g] = sum (a x, b x, b s, c s)  (4 x K)
// plus the global-gradient partials X^T l_m, S^T l_v.  X is read from HBM once.
//
// Layout of the work: every warp owns a contiguous range of rows (a multiple of 32) and streams it
// through a private two-slot shared-memory ring filled by bulk async copies (TMA; X rows, y, g, w
// of 32 observations per stage, one mbarrier per slot): no block barrier in the main loop.
//   phase A  lane = observation: the quadrature (bank-conflict-free row reads by a per-lane skew)
//   phase C  lane = column (plus one "ones" column that yields the scalar group sums): running
//            sums of the current group, flushed when the group id changes.
// A group that lies inside one warp's range is written by that warp; the pieces of a group that
// straddles range boundaries go to per-warp head / tail slots and k_obs_fixup adds them in row
// order, so there are no atomics and the summation order is fixed.
#pragma once
#include "common.cuh"
#include <type_traits>
#include "gram_small.cuh"   // mbarrier / bulk-copy helpers

namespace lrvb {

constexpr int kOfRows = 32;      // observations per stage (= lanes)
constexpr int kOfStages = 2;
#ifndef LRVB_OF_WARPS
#define LRVB_OF_WARPS 12
#endif
#ifndef LRVB_OF_UNROLL
#define LRVB_OF_UNROLL 4
#endif
constexpr int kOfMaxWarps = LRVB_OF_WARPS;
constexpr int kOfUnroll = LRVB_OF_UNROLL;   // quadrature nodes in flight per lane
constexpr int kOfMaxK = 62;      // K + 1 columns in at most two 32-lane chunks

// doubles per stage: X rows | y | w | g (int32, 16 doubles)
__host__ __device__ inline int obs_fused_stage_elems(int K) { return kOfRows * K + 2 * kOfRows + kOfRows / 2; }
// per-warp shared memory (doubles): ring + weights of the current stage (32 rows x 6: l_m, l_v, a, b, c, -)
__host__ __device__ inline int obs_fused_warp_elems(int K, int slots = kOfStages) {
  return slots * obs_fused_stage_elems(K) + 6 * kOfRows;
}
// One-slot variant (SLOTS = 1): from K ~ 36 on a two-slot ring leaves room for fewer than 10 warps per SM
// (7 at K = 50) and the pass is latency-bound; with ONE slot per warp -- the next stage is requested when
// the current one is finished, the other warps cover the copy -- up to 14 warps fit.  It fits at least three
// more warps than two slots for every K <= 62, so the evaluation always runs it; the weight-cross pass
// (launch_weight_pass) and the influence pass (k_obs_influence) keep two slots.
constexpr int kOfMaxWarps1 = 16;
inline int obs_fused_warps(int K, int slots = kOfStages) {
  // all of the 227 KB a CTA may own (one CTA per SM): per warp its ring, weights, gradient partials (2K), KL
  // partial and mbarriers; 2K + 2Q shared by the CTA (Q <= 64 assumed for the budget)
  const size_t per_warp = sizeof(double) * ((size_t)obs_fused_warp_elems(K, slots) + 2 * K + 1) +
                          sizeof(unsigned long long) * slots;
  const size_t fixed = sizeof(double) * (2 * (size_t)K + 2 * 64);
  int w = (int)((227 * 1024 - fixed) / per_warp);
  const int cap = slots == 1 ? kOfMaxWarps1 : kOfMaxWarps;
  if (w > cap) w = cap;
  return w < 1 ? 1 : w;
}
inline size_t obs_fused_smem(int K, int Q, int warps, int slots = kOfStages) {
  return sizeof(double) * ((size_t)warps * obs_fused_warp_elems(K, slots) + 2 * K + 2 * Q + 2 * (size_t)warps * K +
                           warps) + sizeof(unsigned long long) * warps * slots;
}

struct GHSumsF {
  double A, Am, As, Amm, Ams, Ass;
  double App;   // sum what sigma^2 (ORDER >= 3: prediction, csrc/predict.cu)
};

// ---- branch-free fp64 kernels of the quadrature node ----------------------------------------
// The CUDA math library's exp / log1p / division carry rare-case branches, which stop the compiler
// from interleaving the (serial) chains of independent nodes.  These are straight-line: exp on
// x <= 0 by the usual 2^n * P(f) reduction (minimax degree 11, |f| <= ln2/2, error 3.6e-18), and
// r = 1/(1+e), L = log1p(e) for e in [0,1] from ONE reciprocal:
//   y = 1/((1+e)(2+e))   (MUFU seed + 3 Newton steps),  r = y (2+e),  u = e/(2+e) = e y (1+e),
//   log1p(e) = 2 atanh(u) = 2 u P(u^2)   (minimax degree 10 on u^2 <= 1/9, error 1.3e-18).
// Verified against mpmath on [-630, 0]: 2.2e-16 (exp) and 4.9e-16 (log1p o exp) max relative error.
// polynomial coefficients in the constant bank: DFMA takes them as c[bank][offset] operands, which
// saves the two moves per 64-bit immediate the compiler would otherwise issue for every use
__constant__ double kExpC[10] = {0x1.af683d6885e31p-26, 0x1.28b8302ee0724p-22, 0x1.71ddf2a82093ep-19,
                                 0x1.a0198d1fda4aap-16, 0x1.a01a01b251e85p-13, 0x1.6c16c189b379fp-10,
                                 0x1.111111110ef94p-7,  0x1.555555554e879p-5,  0x1.555555555555bp-3,
                                 0x1.0000000000012p-1};
__constant__ double kAtanhC[10] = {0x1.5d1081172f887p-4, 0x1.54f8c703ce149p-5, 0x1.f00852a5c69fap-5,
                                   0x1.106443d797a85p-4, 0x1.3b1e2bc8a12dep-4, 0x1.745caf74cbe5ep-4,
                                   0x1.c71c7445b2127p-4, 0x1.249249201beacp-3, 0x1.99999999a1c4fp-3,
                                   0x1.5555555555527p-2};

__device__ __forceinline__ double exp_nonpos(double x) {
  x = fmax(x, -708.0);                                   // below: e < 1e-307, contributes nothing
  const double magic = 6755399441055744.0;               // 1.5 * 2^52: round-to-nearest-int trick
  double nd = fma(x, 1.4426950408889634, magic);
  const int n = __double2loint(nd);
  nd -= magic;
  double f = fma(nd, -6.93147180369123816490e-01, x);    // ln2 hi / lo (fdlibm split)
  f = fma(nd, -1.90821492927058770002e-10, f);
  double p = kExpC[0];
#pragma unroll
  for (int i = 1; i < 10; ++i) p = fma(p, f, kExpC[i]);
  p = fma(p, f, 1.0);
  p = fma(p, f, 1.0);
  return p * __hiloint2double((n + 1023) << 20, 0);      // n in [-1022, 0]
}

__device__ __forceinline__ void rcp_log1p_unit(double e, double& r, double& L) {
  const double a = 1.0 + e, b = 2.0 + e;
  const double ab = a * b;                               // in [2, 6]
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(ab));
  double t = fma(-ab, y, 1.0);
  y = fma(y, t, y);
  t = fma(-ab, y, 1.0);
  y = fma(y, t, y);
  t = fma(-ab, y, 1.0);
  y = fma(y, t, y);
  r = y * b;
  const double u = e * (y * a);
  const double v = u * u;
  double p = kAtanhC[0];
#pragma unroll
  for (int i = 1; i < 10; ++i) p = fma(p, v, kAtanhC[i]);
  p = fma(p, v, 1.0);
  L = (u + u) * p;
}

// Gauss-Hermite node: softplus(t), sigma(t), sigma'(t) from ONE exp.  Modeling.py:48 evaluates
// log1p(exp(t)) unstabilised; max(t,0) + log1p(exp(-|t|)) is the same function on the finite
// range and stays finite beyond it.
template <int ORDER>
__device__ __forceinline__ void gh_node_f(double t, double c, double wq, GHSumsF& s) {
  const double e = exp_nonpos(-fabs(t));
  double r, L;
  rcp_log1p_unit(e, r, L);
  const double sp = fmax(t, 0.0) + L;
  s.A = fma(wq, sp, s.A);
  if (ORDER >= 1) {
    const double er = e * r;
    const double sg = (t >= 0.0) ? r : er;
    const double wsg = wq * sg;
    s.Am += wsg;
    s.As = fma(wsg, c, s.As);
    if (ORDER >= 2) {
      const double wd = wq * (er * r);
      const double wdc = wd * c;
      s.Amm += wd;
      s.Ams += wdc;
      s.Ass = fma(wdc, c, s.Ass);
    }
  }
}

// U Gauss-Hermite nodes at once, written step by step ACROSS the nodes: a dependent FP64 instruction
// issues ~24 cycles after its producer on this chip, and with gh_node_f called U times the compiler
// overlaps the chains only in pairs (SASS of round 1: the four reciprocal seeds of an "unroll 4" loop were
// ~50, ~220 and ~80 instructions apart).  Here every step of the exp / reciprocal / atanh chains is a loop
// over the U nodes, so U independent instructions sit next to each other in program order.
// Adds the nodes ghc[0..U), ghw[0..U) to s in increasing node order.
template <int ORDER, int U>
__device__ __forceinline__ void gh_nodes_f(double zm, double zs, const double* __restrict__ ghc,
                                           const double* __restrict__ ghw, GHSumsF& s) {
  const double magic = 6755399441055744.0;
  double t[U], c[U], x[U], nd[U], f[U], p[U], e[U];
  int n[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    c[u] = ghc[u];
    t[u] = fma(zs, c[u], zm);
    x[u] = fmax(-fabs(t[u]), -708.0);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) nd[u] = fma(x[u], 1.4426950408889634, magic);
#pragma unroll
  for (int u = 0; u < U; ++u) {
    n[u] = __double2loint(nd[u]);
    nd[u] -= magic;
  }
#pragma unroll
  for (int u = 0; u < U; ++u) f[u] = fma(nd[u], -6.93147180369123816490e-01, x[u]);
#pragma unroll
  for (int u = 0; u < U; ++u) f[u] = fma(nd[u], -1.90821492927058770002e-10, f[u]);
#pragma unroll
  for (int u = 0; u < U; ++u) p[u] = kExpC[0];
#pragma unroll
  for (int i = 1; i < 10; ++i) {
#pragma unroll
    for (int u = 0; u < U; ++u) p[u] = fma(p[u], f[u], kExpC[i]);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) p[u] = fma(p[u], f[u], 1.0);
#pragma unroll
  for (int u = 0; u < U; ++u) p[u] = fma(p[u], f[u], 1.0);
#pragma unroll
  for (int u = 0; u < U; ++u) e[u] = p[u] * __hiloint2double((n[u] + 1023) << 20, 0);
  // r = 1 / (1 + e), L = log1p(e) = 2 atanh(e / (2 + e)) from one reciprocal of (1 + e)(2 + e)
  double a1[U], b2[U], ab[U], y[U], tt[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    a1[u] = 1.0 + e[u];
    b2[u] = 2.0 + e[u];
  }
#pragma unroll
  for (int u = 0; u < U; ++u) ab[u] = a1[u] * b2[u];
#pragma unroll
  for (int u = 0; u < U; ++u) asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y[u]) : "d"(ab[u]));
#pragma unroll
  for (int it = 0; it < 3; ++it) {
#pragma unroll
    for (int u = 0; u < U; ++u) tt[u] = fma(-ab[u], y[u], 1.0);
#pragma unroll
    for (int u = 0; u < U; ++u) y[u] = fma(y[u], tt[u], y[u]);
  }
  double r[U], uu[U], v[U], pl[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    r[u] = y[u] * b2[u];
    uu[u] = e[u] * (y[u] * a1[u]);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    v[u] = uu[u] * uu[u];
    pl[u] = kAtanhC[0];
  }
#pragma unroll
  for (int i = 1; i < 10; ++i) {
#pragma unroll
    for (int u = 0; u < U; ++u) pl[u] = fma(pl[u], v[u], kAtanhC[i]);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) pl[u] = fma(pl[u], v[u], 1.0);
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const double L = (uu[u] + uu[u]) * pl[u];
    const double wq = ghw[u];
    const double sp = fmax(t[u], 0.0) + L;
    s.A = fma(wq, sp, s.A);
    if (ORDER >= 1) {
      const double er = e[u] * r[u];
      const double sg = (t[u] >= 0.0) ? r[u] : er;
      const double wsg = wq * sg;
      s.Am += wsg;
      s.As = fma(wsg, c[u], s.As);
      if (ORDER >= 2) {
        const double wd = wq * (er * r[u]);
        const double wdc = wd * c[u];
        s.Amm += wd;
        s.Ams += wdc;
        s.Ass = fma(wdc, c[u], s.Ass);
      }
      if (ORDER >= 3) s.App = fma(wsg, sg, s.App);
    }
  }
}

// All Q nodes of one observation, U at a time (then 2, then 1).
template <int ORDER, int U>
__device__ __forceinline__ void gh_all_nodes_f(double zm, double zs, const double* __restrict__ ghc,
                                               const double* __restrict__ ghw, int Q, GHSumsF& s) {
  int q = 0;
  for (; q + U <= Q; q += U) gh_nodes_f<ORDER, U>(zm, zs, ghc + q, ghw + q, s);
  if (U > 2)
    for (; q + 2 <= Q; q += 2) gh_nodes_f<ORDER, 2>(zm, zs, ghc + q, ghw + q, s);
  for (; q < Q; ++q) gh_nodes_f<ORDER, 1>(zm, zs, ghc + q, ghw + q, s);
}

// bval: (total_warps, 2, 5 + 4K) head / tail partials of groups that straddle a range boundary.
template <int ORDER, int NCH, int SLOTS = kOfStages>
__global__ void __launch_bounds__(32 * (SLOTS == 1 ? kOfMaxWarps1 : kOfMaxWarps), 1)
k_obs_fused(const double* __restrict__ X, const double* __restrict__ y, const int32_t* __restrict__ g,
            const double* __restrict__ w, const double* __restrict__ vec, const double* __restrict__ gh,
            const int32_t* __restrict__ gptr, double* __restrict__ W, int64_t ldw,
            double* __restrict__ klpart, double* __restrict__ gradpart, double* __restrict__ gsc,
            double* __restrict__ BR, double* __restrict__ bval, int64_t N, int K, int G, int Q,
            int64_t rows_per_warp) {
  pdl_sync();
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int stage_elems = obs_fused_stage_elems(K);
  const int warp_elems = obs_fused_warp_elems(K, SLOTS);
  double* ring = sm + (size_t)warp * warp_elems;
  double* wsm = ring + SLOTS * stage_elems;            // 32 x 6 weights of the current stage
  double* bm = sm + (size_t)nwarp * warp_elems;            // K   E[beta]
  double* bv = bm + K;                                     // K   Var[beta]
  double* ghc = bv + K;                                    // Q   sqrt(2) x_q
  double* ghw = ghc + Q;                                   // Q   w_q / sqrt(pi)
  double* gred = ghw + Q;                                  // nwarp x 2K gradient partials
  double* kred = gred + (size_t)nwarp * 2 * K;             // nwarp
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(kred + nwarp) + warp * SLOTS;
  const unsigned ring_u = smem_u32(ring), bars_u = smem_u32(bars);

  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    bm[k] = vec[4 + k];
    bv[k] = 1.0 / vec[4 + K + k];
  }
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    ghc[q] = gh[q];
    ghw[q] = gh[Q + q];
  }
  if (lane == 0) {
#pragma unroll
    for (int p = 0; p < SLOTS; ++p) mbar_init(bars_u + 8 * p, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();

  const int64_t um0 = 4 + 2 * (int64_t)K, ui0 = um0 + G;
  const int64_t gw = (int64_t)blockIdx.x * nwarp + warp;
  const int64_t rs = gw * rows_per_warp;                             // range start
  const int64_t re = (rs + rows_per_warp < N) ? rs + rows_per_warp : N;   // range end
  const int nst = (rs < re) ? (int)((re - rs + kOfRows - 1) / kOfRows) : 0;
  const unsigned xbytes = (unsigned)(kOfRows * K * sizeof(double));
  const unsigned vbytes = (unsigned)(kOfRows * sizeof(double));
  const unsigned gbytes = (unsigned)(kOfRows * sizeof(int32_t));
  const unsigned nops = w ? 4u : 3u;

  auto issue = [&](int st, int slot) {
    const int64_t n0 = rs + (int64_t)st * kOfRows;
    if (st < nst && n0 + kOfRows <= N && lane < (int)nops) {
      const unsigned bar = bars_u + 8 * slot;
      const unsigned dst = ring_u + (unsigned)(slot * stage_elems * sizeof(double));
      if (lane == 0) {
        mbar_arrive_expect_tx(bar, xbytes + (w ? 2 : 1) * vbytes + gbytes);
        bulk_g2s(dst, X + n0 * K, xbytes, bar);
      } else if (lane == 1) {
        bulk_g2s(dst + xbytes, y + n0, vbytes, bar);
      } else if (lane == 2) {
        bulk_g2s(dst + xbytes + 2 * vbytes, g + n0, gbytes, bar);
      } else {
        bulk_g2s(dst + xbytes + vbytes, w + n0, vbytes, bar);
      }
    }
  };
  auto acquire = [&](int st, int slot, unsigned ph) {
    const int64_t n0 = rs + (int64_t)st * kOfRows;
    if (n0 + kOfRows <= N) {
      mbar_wait(bars_u + 8 * slot, ph);
    } else {   // ragged last stage of the data set: filled by the warp itself
      double* xs = ring + (size_t)slot * stage_elems;
      const int rows = (int)(N - n0);
      for (int e = lane; e < kOfRows * K; e += 32) xs[e] = (e < rows * K) ? X[n0 * K + e] : 0.0;
      double* ys = xs + kOfRows * K;
      ys[lane] = (lane < rows) ? y[n0 + lane] : 0.0;
      ys[kOfRows + lane] = (lane < rows && w) ? w[n0 + lane] : 0.0;
      reinterpret_cast<int32_t*>(ys + 2 * kOfRows)[lane] = (lane < rows) ? g[n0 + lane] : -1;
      __syncwarp();
    }
  };

  // bank-conflict skew for the row-per-lane reads of the stage (row stride K doubles)
  int gcd16 = 1;
  while (gcd16 < 16 && (K % (gcd16 * 2)) == 0) gcd16 *= 2;
  int skew = ((lane & 15) * gcd16) >> 4;
  if (skew >= K) skew = 0;

  // phase C state: lane = column k0 (+32 per chunk); column K is the "ones" column
  double gm[NCH], gv[NCH];                 // global-gradient partials of the warp
  double q0[NCH], q1[NCH], q2[NCH], q3[NCH], q4[NCH], q5[NCH];   // current group: lm x, lv s, a x, b x, b s, c s
#pragma unroll
  for (int c = 0; c < NCH; ++c) gm[c] = gv[c] = q0[c] = q1[c] = q2[c] = q3[c] = q4[c] = q5[c] = 0.0;
  int cur_g = -1;
  double klacc = 0.0;
  const int nb = 5 + 4 * K;

  auto flush = [&]() {
    if (cur_g < 0) return;
    const int64_t gb = gptr[cur_g], ge = gptr[cur_g + 1];
    double* dbr;
    double* dsc;
    if (gb >= rs && ge <= re) {          // the whole group is ours
      dbr = BR + (size_t)cur_g * 4 * K;
      dsc = gsc + (size_t)cur_g * 5;
    } else {                             // head (starts before our range) or tail piece
      double* rec = bval + ((size_t)gw * 2 + (gb < rs ? 0 : 1)) * nb;
      dsc = rec;
      dbr = rec + 5;
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int k = lane + 32 * c;
      if (k < K) {
        if (ORDER >= 2) {
          dbr[k] = q2[c];
          dbr[K + k] = q3[c];
          dbr[2 * K + k] = q4[c];
          dbr[3 * K + k] = q5[c];
        }
        gm[c] += q0[c];
        gv[c] += q1[c];
      } else if (k == K) {               // ones column: sum l_m, l_v, a, b, c
        dsc[0] = q0[c];
        dsc[1] = q1[c];
        dsc[2] = (ORDER >= 2) ? q2[c] : 0.0;
        dsc[3] = (ORDER >= 2) ? q3[c] : 0.0;
        dsc[4] = (ORDER >= 2) ? q5[c] : 0.0;
      }
      q0[c] = q1[c] = q2[c] = q3[c] = q4[c] = q5[c] = 0.0;
    }
  };

#pragma unroll
  for (int p = 0; p < SLOTS; ++p) issue(p, p);

  int slot = 0;
  unsigned phase = 0;
  for (int st = 0; st < nst; ++st) {
    acquire(st, slot, phase);
    const int64_t n0 = rs + (int64_t)st * kOfRows;
    const double* xs = ring + (size_t)slot * stage_elems;
    const double* ys = xs + kOfRows * K;
    const int32_t* gs = reinterpret_cast<const int32_t*>(ys + 2 * kOfRows);
    const int rows = (int)((re - n0 < kOfRows) ? (re - n0) : kOfRows);

    // ---- phase A: lane = observation ----
    unsigned segmask;   // bit r: row r starts a new group segment
    {
      const int64_t n = n0 + lane;
      const bool valid = lane < rows;
      const int gi = valid ? gs[lane] : 0;
      {
        const int gprev = __shfl_up_sync(0xffffffffu, gi, 1);
        segmask = __ballot_sync(0xffffffffu, valid && (lane == 0 ? gi != cur_g : gi != gprev));
      }
      double zm = vec[um0 + gi];
      double zv = 1.0 / vec[ui0 + gi];
      const double* xr = xs + (size_t)lane * K;
      for (int k = skew; k < K; ++k) {
        const double x = xr[k];
        zm = fma(x, bm[k], zm);
        zv = fma(x * x, bv[k], zv);
      }
      for (int k = 0; k < skew; ++k) {
        const double x = xr[k];
        zm = fma(x, bm[k], zm);
        zv = fma(x * x, bv[k], zv);
      }
      const double zs = sqrt(zv);
      GHSumsF s = {0, 0, 0, 0, 0, 0};
      // kOfUnroll independent nodes at a time, interleaved step by step (gh_nodes_f)
      gh_all_nodes_f<ORDER, kOfUnroll>(zm, zs, ghc, ghw, Q, s);
      const double wn = valid ? (w ? ys[kOfRows + lane] : 1.0) : 0.0;
      const double yn = ys[lane];
      klacc += wn * (yn * zm - s.A);
      if (ORDER >= 1) {
        const double h = 0.5 / zs;
        const double lm = wn * (yn - s.Am);
        const double lv = -wn * s.As * h;
        double2* wrow = reinterpret_cast<double2*>(wsm + 6 * lane);
        wrow[0] = make_double2(lm, lv);
        if (valid && W) {     // W == nullptr: sums only (the weight cross-Hessian matvec)
          W[n] = lm;
          W[ldw + n] = lv;
        }
        if (ORDER >= 2) {
          const double a = -wn * s.Amm;
          const double b = -wn * s.Ams * h;
          // l_vv = -(A_ss / (4 z_v) - A_s / (4 z_s^3))
          const double c = -wn * (s.Ass - s.As / zs) / (4.0 * zv);
          wrow[1] = make_double2(a, b);
          wrow[2] = make_double2(c, 0.0);
          if (valid && W) {
            W[2 * ldw + n] = a;
            W[3 * ldw + n] = b;
            W[4 * ldw + n] = c;
          }
        }
      }
    }

    // ---- phase C: lane = column; running sums of the current group over the rows of the stage,
    // one tight loop per group segment (segment starts come from the ballot above) ----
    if (ORDER >= 1) {
      __syncwarp();
      const double2* w2 = reinterpret_cast<const double2*>(wsm);
      int koff[NCH];
      bool isone[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int k = lane + 32 * c;
        koff[c] = (k < K) ? k : 0;        // lanes beyond the ones column compute garbage nobody stores
        isone[c] = (k == K);
      }
      auto rows_acc = [&](int r, auto nrow) {   // nrow consecutive rows of the current group
        constexpr int NR = decltype(nrow)::value;
        double2 wl[NR], wab[NR], wc[NR];
        double x[NR][NCH];
#pragma unroll
        for (int u = 0; u < NR; ++u) {
          wl[u] = w2[3 * (r + u)];
          if (ORDER >= 2) { wab[u] = w2[3 * (r + u) + 1]; wc[u] = w2[3 * (r + u) + 2]; }
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            const double v = xs[(size_t)(r + u) * K + koff[c]];
            x[u][c] = isone[c] ? 1.0 : v;
          }
        }
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0, t4 = 0.0, t5 = 0.0;
#pragma unroll
          for (int u = 0; u < NR; ++u) {
            const double xv = x[u][c], xx = xv * xv;
            t0 = fma(wl[u].x, xv, t0);
            t1 = fma(wl[u].y, xx, t1);
            if (ORDER >= 2) {
              t2 = fma(wab[u].x, xv, t2);
              t3 = fma(wab[u].y, xv, t3);
              t4 = fma(wab[u].y, xx, t4);
              t5 = fma(wc[u].x, xx, t5);
            }
          }
          q0[c] += t0; q1[c] += t1;
          if (ORDER >= 2) { q2[c] += t2; q3[c] += t3; q4[c] += t4; q5[c] += t5; }
        }
      };
      int r = 0;
      unsigned m = segmask;
      while (r < rows) {
        if ((m >> r) & 1u) {            // row r opens a new group
          flush();
          cur_g = gs[r];
        }
        const unsigned rest = (r + 1 < 32) ? (m >> (r + 1)) : 0u;
        const int nxt = rest ? (r + 1 + __ffs((int)rest) - 1) : rows;   // next segment start
        const int r1 = nxt < rows ? nxt : rows;
        for (; r + 4 <= r1; r += 4) rows_acc(r, std::integral_constant<int, 4>());
        for (; r < r1; ++r) rows_acc(r, std::integral_constant<int, 1>());
      }
    }
    __syncwarp();   // every lane is done with this slot (and with wsm) before the refill
    issue(st + SLOTS, slot);
    if (++slot == SLOTS) { slot = 0; phase ^= 1; }
  }
  if (ORDER >= 1) flush();

  // ---- CTA reduction: KL partial and global-gradient partials, fixed order ----
  klacc = warp_sum(klacc);
  if (lane == 0) kred[warp] = klacc;
  if (ORDER >= 1) {
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int k = lane + 32 * c;
      if (k < K) {
        gred[(size_t)warp * 2 * K + k] = gm[c];
        gred[(size_t)warp * 2 * K + K + k] = gv[c];
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < nwarp; ++i) s += kred[i];
    klpart[blockIdx.x] = s;
  }
  if (ORDER >= 1) {
    // layout (2K, n_cta): column-major over CTAs so the finishing reduce reads contiguously
    for (int k = threadIdx.x; k < 2 * K; k += blockDim.x) {
      double s = 0.0;
      for (int i = 0; i < nwarp; ++i) s += gred[(size_t)i * 2 * K + k];
      gradpart[(size_t)k * gridDim.x + blockIdx.x] = s;
    }
  }
}

// Groups whose rows straddle the row ranges of several warps: add their head / tail pieces in
// row order.  One warp per group; empty groups get zeros; groups owned by one warp are skipped.
template <int ORDER>
__global__ void __launch_bounds__(256)
k_obs_fixup(const int32_t* __restrict__ gptr, const double* __restrict__ bval,
            double* __restrict__ gsc, double* __restrict__ BR, int K, int G, int64_t rows_per_warp) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  const int nb = 5 + 4 * K;
  const int gi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (gi >= G) return;
  const int64_t gb = gptr[gi], ge = gptr[gi + 1];
  double* dsc = gsc + (size_t)gi * 5;
  double* dbr = BR + (size_t)gi * 4 * K;
  if (gb == ge) {
    for (int e = lane; e < nb; e += 32) {
      if (e < 5) dsc[e] = 0.0;
      else if (ORDER >= 2) dbr[e - 5] = 0.0;
    }
    return;
  }
  const int64_t wf = gb / rows_per_warp, wl = (ge - 1) / rows_per_warp;
  if (wf == wl) return;
  for (int e = lane; e < nb; e += 32) {
    if (e >= 5 && ORDER < 2) break;
    double s = bval[((size_t)wf * 2 + 1) * nb + e];                       // tail of the first warp
    for (int64_t wi = wf + 1; wi <= wl; ++wi) s += bval[((size_t)wi * 2) * nb + e];   // heads
    if (e < 5) dsc[e] = s;
    else dbr[e - 5] = s;
  }
}

}  // namespace lrvb
