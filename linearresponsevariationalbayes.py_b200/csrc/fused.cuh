// Order-2 evaluation in ONE pass over X: the per-observation quadrature + per-group sums of obs_fused.cuh
// and the packed weighted Gram of gram_mid.cuh as one persistent, warp-specialised kernel (K <= 24), sm_100a.
//
// Why: run back to back, the observation pass keeps the FP64 pipe ~50 % busy and the Gram kernel ~80 %
// (DMMA), and each reads X from HBM.  What limits the observation pass is the DEPENDENT-issue latency of
// FP64 on this chip: the measurements of this round fit ~24 cycles per dependent DFMA (DMMA: 26), so a
// sub-partition needs ~12 independent FP64 chains in flight to fill its pipe (one DFMA per 2 cycles), and
// the 161-register observation kernel reaches 3 warps x ~2 chains.  A DMMA warp needs no such help (16+
// independent accumulator tiles).  So: put quadrature warps and DMMA warps on the same sub-partition and let
// the tensor instructions fill the cycles the quadrature chains leave empty.
//
// A CTA is a set of TEAMS; a team is NQ Q warps (quadrature, lane = observation, 4 nodes in flight; then the
// per-group sums, lane = column -- the code of k_obs_fused) and P D warps (the packed [x|s] triangle on
// DMMA.8x8x4 -- the code of k_gram_mid).  Every Q warp owns a contiguous multiple-of-32 range of rows and
// its own ring of 32-row stages; the team's D warps consume the stages of its Q warps round-robin:
//
//   TMA (Q lane 0) --full--> Q warp: weights l_m,l_v,a,b,c of the 32 rows into the slot --ready--> D warps:
//   8 k-steps of the packed Gram with those weights --empty (Q + P arrivals)--> refill of the slot
//
// X is read from HBM once (8K + 12 B per observation + the 40 B W store), the weights a, b, c never leave
// the SM on their way to the tensor pipe.  Groups inside a Q warp's range are written directly, head / tail
// pieces of straddling groups go to bval and k_obs_fixup adds them in row order.  No atomics, fixed
// summation orders: results are bitwise reproducible for a given launch geometry.
//
// Two earlier versions are kept in the history with their measurements (profiles/r02_onepass_attempts.md):
// one Q warp (2 nodes in flight) per D warp -- Q-bound, exactly as slow as the two kernels; and homogeneous
// teams in which every warp did quadrature, group sums and its share of the Gram -- no faster either (the
// accumulators leave too few registers for enough chains), and 2x slower when the Q/C code was a real call
// (local-memory traffic with the L1 carved down to a few KB).
//
// Slot (doubles): X 32 x K | y 32 | w 32 | g (int32 x 32) | wq 32 x 6 = (l_m, l_v, a, b, c, -) per row.
// Barriers per slot: full (1 arrival + tx bytes), ready (1: the Q warp), empty (1 + P).
#pragma once
#include "common.cuh"
#include "gram_small.cuh"
#include "gram_mid.cuh"
#include "obs_fused.cuh"

namespace lrvb {

constexpr int kFuRows = 32;          // rows per stage (= lanes of the Q warp = 8 k-steps)
#ifndef LRVB_FUSED_UNROLL
#define LRVB_FUSED_UNROLL 4
#endif
constexpr int kFuUnroll = LRVB_FUSED_UNROLL;   // quadrature nodes in flight per lane

// K <= 24 (T2 <= 6), where quadrature and Gram need about the same pipe time
constexpr int kFuMaxK = 24;

struct FusedGeom {
  int teams, NQ, P, warps, slots;    // warps = CTA size / 32; slots = ring depth per Q warp
};
// 4 teams -- one per SM sub-partition -- of 3 Q warps + 1 D warp (15 / 21 accumulator tiles), 2-slot rings
constexpr FusedGeom kFuGeom = {4, 3, 1, 16, 2};
__host__ __device__ inline int fused_slot_elems(int K) { return kFuRows * K + 2 * kFuRows + kFuRows / 2 + 6 * kFuRows; }
inline size_t fused_smem(int K, int Q, int T2) {
  const int nq = kFuGeom.teams * kFuGeom.NQ;
  const size_t ring = sizeof(double) * (size_t)nq * kFuGeom.slots * fused_slot_elems(K);
  const size_t red = sizeof(double) * (size_t)(T2 * (T2 + 1) / 2) * 64;
  const size_t body = ring > red ? ring : red;
  // + beta mean / var (2K), GH nodes (2Q), gradient partials (Q warps x 2K), KL partials (Q warps), barriers
  return body + sizeof(double) * (2 * (size_t)K + 2 * Q + (size_t)nq * 2 * K + nq) +
         sizeof(unsigned long long) * (size_t)nq * kFuGeom.slots * 3;
}

struct FusedArgs {
  const double* X; const double* y; const int32_t* g; const double* w; const double* vec; const double* gh;
  const int32_t* gptr; double* W; int64_t ldw; double* klpart; double* gradpart; double* gsc; double* BR;
  double* bval; double* grampart; int64_t N; int K, G, Q; int64_t rows_per_q;   // rows per Q warp (multiple of 32)
};

// The bulk copies of a Q warp's first SLOTS stages (X rows, y, g, w: inputs no kernel of the chain writes),
// issued AHEAD of the kernel's programmatic-launch wait: they fly while k_prep finishes.
template <int SLOTS>
__device__ __forceinline__ void fused_q_issue_first(const FusedArgs& a, unsigned ring_u, unsigned full_u, int64_t gw) {
  const int lane = threadIdx.x & 31;
  const int K = a.K;
  const int64_t N = a.N;
  const int slot_elems = fused_slot_elems(K);
  const int64_t rs = gw * a.rows_per_q;
  const int64_t re = (rs + a.rows_per_q < N) ? rs + a.rows_per_q : N;
  const int nst = (rs < re) ? (int)((re - rs + kFuRows - 1) / kFuRows) : 0;
  const unsigned xbytes = (unsigned)(kFuRows * K * sizeof(double));
  const unsigned vbytes = (unsigned)(kFuRows * sizeof(double));
  const unsigned gbytes = (unsigned)(kFuRows * sizeof(int32_t));
  const unsigned nops = a.w ? 4u : 3u;
#pragma unroll
  for (int st = 0; st < SLOTS; ++st) {
    const int64_t n0 = rs + (int64_t)st * kFuRows;
    if (st < nst && n0 + kFuRows <= N && lane < (int)nops) {
      const unsigned bar = full_u + 8 * st;
      const unsigned dst = ring_u + (unsigned)(st * slot_elems * sizeof(double));
      if (lane == 0) {
        mbar_arrive_expect_tx(bar, xbytes + (a.w ? 2 : 1) * vbytes + gbytes);
        bulk_g2s(dst, a.X + n0 * K, xbytes, bar);
      } else if (lane == 1) {
        bulk_g2s(dst + xbytes, a.y + n0, vbytes, bar);
      } else if (lane == 2) {
        bulk_g2s(dst + xbytes + 2 * vbytes, a.g + n0, gbytes, bar);
      } else {
        bulk_g2s(dst + xbytes + vbytes, a.w + n0, vbytes, bar);
      }
    }
  }
}

// ---- the Q warp: k_obs_fused's stage loop on the team's ring ------------------------------------------
// (the first SLOTS stages were requested by fused_q_issue_first)
template <int NCH, int SLOTS>
__device__ __forceinline__ void fused_q_run(const FusedArgs& a, double* ring, unsigned ring_u, unsigned full_u,
                                            unsigned ready_u, unsigned empty_u, const double* bm, const double* bv,
                                            const double* ghc, const double* ghw, double* gred_row, double* kred_slot,
                                            int64_t gw) {
  constexpr int kFuStages = SLOTS;
  const int lane = threadIdx.x & 31;
  const int K = a.K, G = a.G, Q = a.Q;
  const int64_t N = a.N, ldw = a.ldw;
  const double* __restrict__ X = a.X;
  const double* __restrict__ y = a.y;
  const int32_t* __restrict__ g = a.g;
  const double* __restrict__ w = a.w;
  const double* __restrict__ vec = a.vec;
  const int32_t* __restrict__ gptr = a.gptr;
  double* __restrict__ W = a.W;
  const int slot_elems = fused_slot_elems(K);
  const int64_t um0 = 4 + 2 * (int64_t)K, ui0 = um0 + G;
  const int64_t rs = gw * a.rows_per_q;
  const int64_t re = (rs + a.rows_per_q < N) ? rs + a.rows_per_q : N;
  const int nst = (rs < re) ? (int)((re - rs + kFuRows - 1) / kFuRows) : 0;
  const unsigned xbytes = (unsigned)(kFuRows * K * sizeof(double));
  const unsigned vbytes = (unsigned)(kFuRows * sizeof(double));
  const unsigned gbytes = (unsigned)(kFuRows * sizeof(int32_t));
  const unsigned nops = w ? 4u : 3u;

  auto issue = [&](int st, int slot) {
    const int64_t n0 = rs + (int64_t)st * kFuRows;
    if (st < nst && n0 + kFuRows <= N && lane < (int)nops) {
      const unsigned bar = full_u + 8 * slot;
      const unsigned dst = ring_u + (unsigned)(slot * slot_elems * sizeof(double));
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

  int gcd16 = 1;
  while (gcd16 < 16 && (K % (gcd16 * 2)) == 0) gcd16 *= 2;
  int skew = ((lane & 15) * gcd16) >> 4;
  if (skew >= K) skew = 0;

  double gm[NCH], gv[NCH];
  double q0[NCH], q1[NCH], q2[NCH], q3[NCH], q4[NCH], q5[NCH];
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
    if (gb >= rs && ge <= re) {
      dbr = a.BR + (size_t)cur_g * 4 * K;
      dsc = a.gsc + (size_t)cur_g * 5;
    } else {
      double* rec = a.bval + ((size_t)gw * 2 + (gb < rs ? 0 : 1)) * nb;
      dsc = rec;
      dbr = rec + 5;
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int k = lane + 32 * c;
      if (k < K) {
        dbr[k] = q2[c];
        dbr[K + k] = q3[c];
        dbr[2 * K + k] = q4[c];
        dbr[3 * K + k] = q5[c];
        gm[c] += q0[c];
        gv[c] += q1[c];
      } else if (k == K) {
        dsc[0] = q0[c];
        dsc[1] = q1[c];
        dsc[2] = q2[c];
        dsc[3] = q3[c];
        dsc[4] = q5[c];
      }
      q0[c] = q1[c] = q2[c] = q3[c] = q4[c] = q5[c] = 0.0;
    }
  };

  int slot = 0, pslot = 0;
  unsigned phase = 0, pphase = 0;
  for (int st = 0; st < nst; ++st) {
    const int64_t n0 = rs + (int64_t)st * kFuRows;
    double* xs = ring + (size_t)slot * slot_elems;
    double* ys = xs + kFuRows * K;
    const int32_t* gs = reinterpret_cast<const int32_t*>(ys + 2 * kFuRows);
    double* wq = ys + 2 * kFuRows + kFuRows / 2;
    const int rows = (int)((re - n0 < kFuRows) ? (re - n0) : kFuRows);
    if (n0 + kFuRows <= N) {
      mbar_wait(full_u + 8 * slot, phase);
    } else {
      // ragged last stage of the data set: filled by the warp itself (zero rows beyond N), then the
      // full barrier is completed by hand so that the D warps see the same protocol
      if (st >= kFuStages) mbar_wait(empty_u + 8 * slot, phase ^ 1u);
      const int vr = (int)(N - n0);
      for (int e = lane; e < kFuRows * K; e += 32) xs[e] = (e < vr * K) ? X[n0 * K + e] : 0.0;
      ys[lane] = (lane < vr) ? y[n0 + lane] : 0.0;
      ys[kFuRows + lane] = (lane < vr && w) ? w[n0 + lane] : 0.0;
      reinterpret_cast<int32_t*>(ys + 2 * kFuRows)[lane] = (lane < vr) ? g[n0 + lane] : -1;
      __syncwarp();
      if (lane == 0) mbar_arrive(full_u + 8 * slot);
      mbar_wait(full_u + 8 * slot, phase);
    }

    // ---- phase A: lane = observation ----
    unsigned segmask;
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
      gh_all_nodes_f<2, kFuUnroll>(zm, zs, ghc, ghw, Q, s);
      const double wn = valid ? (w ? ys[kFuRows + lane] : 1.0) : 0.0;
      const double yn = ys[lane];
      klacc += wn * (yn * zm - s.A);
      const double h = 0.5 / zs;
      const double lm = wn * (yn - s.Am);
      const double lv = -wn * s.As * h;
      const double wa = -wn * s.Amm;
      const double wb = -wn * s.Ams * h;
      const double wc = -wn * (s.Ass - s.As / zs) / (4.0 * zv);
      double2* wrow = reinterpret_cast<double2*>(wq + 6 * lane);
      wrow[0] = make_double2(lm, lv);
      wrow[1] = make_double2(wa, wb);
      wrow[2] = make_double2(wc, 0.0);
      if (valid && W) {
        W[n] = lm;
        W[ldw + n] = lv;
        W[2 * ldw + n] = wa;
        W[3 * ldw + n] = wb;
        W[4 * ldw + n] = wc;
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(ready_u + 8 * slot);     // release: the D warps may consume the stage
    // the slot of the previous stage: refill it as soon as the D warps have released it (polled here,
    // waited for at the end of the stage) so that the copy overlaps the group sums
    bool refill = (st > 0) && (st - 1 + kFuStages < nst);
    if (refill && mbar_test(empty_u + 8 * pslot, pphase)) {
      issue(st - 1 + kFuStages, pslot);
      refill = false;
    }

    // ---- phase C: lane = column; per-group running sums ----
    {
      const double2* w2 = reinterpret_cast<const double2*>(wq);
      int koff[NCH];
      bool isone[NCH];
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int k = lane + 32 * c;
        koff[c] = (k < K) ? k : 0;
        isone[c] = (k == K);
      }
      auto rows_acc = [&](int r, auto nrow) {
        constexpr int NR = decltype(nrow)::value;
        double2 wl[NR], wab[NR], wc[NR];
        double x[NR][NCH];
#pragma unroll
        for (int u = 0; u < NR; ++u) {
          wl[u] = w2[3 * (r + u)];
          wab[u] = w2[3 * (r + u) + 1];
          wc[u] = w2[3 * (r + u) + 2];
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
            t2 = fma(wab[u].x, xv, t2);
            t3 = fma(wab[u].y, xv, t3);
            t4 = fma(wab[u].y, xx, t4);
            t5 = fma(wc[u].x, xx, t5);
          }
          q0[c] += t0; q1[c] += t1; q2[c] += t2; q3[c] += t3; q4[c] += t4; q5[c] += t5;
        }
      };
      int r = 0;
      const unsigned m = segmask;
      while (r < rows) {
        if ((m >> r) & 1u) {
          flush();
          cur_g = gs[r];
        }
        const unsigned rest = (r + 1 < 32) ? (m >> (r + 1)) : 0u;
        const int nxt = rest ? (r + 1 + __ffs((int)rest) - 1) : rows;
        const int r1 = nxt < rows ? nxt : rows;
        for (; r + 4 <= r1; r += 4) rows_acc(r, std::integral_constant<int, 4>());
        for (; r < r1; ++r) rows_acc(r, std::integral_constant<int, 1>());
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty_u + 8 * slot);     // the Q warp's share of the slot's release
    // refill the slot of the PREVIOUS stage once the D warps have released it too: the Q warp may run
    // a stage ahead of its D warps instead of meeting them at every stage
    if (refill) {
      mbar_wait(empty_u + 8 * pslot, pphase);
      issue(st - 1 + kFuStages, pslot);
    }
    pslot = slot;
    pphase = phase;
    if (++slot == kFuStages) { slot = 0; phase ^= 1u; }
  }
  flush();

  klacc = warp_sum(klacc);
  if (lane == 0) *kred_slot = klacc;
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const int k = lane + 32 * c;
    if (k < K) {
      gred_row[k] = gm[c];
      gred_row[K + k] = gv[c];
    }
  }
}

// ---- a D warp: k_gram_mid's k-step on the 32-row stages of the team's NQ rings, round-robin ----------------
template <int T2, int T0, bool HAS_M, int P, int TLO, int THI, int NQ, int SLOTS, int TEAMS>
__device__ __forceinline__ void fused_d_run(const FusedArgs& a, unsigned sm_u, unsigned bars_u, int team,
                                            double (&acc)[THI - TLO][2]) {
  constexpr int TS = HAS_M ? T0 : -1;
  constexpr int TB = HAS_M ? T0 + 1 : T0;
  constexpr int JLO = gram_mid_col(TLO), JHI = gram_mid_col(THI - 1) + 1;
  constexpr int T_LO = TLO;
  auto mine = [](int i, int j) constexpr { return j * (j + 1) / 2 + i >= TLO && j * (j + 1) / 2 + i < THI; };
  constexpr int KSTEPS = kFuRows / 4;
  const int K = a.K;
  const int lane = threadIdx.x & 31;
  const int lr = lane & 3, lc = lane >> 2;
  const int slot_elems = fused_slot_elems(K);

  const int base = lr * K + lc;
  bool cls1 = false, valid_m = true, valid_last = true;
  int off_m = 0, off_last = 0;
  if (HAS_M) {
    const int col = 8 * TS + lc;
    cls1 = col >= K;
    valid_m = col < 2 * K;
    off_m = lr * K + (valid_m ? (cls1 ? col - K : col) : 0);
  }
  {
    const int col = 8 * (T2 - 1) + lc;
    valid_last = col < 2 * K;
    off_last = lr * K + (valid_last ? col - K : 0);
  }

  // Q warp qi of this team is CTA-local Q warp qi * TEAMS + team; its rows: [gq * rows_per_q, ...)
  int nst_q[NQ];
  int max_nst = 0;
#pragma unroll
  for (int qi = 0; qi < NQ; ++qi) {
    const int64_t gq = (int64_t)blockIdx.x * (TEAMS * NQ) + qi * TEAMS + team;
    const int64_t rs = gq * a.rows_per_q;
    const int64_t re = (rs + a.rows_per_q < a.N) ? rs + a.rows_per_q : a.N;
    nst_q[qi] = (rs < re) ? (int)((re - rs + kFuRows - 1) / kFuRows) : 0;
    max_nst = nst_q[qi] > max_nst ? nst_q[qi] : max_nst;
  }

  int slot = 0;
  unsigned phase = 0;
  for (int st = 0; st < max_nst; ++st) {
#pragma unroll 1
    for (int qi = 0; qi < NQ; ++qi) {
      if (st >= nst_q[qi]) continue;
      const int ql = qi * TEAMS + team;
      const unsigned full_u = bars_u + 8u * (unsigned)(ql * SLOTS * 3);
      const unsigned ready_u = full_u + 8 * SLOTS, empty_u = full_u + 16 * SLOTS;
      mbar_wait(ready_u + 8 * slot, phase);      // weights written (the Q warp saw the TMA data first)
      mbar_wait(full_u + 8 * slot, phase);       // and this warp observes the bulk copies itself
      const unsigned xs_u = sm_u + 8u * (unsigned)((ql * SLOTS + slot) * slot_elems);
      const unsigned wq_u = xs_u + 8u * (unsigned)(kFuRows * K + 2 * kFuRows + kFuRows / 2 + 6 * lr);
#pragma unroll 1
      for (int ks = 0; ks < KSTEPS; ++ks) {
        const unsigned row_u = xs_u + 8u * (unsigned)(4 * ks * K);
        double z[JHI];
#pragma unroll
        for (int t = 0; t < JHI; ++t) {
          int o;
          if (t == TS) o = off_m;
          else if (t == T2 - 1 && t >= TB) o = off_last;
          else o = base + ((t < T0) ? 8 * t : 8 * t - K);
          z[t] = lds_f64(row_u + 8u * (unsigned)o);
        }
        const unsigned wrow_u = wq_u + 8u * (unsigned)(24 * ks);     // row 4 ks + lr, 6 doubles per row
        const double wa = lds_f64(wrow_u + 16u);
        const double wb = lds_f64(wrow_u + 24u);
        const double wc = lds_f64(wrow_u + 32u);
#pragma unroll
        for (int t = 0; t < JHI; ++t) {
          if (t == TS) {
            const double xx = vmul(z[t], z[t]);
            z[t] = cls1 ? xx : z[t];
            if (!valid_m) z[t] = 0.0;
          } else if (t >= TB) {
            z[t] = vmul(z[t], z[t]);
            if (t == T2 - 1 && !valid_last) z[t] = 0.0;
          }
        }
        double aw2 = 0.0;
        if (HAS_M && JHI > TS) aw2 = vmul(z[(HAS_M && JHI > TS) ? TS : 0], cls1 ? wc : wb);
#pragma unroll
        for (int j = JLO; j < JHI; ++j) {
          const int cb = j * (j + 1) / 2 - T_LO;
          bool need0 = (HAS_M && j == TS && mine(j, j)), needc = false;
#pragma unroll
          for (int i = 0; i < T0; ++i)
            if (i <= j && mine(i, j)) need0 = true;
#pragma unroll
          for (int i = TB; i < T2; ++i)
            if (i <= j && mine(i, j)) needc = true;
          double bw0 = 0.0, bc = 0.0;
          if (need0) bw0 = vmul(z[j], (j < T0) ? wa : ((j == TS) ? (cls1 ? wb : wa) : wb));
          if (needc) bc = vmul(z[j], wc);
#pragma unroll
          for (int i = 0; i < T0; ++i)
            if (i <= j && mine(i, j)) dmma884(acc[cb + i][0], acc[cb + i][1], z[i], bw0);
          if (HAS_M && j == TS && mine(j, j)) {
            dmma884(acc[cb + j][0], acc[cb + j][1], cls1 ? 0.0 : z[j], bw0);
            dmma884(acc[cb + j][0], acc[cb + j][1], cls1 ? z[j] : 0.0, aw2);
          }
          if (HAS_M && j > TS && mine(HAS_M ? TS : 0, j))
            dmma884(acc[cb + (HAS_M ? TS : 0)][0], acc[cb + (HAS_M ? TS : 0)][1], aw2, z[j]);
#pragma unroll
          for (int i = TB; i < T2; ++i)
            if (i <= j && mine(i, j)) dmma884(acc[cb + i][0], acc[cb + i][1], z[i], bc);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(empty_u + 8 * slot);
    }
    if (++slot == SLOTS) { slot = 0; phase ^= 1u; }
  }
}

template <int T2, int T0, bool HAS_M, int P, int R, int NQ, int SLOTS, int TEAMS>
__device__ __forceinline__ void fused_d_dispatch(int role, const FusedArgs& a, unsigned sm_u, unsigned bars_u, int team,
                                                 double* red, int warp, int nwarps) {
  if constexpr (R < P) {
    if (role == R) {
      constexpr int LO = gram_mid_bound(T2, T0, HAS_M, P, R), HI = gram_mid_bound(T2, T0, HAS_M, P, R + 1);
      double acc[HI - LO][2];
#pragma unroll
      for (int t = 0; t < HI - LO; ++t) acc[t][0] = acc[t][1] = 0.0;
      fused_d_run<T2, T0, HAS_M, P, LO, HI, NQ, SLOTS, TEAMS>(a, sm_u, bars_u, team, acc);
      // every warp of the CTA is done with the rings: they become the (NT, 64) tile buffer; the D warps
      // add their accumulators one after the other (fixed order)
      __syncthreads();
      for (int e = threadIdx.x; e < (T2 * (T2 + 1) / 2) * 64; e += blockDim.x) red[e] = 0.0;
      __syncthreads();
      const int lane = threadIdx.x & 31;
      const int e0 = (lane >> 2) * 8 + 2 * (lane & 3);
#pragma unroll 1
      for (int w = 0; w < nwarps; ++w) {
        if (warp == w) {
#pragma unroll
          for (int t = 0; t < HI - LO; ++t) {
            double* d = red + (size_t)(LO + t) * 64 + e0;
            d[0] += acc[t][0];
            d[1] += acc[t][1];
          }
        }
        __syncthreads();
      }
    } else {
      fused_d_dispatch<T2, T0, HAS_M, P, R + 1, NQ, SLOTS, TEAMS>(role, a, sm_u, bars_u, team, red, warp, nwarps);
    }
  }
}

// warps [0, TEAMS * NQ): Q warp ql = qi * TEAMS + team;  then D warp dw = warp - TEAMS * NQ: team dw % TEAMS,
// role dw / TEAMS (with TEAMS = 4 a team's warps share one SM sub-partition)
template <int T2, int T0, bool HAS_M, int NCH, int TEAMS, int NQ, int P, int WARPS, int SLOTS>
__global__ void __launch_bounds__(32 * WARPS, 1)
k_fused_eval(const FusedArgs a) {
  pdl_launch_dependents();
  constexpr int NT = T2 * (T2 + 1) / 2;
  constexpr int NQW = TEAMS * NQ;
  extern __shared__ __align__(16) double sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int K = a.K, Q = a.Q;
  const int slot_elems = fused_slot_elems(K);
  const size_t ring_elems = (size_t)NQW * SLOTS * slot_elems;
  const size_t red_elems = (size_t)NT * 64;
  double* tail = sm + (ring_elems > red_elems ? ring_elems : red_elems);
  double* bm = tail;                              // K   E[beta]
  double* bv = bm + K;                            // K   Var[beta]
  double* ghc = bv + K;                           // Q
  double* ghw = ghc + Q;                          // Q
  double* gred = ghw + Q;                         // NQW x 2K
  double* kred = gred + (size_t)NQW * 2 * K;      // NQW
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(kred + NQW);
  const unsigned sm_u = smem_u32(sm), bars_u = smem_u32(bars);

  const bool is_q = warp < NQW;
  const int dw = warp - NQW;
  const int team = is_q ? warp % TEAMS : dw % TEAMS;
  const int role = is_q ? -1 : dw / TEAMS;
  const bool active = is_q || role < P;

  // ahead of the wait for k_prep: barriers and the first stages of every Q warp's ring (static inputs only)
  if (is_q) {
    const unsigned full_u = bars_u + 8u * (unsigned)(warp * SLOTS * 3);
    if (lane == 0) {
#pragma unroll
      for (int p = 0; p < SLOTS; ++p) {
        mbar_init(full_u + 8 * p, 1);
        mbar_init(full_u + 8 * SLOTS + 8 * p, 1);
        mbar_init(full_u + 16 * SLOTS + 8 * p, 1 + P);
      }
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncwarp();
    fused_q_issue_first<SLOTS>(a, smem_u32(sm + (size_t)warp * SLOTS * slot_elems), full_u,
                               (int64_t)blockIdx.x * NQW + warp);
  }
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    ghc[q] = a.gh[q];
    ghw[q] = a.gh[Q + q];
  }
  pdl_wait();
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    bm[k] = a.vec[4 + k];
    bv[k] = 1.0 / a.vec[4 + K + k];
  }
  __syncthreads();

  double* red = sm;
  if (is_q) {
    double* ring = sm + (size_t)warp * SLOTS * slot_elems;
    const unsigned full_u = bars_u + 8u * (unsigned)(warp * SLOTS * 3);
    const int64_t gq = (int64_t)blockIdx.x * NQW + warp;
    fused_q_run<NCH, SLOTS>(a, ring, smem_u32(ring), full_u, full_u + 8 * SLOTS, full_u + 16 * SLOTS, bm, bv, ghc, ghw,
                            gred + (size_t)warp * 2 * K, kred + warp, gq);
    // meet the D warps at the barriers of their reduction (the same number on every path)
    __syncthreads();
    for (int e = threadIdx.x; e < NT * 64; e += blockDim.x) red[e] = 0.0;
    __syncthreads();
#pragma unroll 1
    for (int w = 0; w < WARPS; ++w) __syncthreads();
  } else if (active) {
    fused_d_dispatch<T2, T0, HAS_M, P, 0, NQ, SLOTS, TEAMS>(role, a, sm_u, bars_u, team, red, warp, WARPS);
  } else {
    __syncthreads();
    for (int e = threadIdx.x; e < NT * 64; e += blockDim.x) red[e] = 0.0;
    __syncthreads();
#pragma unroll 1
    for (int w = 0; w < WARPS; ++w) __syncthreads();
  }
  // ---- CTA outputs: Gram tiles, KL partial, global-gradient partials (fixed order) ----
  double* out = a.grampart + (size_t)blockIdx.x * NT * 64;
  for (int e = threadIdx.x; e < NT * 64; e += blockDim.x) out[e] = red[e];
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < NQW; ++i) s += kred[i];
    a.klpart[blockIdx.x] = s;
  }
  for (int k = threadIdx.x; k < 2 * K; k += blockDim.x) {
    double s = 0.0;
    for (int i = 0; i < NQW; ++i) s += gred[(size_t)i * 2 * K + k];
    a.gradpart[(size_t)k * gridDim.x + blockIdx.x] = s;
  }
}

// the instantiation for K (K <= kFuMaxK), launched with 32 * kFuGeom.warps threads and fused_smem bytes; null
// outside that range
inline auto fused_eval_kernel(int K) -> void (*)(FusedArgs) {
  const int T2 = (2 * K + 7) / 8, T0 = K / 8;
  const bool M = (K % 8) != 0;
  const int nch = obs_fused_chunks(K);
#define LRVB_FU(T2_, T0_, M_, NCH_)                                                                  \
  if (T2 == T2_ && T0 == T0_ && M == M_ && nch == NCH_) {                                            \
    return k_fused_eval<T2_, T0_, M_, NCH_, kFuGeom.teams, kFuGeom.NQ, kFuGeom.P, kFuGeom.warps,       \
                        kFuGeom.slots>;                                                              \
  }
  LRVB_FU(1, 0, true, 1)
  LRVB_FU(2, 0, true, 1)
  LRVB_FU(2, 1, false, 1)
  LRVB_FU(3, 1, true, 1)
  LRVB_FU(4, 1, true, 1)
  LRVB_FU(4, 2, false, 1)
  LRVB_FU(5, 2, true, 1)
  LRVB_FU(6, 2, true, 1)
  LRVB_FU(6, 3, false, 1)
#undef LRVB_FU
  return nullptr;
}

}  // namespace lrvb
