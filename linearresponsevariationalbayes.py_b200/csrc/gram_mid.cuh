// Weighted Grams of the beta block for 25 <= K <= 104 on the FP64 tensor cores (DMMA.8x8x4), sm_100a.
//
// Same packed formulation as gram_small.cuh (ONE weighted Gram of z = [x | s], upper triangle of
// the T2 x T2 tile grid, tile classes pure-x / straddle / pure-s) and the same execution model:
// the WHOLE TRIANGLE is owned, for a set of rows, by one warp -- or by a TEAM of 2 / 4 / 8 warps when
// its NT = T2 (T2 + 1) / 2 accumulator tiles do not fit the registers of one (2 registers per tile and
// thread; 255 registers per thread at 8 warps per SM).  A team streams its own 16- / 32-row stages (gram_mid_rows)
// through a private shared-memory ring filled by bulk async copies, and all teams of all CTAs do identical
// work, so the four FP64 pipes of an SM are evenly loaded -- which the rectangle jobs of gram_big.cuh
// never quite achieve (0.29 - 0.63 of the DMMA peak on the same sizes, 0.73 - 0.85 here).
//   * Roles: the tiles in column-major order are cut into P contiguous ranges of equal DMMA count
//     (gram_mid_bound); role r of a team is a separate instantiation with compile-time tile indices.
//     The fewer warps per team the better (a k-step's operand fetch is amortised over more DMMAs):
//     P = 1 up to T2 = 8, 2 up to 13, 4 up to 20, 8 up to 26.
//   * Ring: full / empty mbarriers per slot; role 0 issues the copies and refills a slot one stage late,
//     so it may run a stage ahead of its partners instead of meeting them at every stage.
//   * No register prefetch of the next k-step: a k-step is 16 - 46 independent DMMAs per warp, the other
//     warps of the sub-partition cover the operand fetch.  B operands are weighted per column tile right
//     before its DMMAs; the per-lane offsets of the packed columns are compile-time constants plus one base.
//   * The CTA's warps add their accumulators into one shared tile set one after the other (fixed order).
// Output layout = gram_small's: part (gridDim.x, NT, 64), tile (i <= j) at slot j (j+1)/2 + i.
#pragma once
#include "common.cuh"
#include "gram_small.cuh"   // mbarrier / bulk-copy / lds / vmul helpers

namespace lrvb {

// rows per stage: 32 (8 k-steps between two ring hand-overs) wherever three slots of them fit beside the
// other teams' rings -- from T2 = 9 on (<= 6 teams per CTA); measured 0.7 - 3.5 % faster than 16 for K = 36 .. 104
// (K = 50: 3.680 -> 3.654 ms at N = 10M); the 12 single-warp teams of T2 <= 8 stay at 16 rows
__host__ __device__ constexpr int gram_mid_rows(int T2) { return T2 >= 9 ? 32 : 16; }
constexpr int kGmStages = 3;      // ring depth per team
constexpr int kGmMaxK = 104;      // T2 = ceil(2K / 8) <= 26

// launch geometry by tile-grid size: T2 <= 8 leaves room for 12 single-warp teams at 168 registers;
// 9 and 10 need the 255-register budget (8 warps); from 11 on the triangle is split between the two
// warps of a team (8 warps = 4 teams)
struct GramMidGeom {
  int warps, P;
};
// T2 <= 8: 12 single-warp teams at <= 168 registers; 9..13: pairs of warps; 14..20: teams of four;
// 21..26: one team of eight (8 warps x 255 registers from T2 = 11 on).  Fewer, larger roles amortise the
// operand fetch of a k-step over more DMMAs: as few warps per team as the 255-register budget allows
__host__ __device__ constexpr GramMidGeom gram_mid_geom(int T2) {
  return T2 <= 8 ? GramMidGeom{12, 1}
       : T2 <= 10 ? GramMidGeom{12, 2}
       : T2 <= 13 ? GramMidGeom{8, 2}
       : T2 <= 20 ? GramMidGeom{8, 4} : GramMidGeom{8, 8};
}
// Tiles of the packed upper triangle in column-major order: t(i, j) = j (j + 1) / 2 + i, i <= j.  Role r
// of a P-warp team owns the tiles [bound(r), bound(r + 1)): equal DMMA counts (the diagonal straddle
// tile costs two).
__host__ __device__ constexpr int gram_mid_col(int t) {
  int j = 0;
  while ((j + 1) * (j + 2) / 2 <= t) ++j;
  return j;
}
__host__ __device__ constexpr int gram_mid_bound(int T2, int T0, bool has_m, int P, int r) {
  const int NT = T2 * (T2 + 1) / 2;
  if (r <= 0) return 0;
  if (r >= P) return NT;
  const int ts = has_m ? T0 * (T0 + 1) / 2 + T0 : -1;      // the straddle diagonal tile
  const int total = NT + (has_m ? 1 : 0);
  const int want = (int)(((long long)total * r + P / 2) / P);
  int acc = 0;
  for (int t = 0; t < NT; ++t) {
    if (acc >= want) return t;
    acc += (t == ts) ? 2 : 1;
  }
  return NT;
}
__host__ __device__ inline size_t gram_mid_stage_elems(int K, int T2) {
  return (size_t)gram_mid_rows(T2) * K + 3 * gram_mid_rows(T2);
}
inline size_t gram_mid_smem(int K, int T2) {
  const GramMidGeom g = gram_mid_geom(T2);
  const int teams = g.warps / g.P;
  const size_t ring = sizeof(double) * teams * kGmStages * gram_mid_stage_elems(K, T2) +
                      sizeof(unsigned long long) * teams * kGmStages * 2;
  const size_t red = sizeof(double) * (size_t)(T2 * (T2 + 1) / 2) * 64;
  return ring > red ? ring : red;
}

// The stream of one warp: column tiles [JLO, JHI) of the packed upper triangle over the stages of
// its team.  PRODUCER issues the bulk copies (the first warp of a team).
template <int T2, int T0, bool HAS_M, int P, int TLO, int THI, bool PRODUCER>
__device__ __forceinline__ void gram_mid_run(const double* __restrict__ X, const double* __restrict__ Wabc,
                                             double* __restrict__ red, int64_t N, int64_t ldw, int K,
                                             unsigned ring_u, unsigned full_u, unsigned empty_u, double* ring,
                                             int gt, int tt, int warp, int nwarps) {
  constexpr int TS = HAS_M ? T0 : -1;        // straddle tile
  constexpr int TB = HAS_M ? T0 + 1 : T0;    // first pure-s tile
  constexpr int JLO = gram_mid_col(TLO), JHI = gram_mid_col(THI - 1) + 1;   // column tiles touched
  constexpr int T_LO = TLO;
  constexpr int NTL = THI - TLO;                       // accumulator tiles of this warp
  auto mine = [](int i, int j) constexpr { return j * (j + 1) / 2 + i >= TLO && j * (j + 1) / 2 + i < THI; };
  constexpr int ROWS = gram_mid_rows(T2);
  constexpr int KSTEPS = ROWS / 4;
  const int lane = threadIdx.x & 31;
  const int lr = lane & 3, lc = lane >> 2;
  const int stage_elems = ROWS * K + 3 * ROWS;

  // packed column `col = 8 t + lc` of tile t sits at x column `col` (x class) or `col - K` (s class)
  // of the staged row: compile-time per tile except in the straddle tile and beyond 2K in the last
  const int base = lr * K + lc;                                   // + 8 t (x tiles), + 8 t - K (s tiles)
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

  double acc[NTL][2];
#pragma unroll
  for (int t = 0; t < NTL; ++t) acc[t][0] = acc[t][1] = 0.0;

  // 32-bit stage counters (N < 2^35): registers are the scarce resource of this kernel
  const int nstage = (int)((N + ROWS - 1) / ROWS);
  const int nfull = (int)(N / ROWS);
  const unsigned xbytes = (unsigned)(ROWS * K * sizeof(double));
  const unsigned wbytes = (unsigned)(ROWS * sizeof(double));

  auto issue = [&](int s, int slot) {
    if (s < nfull && lane < 4) {
      const unsigned bar = full_u + 8 * slot;
      const unsigned dst = ring_u + (unsigned)(slot * stage_elems * sizeof(double));
      const int64_t n0 = (int64_t)s * ROWS;
      if (lane == 0) {
        mbar_arrive_expect_tx(bar, xbytes + 3 * wbytes);
        bulk_g2s(dst, X + n0 * K, xbytes, bar);
      } else {
        bulk_g2s(dst + xbytes + (lane - 1) * wbytes, Wabc + (int64_t)(lane - 1) * ldw + n0, wbytes, bar);
      }
    }
  };

  if (PRODUCER) {
#pragma unroll
    for (int p = 0; p < kGmStages; ++p) issue(gt + p * tt, p);
  }

  int slot = 0, pslot = 0;
  unsigned phase = 0, pphase = 0;
  bool first = true;
  for (int s = gt; s < nstage; s += tt) {
    // ---- make the stage readable ----
    if (s < nfull) {
      mbar_wait(full_u + 8 * slot, phase);
    } else if (PRODUCER) {   // ragged last stage: filled by the producer warp itself, zero rows beyond N
      if (P > 1 && (s - gt) / tt >= kGmStages) mbar_wait(empty_u + 8 * slot, phase ^ 1u);   // previous use released
      double* xs = ring + (size_t)slot * stage_elems;
      double* ws = xs + ROWS * K;
      const int64_t n0 = (int64_t)s * ROWS;
      const int rows = (int)(N - n0);
      for (int e = lane; e < ROWS * K; e += 32) xs[e] = (e < rows * K) ? X[n0 * K + e] : 0.0;
      for (int e = lane; e < 3 * ROWS; e += 32) {
        const int f = e / ROWS, r = e % ROWS;
        ws[e] = (r < rows) ? Wabc[(int64_t)f * ldw + n0 + r] : 0.0;
      }
      __syncwarp();
      if (P > 1 && lane == 0) mbar_arrive(full_u + 8 * slot);
    } else {
      mbar_wait(full_u + 8 * slot, phase);
    }
    const unsigned xs_u = ring_u + (unsigned)(slot * stage_elems * sizeof(double));
    const unsigned ws_u = xs_u + 8u * (unsigned)(ROWS * K + lr);
#pragma unroll 1
    for (int ks = 0; ks < KSTEPS; ++ks) {
      const unsigned row_u = xs_u + 8u * (unsigned)(4 * ks * K);
      double z[JHI];                     // row tiles 0 .. JHI-1 are all this warp ever multiplies
#pragma unroll
      for (int t = 0; t < JHI; ++t) {
        int o;
        if (t == TS) o = off_m;
        else if (t == T2 - 1 && t >= TB) o = off_last;
        else o = base + ((t < T0) ? 8 * t : 8 * t - K);
        z[t] = lds_f64(row_u + 8u * (unsigned)o);
      }
      const double wa = lds_f64(ws_u + 8u * (unsigned)(4 * ks));
      const double wb = lds_f64(ws_u + 8u * (unsigned)(ROWS + 4 * ks));
      const double wc = lds_f64(ws_u + 8u * (unsigned)(2 * ROWS + 4 * ks));
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
        // B operands of column tile j: x rows see (a | b), s rows see c -- formed only when this
        // warp owns such a tile of the column (the conditions fold at compile time)
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
          dmma884(acc[cb + j][0], acc[cb + j][1], cls1 ? 0.0 : z[j], bw0);   // x rows of the tile
          dmma884(acc[cb + j][0], acc[cb + j][1], cls1 ? z[j] : 0.0, aw2);   // s rows of the tile
        }
        if (HAS_M && j > TS && mine(HAS_M ? TS : 0, j))
          dmma884(acc[cb + (HAS_M ? TS : 0)][0], acc[cb + (HAS_M ? TS : 0)][1], aw2, z[j]);
#pragma unroll
        for (int i = TB; i < T2; ++i)
          if (i <= j && mine(i, j)) dmma884(acc[cb + i][0], acc[cb + i][1], z[i], bc);
      }
    }
    __syncwarp();            // every lane has read its last operands of this slot
    if (P == 1) {
      issue(s + kGmStages * tt, slot);
    } else {
      if (lane == 0) mbar_arrive(empty_u + 8 * slot);
      if (PRODUCER) {
        // refill the slot of the PREVIOUS stage once both warps of the team have released it: the
        // producer may run one stage ahead of its partner instead of meeting it at every stage
        if (!first) {
          mbar_wait(empty_u + 8 * pslot, pphase);
          issue(s - tt + kGmStages * tt, pslot);
        }
        pslot = slot;
        pphase = phase;
        first = false;
      }
    }
    if (++slot == kGmStages) { slot = 0; phase ^= 1u; }
  }
  __syncthreads();           // every warp of the CTA is done with the rings: they become the tile buffer
  for (int e = threadIdx.x; e < (T2 * (T2 + 1) / 2) * 64; e += blockDim.x) red[e] = 0.0;
  __syncthreads();

  // the warps add their accumulators into one tile set, one warp after the other (fixed order)
  const int e0 = (lane >> 2) * 8 + 2 * (lane & 3);
#pragma unroll 1
  for (int w = 0; w < nwarps; ++w) {
    if (warp == w) {
#pragma unroll
      for (int t = 0; t < NTL; ++t) {
        double* d = red + (size_t)(T_LO + t) * 64 + e0;
        d[0] += acc[t][0];
        d[1] += acc[t][1];
      }
    }
    __syncthreads();
  }
}

// role r of the team runs the instantiation for its tile range; role 0 is the producer
template <int T2, int T0, bool HAS_M, int P, int R>
__device__ __forceinline__ void gram_mid_dispatch(int role, const double* __restrict__ X,
                                                  const double* __restrict__ Wabc, double* __restrict__ red,
                                                  int64_t N, int64_t ldw, int K, unsigned ring_u, unsigned full_u,
                                                  unsigned empty_u, double* ring, int gt, int tt, int warp,
                                                  int nwarps) {
  if constexpr (R < P) {
    if (role == R) {
      constexpr int LO = gram_mid_bound(T2, T0, HAS_M, P, R), HI = gram_mid_bound(T2, T0, HAS_M, P, R + 1);
      gram_mid_run<T2, T0, HAS_M, P, LO, HI, R == 0>(X, Wabc, red, N, ldw, K, ring_u, full_u, empty_u, ring, gt,
                                                      tt, warp, nwarps);
    } else {
      gram_mid_dispatch<T2, T0, HAS_M, P, R + 1>(role, X, Wabc, red, N, ldw, K, ring_u, full_u, empty_u, ring, gt,
                                                 tt, warp, nwarps);
    }
  }
}

template <int T2, int T0, bool HAS_M, int WARPS, int P>
__global__ void __launch_bounds__(32 * WARPS, 1)
k_gram_mid(const double* __restrict__ X, const double* __restrict__ Wabc, double* __restrict__ part,
           int64_t N, int64_t ldw, int K) {
  pdl_sync();
  constexpr int NT = T2 * (T2 + 1) / 2;
  constexpr int TEAMS = WARPS / P;
  extern __shared__ __align__(16) double sm[];
  constexpr int ROWS = gram_mid_rows(T2);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int team = warp % TEAMS, role = warp / TEAMS;      // partners sit on the same sub-partition
  const int stage_elems = ROWS * K + 3 * ROWS;
  double* ring = sm + (size_t)team * kGmStages * stage_elems;
  unsigned long long* bars =
      reinterpret_cast<unsigned long long*>(sm + (size_t)TEAMS * kGmStages * stage_elems) + team * kGmStages * 2;
  const unsigned ring_u = smem_u32(ring), full_u = smem_u32(bars), empty_u = full_u + 8 * kGmStages;
  if (role == 0 && lane == 0) {
#pragma unroll
    for (int p = 0; p < kGmStages; ++p) {
      mbar_init(full_u + 8 * p, 1);
      mbar_init(empty_u + 8 * p, P);
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  __syncthreads();
  const int gt = (int)blockIdx.x * TEAMS + team, tt = (int)gridDim.x * TEAMS;
  double* red = sm;          // the rings are reused as the (NT, 64) tile buffer at the end
  gram_mid_dispatch<T2, T0, HAS_M, P, 0>(role, X, Wabc, red, N, ldw, K, ring_u, full_u, empty_u, ring, gt, tt, warp,
                                         WARPS);
  double* out = part + (size_t)blockIdx.x * NT * 64;
  for (int e = threadIdx.x; e < NT * 64; e += blockDim.x) out[e] = red[e];
}

// the instantiation for K (24 < K <= 104; below, the one-pass kernel of fused.cuh computes the Gram) and its CTA
// size in warps; a null kernel outside that range
struct GramMidKernel {
  void (*fn)(const double*, const double*, double*, int64_t, int64_t, int);
  int warps;
};
inline GramMidKernel gram_mid_kernel(int K) {
  const int T2 = (2 * K + 7) / 8, T0 = K / 8;
  const bool M = (K % 8) != 0;
#define LRVB_GM(T2_, T0_, M_)                                                                       \
  if (T2 == T2_ && T0 == T0_ && M == M_) {                                                          \
    constexpr GramMidGeom g = gram_mid_geom(T2_);                                                   \
    return {k_gram_mid<T2_, T0_, M_, g.warps, g.P>, g.warps};                                        \
  }
  LRVB_GM(7, 3, true)
  LRVB_GM(8, 3, true)
  LRVB_GM(8, 4, false)
  LRVB_GM(9, 4, true)
  LRVB_GM(10, 4, true)
  LRVB_GM(10, 5, false)
  LRVB_GM(11, 5, true)
  LRVB_GM(12, 5, true)
  LRVB_GM(12, 6, false)
  LRVB_GM(13, 6, true)
  LRVB_GM(14, 6, true)
  LRVB_GM(14, 7, false)
  LRVB_GM(15, 7, true)
  LRVB_GM(16, 7, true)
  LRVB_GM(16, 8, false)
  LRVB_GM(17, 8, true)
  LRVB_GM(18, 8, true)
  LRVB_GM(18, 9, false)
  LRVB_GM(19, 9, true)
  LRVB_GM(20, 9, true)
  LRVB_GM(20, 10, false)
  LRVB_GM(21, 10, true)
  LRVB_GM(22, 10, true)
  LRVB_GM(22, 11, false)
  LRVB_GM(23, 11, true)
  LRVB_GM(24, 11, true)
  LRVB_GM(24, 12, false)
  LRVB_GM(25, 12, true)
  LRVB_GM(26, 12, true)
  LRVB_GM(26, 13, false)
#undef LRVB_GM
  return {nullptr, 0};
}

}  // namespace lrvb
