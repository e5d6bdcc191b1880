// Weighted Grams of the beta block for K > 20 on the FP64 tensor cores (DMMA.8x8x4), sm_100a.
//
// Same packed formulation as gram_small.cuh: one weighted Gram of z_n = [x_n | s_n] (2K columns,
// T2 = ceil(2K/8) tiles) whose weight depends on the classes of the two columns, upper triangle
// only.  Here the triangle does not fit one warp's registers, so it is cut into warp jobs:
// rectangles of at most 4 x 4 tiles inside regions where one operand recipe holds
//   R0  x rows  x  all columns to the right    A = z_i                B = z_j * (a | b by column class)
//   R1  s rows  x  s columns to the right      A = z_i                B = z_j * c
//   R2  s rows  x  the straddle tile           A = z_i                B = z_j * (b | c)   (stored transposed)
//   R3  the straddle tile against itself       two DMMAs into one accumulator (as in gram_small)
// A CTA of 16 warps stages TN rows of X by bulk async copies (TMA, one piece per warp) into a
// two-slot ring and packs them once into Z = [x | x*x] rows with a bank-conflict-free stride (so
// no warp squares anything in the DMMA loop: the only FP64 work beside the DMMAs is one DMUL per B
// fragment and k-step); the packing of stage j+1 is done by the warps that finish stage j early,
// one block barrier per stage.  Every warp runs the job of its slot.  The host deals the jobs of a job group to the warps so that the
// four sub-partitions of the SM (warp % 4) carry the same number of DMMAs (longest-first); the
// unbalanced version this replaces kept the DMMA pipes 45 % busy.
#pragma once
#include <algorithm>
#include <vector>
#include "common.cuh"
#include "gram_small.cuh"   // mbarrier / bulk-copy helpers

namespace lrvb {

#ifndef LRVB_GB_WARPS
#define LRVB_GB_WARPS 16
#endif
constexpr int kGbWarps = LRVB_GB_WARPS;          // warps per CTA; 8 -> two CTAs per SM
constexpr int kGbCtasPerSM = (LRVB_GB_WARPS <= 8) ? 2 : 1;

struct GbJob {
  int kind;        // 0: rectangle, 1: straddle tile against itself
  int i0, j0;      // first A / B packed tile
  int ni, nj;      // rectangle size in tiles
  int stair;       // live iff i <= j (rectangles on the diagonal, i0 == j0)
  int w0, w1;      // weight row (0 a, 1 b, 2 c) applied to class-0 (x) / class-1 (s) B columns
  int transposed;  // output tile holds (B tile, A tile) entries: mirror into the upper triangle
  int ntiles;      // live tiles (for balancing)
  int group;       // job group (CTA column) that computes it
  int pad;
};
struct GbSlot {
  int job;         // -1: idle warp
  int split, nsplit;   // this warp takes k-steps split, split + nsplit, ...
  int pad;
};

struct GbPlan {
  std::vector<GbJob> jobs;
  std::vector<GbSlot> slots;   // n_groups x kGbWarps
  int n_groups = 0;
  int TN = 0;                  // rows per stage
  size_t smem = 0;
};

// shared memory: a ring of three stage buffers [Z rows | a b c], Z row = [x | s | 0] with stride
// ZS = 8 T2 + 4 (== 4 mod 8), which spreads the four rows a DMMA operand load touches over distinct
// bank groups; the x part of every row and the weights arrive by TMA, columns 2K .. ZS stay zero
constexpr int kGbBuffers = 3;
inline int gram_big_zs(int K) { return 8 * ((2 * K + 7) / 8) + 4; }
inline size_t gram_big_z_elems(int K, int TN) { return (size_t)TN * (gram_big_zs(K) + 3); }
inline size_t gram_big_smem(int K, int TN) {
  return sizeof(double) * kGbBuffers * gram_big_z_elems(K, TN) + 64;
}

inline GbPlan gram_big_plan(int K) {
  GbPlan pl;
  const int T2 = (2 * K + 7) / 8, T0 = K / 8;
  const bool has_m = (K % 8) != 0;
  const int TS = has_m ? T0 : -1, TB = has_m ? T0 + 1 : T0;
  auto add_rect = [&](int i0, int j0, int ni, int nj, int stair, int w0, int w1, int tr) {
    GbJob j = {0, i0, j0, ni, nj, stair, w0, w1, tr, 0, 0, 0};
    for (int a = 0; a < ni; ++a)
      for (int b = 0; b < nj; ++b)
        if (!stair || a <= b) ++j.ntiles;
    pl.jobs.push_back(j);
  };
  // R0: x rows [0, T0) against columns [i, T2), blocks aligned at multiples of 4
  for (int i0 = 0; i0 < T0; i0 += 4)
    for (int j0 = i0; j0 < T2; j0 += 4)
      add_rect(i0, j0, std::min(4, T0 - i0), std::min(4, T2 - j0), i0 == j0, 0, 1, 0);
  // R1: s rows [TB, T2) against s columns to the right, blocks aligned at TB
  for (int i0 = TB; i0 < T2; i0 += 4)
    for (int j0 = i0; j0 < T2; j0 += 4)
      add_rect(i0, j0, std::min(4, T2 - i0), std::min(4, T2 - j0), i0 == j0, 2, 2, 0);
  if (has_m) {
    // R2: s rows against the straddle tile (transposed), R3: the straddle tile against itself
    for (int i0 = TB; i0 < T2; i0 += 4) add_rect(i0, TS, std::min(4, T2 - i0), 1, 0, 1, 2, 1);
    GbJob j = {1, TS, TS, 1, 1, 0, 0, 0, 0, 2, 0, 0};
    pl.jobs.push_back(j);
  }
  // job groups of <= 16 jobs with (nearly) equal DMMA totals: longest-first, round robin
  const int J = (int)pl.jobs.size();
  pl.n_groups = (J + kGbWarps - 1) / kGbWarps;
  std::vector<int> order(J);
  for (int i = 0; i < J; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(),
                   [&](int a, int b) { return pl.jobs[a].ntiles > pl.jobs[b].ntiles; });
  std::vector<std::vector<int>> members(pl.n_groups);
  {
    std::vector<int> load(pl.n_groups, 0);
    for (int idx : order) {
      int best = -1;
      for (int g = 0; g < pl.n_groups; ++g)
        if ((int)members[g].size() < kGbWarps && (best < 0 || load[g] < load[best])) best = g;
      members[best].push_back(idx);
      load[best] += pl.jobs[idx].ntiles;
      pl.jobs[idx].group = best;
    }
  }
  // inside a group: k-split small groups to fill the 16 warps, then deal the (job, split) pairs to
  // the 4 sub-partitions longest-first (warp w runs on sub-partition w % 4)
  pl.slots.assign((size_t)pl.n_groups * kGbWarps, GbSlot{-1, 0, 1, 0});
  for (int g = 0; g < pl.n_groups; ++g) {
    const int nj = (int)members[g].size();
    // k-split factors: all jobs by the same factor when the group is small; then the largest
    // jobs once more while warps are free (finer grains balance better)
    std::vector<int> ns(nj, 1);
    int base = kGbWarps / nj;
    if (base > 4) base = 4;
    if (base < 1) base = 1;
    int slots_used = 0;
    for (int m = 0; m < nj; ++m) { ns[m] = base; slots_used += base; }
    for (int m = 0; m < nj && slots_used + ns[m] <= kGbWarps; ++m)   // members are sorted, largest first
      if (ns[m] * 2 <= 4 && pl.jobs[members[g][m]].ntiles > 8) { slots_used += ns[m]; ns[m] *= 2; }
    // longest-first over (job, split) pairs, load = tiles / nsplit (in 1/4 tiles)
    struct Item { int job, split, nsplit, load; };
    std::vector<Item> items;
    for (int m = 0; m < nj; ++m)
      for (int sp = 0; sp < ns[m]; ++sp)
        items.push_back(Item{members[g][m], sp, ns[m], 4 * pl.jobs[members[g][m]].ntiles / ns[m]});
    std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.load > b.load; });
    int load[4] = {0, 0, 0, 0}, used[4] = {0, 0, 0, 0};
    for (const Item& it : items) {
      int best = -1;
      for (int q = 0; q < 4; ++q)
        if (used[q] < kGbWarps / 4 && (best < 0 || load[q] < load[best])) best = q;
      const int warp = best + 4 * used[best];
      ++used[best];
      load[best] += it.load;
      pl.slots[(size_t)g * kGbWarps + warp] = GbSlot{it.job, it.split, it.nsplit, 0};
    }
  }
  // rows per stage: a multiple of 16 (k-split 4), everything in <= 200 KB
  int TN = 64;
  while (TN > 16 && gram_big_smem(K, TN) > (size_t)(200 / kGbCtasPerSM) * 1024) TN -= 16;
  pl.TN = TN;
  pl.smem = gram_big_smem(K, TN);
  return pl;
}

// ---- device side (compiled by the translation unit that defines LRVB_GRAM_BIG_KERNELS) ------
#ifdef LRVB_GRAM_BIG_KERNELS
struct GbLane {          // per-lane operand recipe of a rectangle job
  int offA[4], offB[4];  // packed column of each fragment inside a Z row (columns >= 2K are zero)
  unsigned selB;         // bit f: B fragment f is a class-1 (s) column -> weight w1
};

template <int NI, int NJ, bool STAIR>
__device__ __forceinline__ void gb_ksteps(double (&acc)[4][4][2], const double* st, const double* sw,
                                          const GbLane& L, int w0off, int w1off, int ZS, int split,
                                          int nsplit, int ksteps, int lr) {
  // byte addresses of this lane's fragments in k-step 0; a k-step advances every one by 32 ZS
  const unsigned zu = smem_u32(st) + 8u * (unsigned)(lr * ZS), wu = smem_u32(sw) + 8u * (unsigned)lr;
  unsigned aA[4], aB[4];
#pragma unroll
  for (int f = 0; f < 4; ++f) {
    aA[f] = zu + 8u * (unsigned)L.offA[f];
    aB[f] = zu + 8u * (unsigned)L.offB[f];
  }
  const unsigned aw0 = wu + 8u * (unsigned)w0off, aw1 = wu + 8u * (unsigned)w1off;
  const unsigned zstep = 32u * (unsigned)ZS;
  for (int ks = split; ks < ksteps; ks += nsplit) {
    const unsigned zo = zstep * (unsigned)ks, wo = 32u * (unsigned)ks;
    double fa[4], fb[4];
    // all loads first (volatile asm keeps them ahead of the DMMAs), then the weights, then the MMAs
#pragma unroll
    for (int f = 0; f < 4; ++f) {
      if (f < NI) fa[f] = lds_f64(aA[f] + zo);
      if (f < NJ) fb[f] = lds_f64(aB[f] + zo);
    }
    const double w0 = lds_f64(aw0 + wo), w1 = lds_f64(aw1 + wo);
#pragma unroll
    for (int f = 0; f < 4; ++f)
      if (f < NJ) fb[f] *= ((L.selB >> f) & 1u) ? w1 : w0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (i < NI && j < NJ && (!STAIR || i <= j)) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
  }
}

__device__ __forceinline__ void gb_dispatch(double (&acc)[4][4][2], int ni, int nj, bool stair,
                                            const double* st, const double* sw, const GbLane& L,
                                            int w0off, int w1off, int ZS, int split, int nsplit,
                                            int ksteps, int lr) {
#define LRVB_GB(NI, NJ, S) gb_ksteps<NI, NJ, S>(acc, st, sw, L, w0off, w1off, ZS, split, nsplit, ksteps, lr)
  if (stair) {
    switch (ni * 4 + nj) {
      case 5: LRVB_GB(1, 1, true); break;
      case 6: LRVB_GB(1, 2, true); break;
      case 7: LRVB_GB(1, 3, true); break;
      case 8: LRVB_GB(1, 4, true); break;
      case 10: LRVB_GB(2, 2, true); break;
      case 11: LRVB_GB(2, 3, true); break;
      case 12: LRVB_GB(2, 4, true); break;
      case 15: LRVB_GB(3, 3, true); break;
      case 16: LRVB_GB(3, 4, true); break;
      default: LRVB_GB(4, 4, true); break;
    }
  } else {
    switch (ni * 4 + nj) {
      case 5: LRVB_GB(1, 1, false); break;
      case 6: LRVB_GB(1, 2, false); break;
      case 7: LRVB_GB(1, 3, false); break;
      case 8: LRVB_GB(1, 4, false); break;
      case 9: LRVB_GB(2, 1, false); break;
      case 10: LRVB_GB(2, 2, false); break;
      case 11: LRVB_GB(2, 3, false); break;
      case 12: LRVB_GB(2, 4, false); break;
      case 13: LRVB_GB(3, 1, false); break;
      case 14: LRVB_GB(3, 2, false); break;
      case 15: LRVB_GB(3, 3, false); break;
      case 16: LRVB_GB(3, 4, false); break;
      case 17: LRVB_GB(4, 1, false); break;
      case 18: LRVB_GB(4, 2, false); break;
      case 19: LRVB_GB(4, 3, false); break;
      default: LRVB_GB(4, 4, false); break;
    }
  }
#undef LRVB_GB
}

// part: (n_chunk, n_groups * 16 warps, 16 tiles, 64); grid = n_groups * n_chunk CTAs of 512 threads
__global__ void __launch_bounds__(32 * kGbWarps, kGbCtasPerSM)
k_gram_big(const double* __restrict__ X, const double* __restrict__ Wabc, int64_t ldw,
           const GbJob* __restrict__ jobs, const GbSlot* __restrict__ slots,
           double* __restrict__ part, int64_t N, int K, int TN, int n_groups, int n_chunk) {
  pdl_sync();
  extern __shared__ __align__(16) double sm[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lr = lane & 3, lc = lane >> 2;
  const int grp = blockIdx.x % n_groups, chunk = blockIdx.x / n_groups;
  const int ZS = 8 * ((2 * K + 7) / 8) + 4;
  const size_t z_elems = (size_t)TN * (ZS + 3);
  double* zbase = sm;                                      // kGbBuffers x [TN x ZS packed rows | a b c]
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(zbase + kGbBuffers * z_elems);
  const unsigned sm_u = smem_u32(sm), bars_u = smem_u32(bars);
  if (tid == 0) {
#pragma unroll
    for (int b2 = 0; b2 < kGbBuffers; ++b2) mbar_init(bars_u + 8 * b2, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  for (int b2 = 0; b2 < kGbBuffers; ++b2)                  // the zero tail of every Z row, once
    for (int r = warp; r < TN; r += kGbWarps)
      for (int c = 2 * K + lane; c < ZS; c += 32) zbase[b2 * z_elems + (size_t)r * ZS + c] = 0.0;

  const GbSlot sl = slots[(size_t)grp * kGbWarps + warp];
  const bool active = sl.job >= 0;
  GbJob jb = {0, 0, 0, 1, 1, 0, 0, 0, 0, 0, 0, 0};
  if (active) jb = jobs[sl.job];

  // per-lane operand recipe
  GbLane L;
  L.selB = 0u;
#pragma unroll
  for (int f = 0; f < 4; ++f) {
    const int ca = 8 * (jb.i0 + f) + lc, cb = 8 * (jb.j0 + f) + lc;
    L.offA[f] = (f < jb.ni) ? ca : 0;
    L.offB[f] = (f < jb.nj) ? cb : 0;
    if (f < jb.nj && cb >= K) L.selB |= 1u << f;
  }
  const bool mcls1 = 8 * jb.i0 + lc >= K;
  const int w0off = jb.w0 * TN, w1off = jb.w1 * TN;

  double acc[4][4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  __syncthreads();

  // Stage j of this CTA is global stage chunk + j n_chunk and lives in buffer j % 3.  The x part
  // of its rows and its weights arrive by bulk async copies (TMA), one per row, straight into the
  // packed layout (K even; odd K rows are not 16-B aligned and are loaded by the warps instead);
  // the s part is squared in place by the warps that finish stage j - 1 early; ONE block barrier
  // per stage.  A buffer is refilled two stages ahead.
  const int64_t nstage = (N + TN - 1) / TN;
  const int64_t nfull = N / TN;
  const int64_t nmine = (chunk < nstage) ? (nstage - chunk + n_chunk - 1) / n_chunk : 0;
  const bool tma_x = (K & 1) == 0;
  const unsigned rbytes = (unsigned)(K * sizeof(double));
  const unsigned wbytes = (unsigned)(TN * sizeof(double));
  auto arm = [&](int64_t j) {      // thread 0, BEFORE the barrier that precedes issue(j)
    if (j < nmine && chunk + j * n_chunk < nfull)
      mbar_arrive_expect_tx(bars_u + 8 * (unsigned)(j % kGbBuffers), (tma_x ? TN * rbytes : 0u) + 3 * wbytes);
  };
  auto issue = [&](int64_t j) {    // threads 0 .. TN-1: one row each; threads TN .. TN+2: the weights
    const int64_t s = chunk + j * n_chunk;
    if (j < nmine && s < nfull && tid < TN + 3) {
      const unsigned b2 = (unsigned)(j % kGbBuffers);
      const unsigned bar = bars_u + 8 * b2;
      const unsigned dst = sm_u + (unsigned)(b2 * z_elems * sizeof(double));
      if (tid < TN) {
        if (tma_x) bulk_g2s(dst + (unsigned)tid * (unsigned)(ZS * sizeof(double)), X + (s * TN + tid) * K, rbytes, bar);
      } else {
        const int f = tid - TN;
        bulk_g2s(dst + (unsigned)((size_t)TN * ZS * sizeof(double)) + f * wbytes,
                 Wabc + (int64_t)f * ldw + s * TN, wbytes, bar);
      }
    }
  };
  auto square = [&](int64_t j) {   // all warps: finish stage j in its buffer (s = x * x)
    const int64_t s = chunk + j * n_chunk;
    double* zb = zbase + (j % kGbBuffers) * z_elems;
    double* zw = zb + (size_t)TN * ZS;
    if (s < nfull) {
      mbar_wait(bars_u + 8 * (unsigned)(j % kGbBuffers), (unsigned)(j / kGbBuffers) & 1u);
      for (int r0 = 4 * warp; r0 < TN; r0 += 4 * kGbWarps)
        for (int k = lane; k < K; k += 32) {
          double v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u)
            v[u] = tma_x ? zb[(size_t)(r0 + u) * ZS + k] : X[(s * TN + r0 + u) * K + k];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (!tma_x) zb[(size_t)(r0 + u) * ZS + k] = v[u];
            zb[(size_t)(r0 + u) * ZS + K + k] = v[u] * v[u];
          }
        }
    } else {   // ragged last stage of the data: straight from global memory, zero fill
      const int rows = (int)(N - s * TN);
      for (int r = warp; r < TN; r += kGbWarps)
        for (int k = lane; k < K; k += 32) {
          const double v = (r < rows) ? X[(s * TN + r) * K + k] : 0.0;
          zb[(size_t)r * ZS + k] = v;
          zb[(size_t)r * ZS + K + k] = v * v;
        }
      for (int e = tid; e < 3 * TN; e += blockDim.x) {
        const int f = e / TN, r = e % TN;
        zw[e] = (r < rows) ? Wabc[(int64_t)f * ldw + s * TN + r] : 0.0;
      }
    }
  };

  if (tid == 0) { arm(0); arm(1); }
  __syncthreads();
  issue(0);
  issue(1);
  if (nmine > 0) square(0);
  if (tid == 0) arm(2);
  __syncthreads();
  issue(2);
  for (int64_t j = 0; j < nmine; ++j) {
    const int64_t s = chunk + j * n_chunk;
    const double* zb = zbase + (j % kGbBuffers) * z_elems;
    const double* sw = zb + (size_t)TN * ZS;
    const int rows = (s < nfull) ? TN : (int)(N - s * TN);
    const int ksteps = (rows + 3) >> 2;
    if (active) {
      if (jb.kind == 0) {
        gb_dispatch(acc, jb.ni, jb.nj, jb.stair != 0, zb, sw, L, w0off, w1off, ZS, sl.split, sl.nsplit,
                    ksteps, lr);
      } else {
        // straddle tile against itself: x rows use B = z (a | b), s rows use B = z (b | c)
        for (int ks = sl.split; ks < ksteps; ks += sl.nsplit) {
          const int n = 4 * ks + lr;
          const double v = zb[(size_t)n * ZS + L.offA[0]];
          const double wa = sw[n], wb = sw[TN + n], wc = sw[2 * TN + n];
          const double b0 = v * (mcls1 ? wb : wa), b1 = v * (mcls1 ? wc : wb);
          dmma884(acc[0][0][0], acc[0][0][1], mcls1 ? 0.0 : v, b0);
          dmma884(acc[0][0][0], acc[0][0][1], mcls1 ? v : 0.0, b1);
        }
      }
    }
    if (j + 1 < nmine) square(j + 1);    // its TMA was issued two barriers ago
    if (tid == 0) arm(j + 3);            // buffer j % 3: its phase for stage j completed long ago
    __syncthreads();                     // stage j + 1 complete in shared memory; buffer j % 3 is free
    issue(j + 3);
  }

  if (active) {
    double* out = part + (((size_t)chunk * n_groups + grp) * kGbWarps + warp) * (16 * 64);
    const int crow = lane >> 2, ccol = 2 * (lane & 3);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (i < jb.ni && j < jb.nj && (!jb.stair || i <= j))
          *reinterpret_cast<double2*>(out + (i * 4 + j) * 64 + crow * 8 + ccol) =
              make_double2(acc[i][j][0], acc[i][j][1]);
  }
}

// Sum the partials of one (job, tile) over the row chunks and the k-splits in a fixed order and
// write the beta block of A in free coordinates (same chain rule as gram_small_finish_body).
__device__ __forceinline__ void gram_big_finish_body(int bid, const double* __restrict__ part, const GbJob* __restrict__ jobs,
                  const GbSlot* __restrict__ slots, const double* __restrict__ vec,
                  double* __restrict__ A, int K, int Dg, int n_groups, int n_chunk,
                  lrvb_glmm_bounds bd, int vecmode) {
  __shared__ double red[4][64];
  const int job = bid / 16, t = bid % 16;
  const GbJob jb = jobs[job];
  const int ti = t / 4, tj = t % 4;
  if (ti >= jb.ni || tj >= jb.nj || (jb.stair && ti > tj)) return;
  const int e = threadIdx.x & 63, ps = threadIdx.x >> 6;
  double s = 0.0;
  for (int c = ps; c < n_chunk; c += 4)
    for (int w = 0; w < kGbWarps; ++w)
      if (slots[(size_t)jb.group * kGbWarps + w].job == job)
        s += part[((((size_t)c * n_groups + jb.group) * kGbWarps + w) * 16 + t) * 64 + e];
  red[ps][e] = s;
  __syncthreads();
  if (ps != 0) return;
  s = (red[0][e] + red[1][e]) + (red[2][e] + red[3][e]);
  int p = 8 * (jb.i0 + ti) + (e >> 3), q = 8 * (jb.j0 + tj) + (e & 7);
  if (jb.transposed) { const int tmp = p; p = q; q = tmp; }
  if (p > q || q >= 2 * K) return;
  const int bm0 = 4, bi0 = 4 + K;
  if (q < K) {
    const double v = -s;
    A[(size_t)(bm0 + p) * Dg + bm0 + q] = v;
    A[(size_t)(bm0 + q) * Dg + bm0 + p] = v;
  } else if (p < K) {
    const int k2 = q - K;
    const double iq = vec[bi0 + k2];
    const double v = -s * (-1.0 / (iq * iq)) * (vecmode ? 1.0 : iq - bd.beta_info);
    A[(size_t)(bm0 + p) * Dg + bi0 + k2] = v;
    A[(size_t)(bi0 + k2) * Dg + bm0 + p] = v;
  } else {
    const int k1 = p - K, k2 = q - K;
    const double ip = vec[bi0 + k1], iq = vec[bi0 + k2];
    const double v = -s * (1.0 / (ip * ip * iq * iq)) *
                     (vecmode ? 1.0 : (ip - bd.beta_info) * (iq - bd.beta_info));
    A[(size_t)(bi0 + k1) * Dg + bi0 + k2] = v;
    A[(size_t)(bi0 + k2) * Dg + bi0 + k1] = v;
  }
}

#endif  // LRVB_GRAM_BIG_KERNELS

}  // namespace lrvb
