// Weighted Grams of the beta block for LARGE K (K % 8 == 0, K = 176 .. 240; BASELINE configs[3]: K = 200) on the
// FP64 tensor cores (DMMA.8x8x4), sm_100a.  The planner covers every K >= 96 with K % 8 == 0.
//
// Same packed formulation as gram_small / gram_mid / gram_big: one weighted Gram of z_n = [x_n | s_n]
// (2K columns, T2 = K/4 tiles of 8), upper triangle only; with K % 8 == 0 no tile straddles the x | s
// boundary, so the weight of a tile is one of a (x,x), b (x,s), c (s,s).  What this kernel changes against
// the rectangle kernel (gram_big.cuh: 16 warps x 128 registers, jobs of <= 4 x 4 tiles of every shape,
// every CTA stages all 2K columns -> 16 rows per stage at K = 200, 51 % of the DGEMM peak):
//   * the measured rule of this pipe (tools/dmma_probe4.cu, gram_mid.cuh): a warp needs >= ~24 independent
//     accumulator tiles per k-step and every warp of a CTA the SAME work.  Each half of the packed columns
//     is cut into blocks of 4 or 5 tiles; a warp job is one block against another (16 - 25 tiles, 200
//     registers, 8 warps per SM) or a block against itself (a "stair": 10 / 15 live tiles);
//   * a CTA (job group) runs 8 jobs and stages ONLY the column blocks its jobs touch (4 - 8 of the 2K/40
//     blocks) by bulk async copies (TMA, one per row and run of adjacent blocks) into a 3-slot ring: 28 - 56
//     rows per stage instead of 16, and the groups that share rows run at the same time, so the re-reads of
//     X are L2 hits (ncu: DRAM read 1.18 GB for 0.8 GB of X);
//   * the s = x * x blocks of stage j + 1 are squared in place DURING the k-steps of stage j (two pairs per
//     k-step: loads ahead of the DMMAs, stores behind) -- as a separate pass between stages it cost 20 % of
//     the kernel;
//   * groups are composed so that the two warps of every SM sub-partition carry the same DMMA count
//     (4 rectangle + 4 stair jobs, or 8 rectangle jobs), and the 148 CTAs are dealt to the groups in
//     proportion to their load (a group with lighter jobs gets fewer CTAs, i.e. more rows each);
//   * partials go to the packed layout (n_cta, NT, 64) of gram_small / gram_mid (slot j (j+1)/2 + i), a CTA
//     writes the tiles of its jobs and never touches the others (zero since creation), so the finishing
//     pass is gram_small_finish_body unchanged;
//   * at 200 registers x 256 threads the CTA leaves room for one 48-register CTA per SM: launch_eval runs
//     k_group beside it on a side stream.
// Measured (profiles/r02_gram_wide.md, every step incl. the failed ones): K = 200: 0.68 of the DGEMM peak
// (DMMA pipe 69 % active; rectangle kernel 0.51); faster than the rectangle kernel for K = 176 .. 240.
#pragma once
#include <algorithm>
#include <vector>
#include "common.cuh"
#include "gram_small.cuh"   // mbarrier / bulk-copy helpers, packed partial layout

namespace lrvb {

constexpr int kGwWarps = 8;
#ifndef LRVB_GW_MAXBLK
#define LRVB_GW_MAXBLK 8
#endif
constexpr int kGwMaxBlk = LRVB_GW_MAXBLK;   // distinct column blocks a CTA may stage
constexpr int kGwBuffers = 3;
constexpr int kGwBlkTiles = 5;     // largest block (tiles); a job has <= 5 x 5 accumulator tiles
constexpr size_t kGwSmemCap = 225 * 1024;

struct GwJob {        // one warp's job inside a group
  int offA, offB;     // staged column of the first A / B column of the job
  int ni, nj;         // tiles (4 or 5 each; ni == 0: idle warp)
  int stair;          // a block against itself: tiles i <= j only
  int wrow;           // weight row: 0 a, 1 b, 2 c
  int ti0, tj0;       // packed tile coordinates of the job's first tile
};
struct GwGroup {
  int nblk, ZS, TN, ncols;     // staged row stride in doubles (== 4 mod 8), rows per stage, sum of blk_cols
  int blk_x[kGwMaxBlk];        // first X column of the block
  int blk_cols[kGwMaxBlk];     // columns (8 per tile)
  int blk_off[kGwMaxBlk];      // first staged column
  int blk_sq[kGwMaxBlk];       // 1: s block (squared in place after the copy)
  int sq_off, sq_cols;         // the s blocks are the tail [sq_off, sq_off + sq_cols) of a staged row
  int nrun;                    // bulk copies per row: maximal runs of staged blocks with adjacent X columns
  int run_x[kGwMaxBlk], run_cols[kGwMaxBlk], run_off[kGwMaxBlk];
  GwJob job[kGwWarps];
};
struct GwCta { int group, chunk, nchunk, pad; };

struct GwPlan {
  std::vector<GwGroup> groups;
  std::vector<GwCta> ctas;     // one entry per CTA of the grid (<= kNumSMs)
  std::vector<int> load;       // per group: DMMAs per k-step of its busiest sub-partition
  size_t smem = 0;             // largest dynamic shared memory of a group
  int tiles_live = 0;
};

inline size_t gram_wide_smem(int ZS, int TN) {
  return sizeof(double) * kGwBuffers * (size_t)TN * (ZS + 3) + 64;
}
// where it beats the rectangle kernel (profiles/r02_gram_wide.md: 56 - 66 % against 49 - 55 % of the DMMA peak
// for K = 176 .. 240; below, the 4-tile blocks starve the warps and the staged bytes per DMMA grow)
inline bool gram_wide_eligible(int K) { return K >= 176 && K <= 240 && K % 8 == 0; }

inline GwPlan gram_wide_plan(int K) {
  GwPlan pl;
  const int T0 = K / 8;
  const int nb0 = (T0 + kGwBlkTiles - 1) / kGwBlkTiles, nb = 2 * nb0;
  struct Blk { int tile0, nt, xcol, sq; };
  std::vector<Blk> blk;
  for (int h = 0; h < 2; ++h) {
    int t = 0;
    for (int b = 0; b < nb0; ++b) {
      const int nt = T0 / nb0 + (b < T0 % nb0 ? 1 : 0);
      blk.push_back(Blk{h * T0 + t, nt, 8 * t, h});
      t += nt;
    }
  }
  struct J { int I, Jb, nt; };
  auto mk = [&](int I, int Jb) {
    const int ni = blk[I].nt, nj = blk[Jb].nt;
    return J{I, Jb, I == Jb ? ni * (ni + 1) / 2 : ni * nj};
  };
  std::vector<std::vector<J>> members;
  std::vector<char> used((size_t)nb * nb, 0);
  // (1) cliques of 4 consecutive blocks: their 4 stairs + 4 of their 6 rectangles -> every sub-partition
  //     carries one rectangle and one stair
  for (int b0 = 0; b0 + 4 <= nb; b0 += 4) {
    std::vector<J> m;
    for (int d = 0; d < 4; ++d) m.push_back(mk(b0 + d, b0 + d));
    const int pr[4][2] = {{0, 1}, {2, 3}, {0, 2}, {1, 3}};
    for (auto& p : pr) m.push_back(mk(b0 + p[0], b0 + p[1]));
    for (auto& j : m) used[(size_t)j.I * nb + j.Jb] = 1;
    members.push_back(m);
  }
  // (2) everything else in macro-row order (two block rows at a time, column by column), 8 jobs per group,
  //     a group closes early when the next job would need a 9th column block
  std::vector<J> seq;
  for (int r = 0; 2 * r < nb; ++r)
    for (int Jb = 2 * r; Jb < nb; ++Jb)
      for (int I = 2 * r; I <= 2 * r + 1 && I < nb && I <= Jb; ++I)
        if (!used[(size_t)I * nb + Jb]) seq.push_back(mk(I, Jb));
  {
    std::vector<J> m;
    std::vector<int> bs;
    auto nblocks_with = [&](const J& j) {
      int n = (int)bs.size();
      if (std::find(bs.begin(), bs.end(), j.I) == bs.end()) ++n;
      if (j.Jb != j.I && std::find(bs.begin(), bs.end(), j.Jb) == bs.end()) ++n;
      return n;
    };
    for (const J& j : seq) {
      if ((int)m.size() == kGwWarps || nblocks_with(j) > kGwMaxBlk) {
        members.push_back(m);
        m.clear();
        bs.clear();
      }
      m.push_back(j);
      if (std::find(bs.begin(), bs.end(), j.I) == bs.end()) bs.push_back(j.I);
      if (std::find(bs.begin(), bs.end(), j.Jb) == bs.end()) bs.push_back(j.Jb);
    }
    if (!m.empty()) members.push_back(m);
  }
  // groups: staged blocks, warp slots dealt longest-first to the sub-partitions (warp w runs on w % 4)
  for (auto& m : members) {
    GwGroup g = {};
    std::vector<int> bs;
    for (auto& j : m) {
      if (std::find(bs.begin(), bs.end(), j.I) == bs.end()) bs.push_back(j.I);
      if (std::find(bs.begin(), bs.end(), j.Jb) == bs.end()) bs.push_back(j.Jb);
    }
    std::sort(bs.begin(), bs.end());
    g.nblk = (int)bs.size();
    int off = 0;
    for (int i = 0; i < g.nblk; ++i) {
      const Blk& b = blk[bs[i]];
      g.blk_x[i] = b.xcol; g.blk_cols[i] = 8 * b.nt; g.blk_off[i] = off; g.blk_sq[i] = b.sq;
      off += 8 * b.nt;
    }
    g.ncols = off;
    g.ZS = off + 4;
    g.sq_off = off;
    for (int i = g.nblk - 1; i >= 0 && g.blk_sq[i]; --i) g.sq_off = g.blk_off[i];
    g.sq_cols = off - g.sq_off;
    for (int i = 0; i < g.nblk; ++i) {
      if (i > 0 && g.blk_sq[i] == g.blk_sq[i - 1] && g.blk_x[i] == g.blk_x[i - 1] + g.blk_cols[i - 1]) {
        g.run_cols[g.nrun - 1] += g.blk_cols[i];
      } else {
        g.run_x[g.nrun] = g.blk_x[i]; g.run_cols[g.nrun] = g.blk_cols[i]; g.run_off[g.nrun] = g.blk_off[i];
        ++g.nrun;
      }
    }
    int TN = 64;
    while (TN > 8 && gram_wide_smem(g.ZS, TN) > kGwSmemCap) TN -= 4;
    g.TN = TN;
    pl.smem = std::max(pl.smem, gram_wide_smem(g.ZS, TN));
    std::stable_sort(m.begin(), m.end(), [](const J& a, const J& b) { return a.nt > b.nt; });
    int load[4] = {0, 0, 0, 0}, cnt[4] = {0, 0, 0, 0};
    for (auto& j : m) {
      int best = -1;
      for (int q = 0; q < 4; ++q)
        if (cnt[q] < kGwWarps / 4 && (best < 0 || load[q] < load[best])) best = q;
      const int w = best + 4 * cnt[best];
      ++cnt[best];
      load[best] += j.nt;
      pl.tiles_live += j.nt;
      GwJob& jb = g.job[w];
      auto staged = [&](int b) {
        return g.blk_off[std::find(bs.begin(), bs.end(), b) - bs.begin()];
      };
      jb.offA = staged(j.I); jb.offB = staged(j.Jb);
      jb.ni = blk[j.I].nt; jb.nj = blk[j.Jb].nt;
      jb.stair = (j.I == j.Jb) ? 1 : 0;
      jb.wrow = blk[j.Jb].sq == 0 ? 0 : (blk[j.I].sq == 0 ? 1 : 2);
      jb.ti0 = blk[j.I].tile0; jb.tj0 = blk[j.Jb].tile0;
    }
    pl.load.push_back(std::max(std::max(load[0], load[1]), std::max(load[2], load[3])));
    pl.groups.push_back(g);
  }
  // CTAs per group in proportion to the load (largest remainder), at least one each
  const int ng = (int)pl.groups.size();
  long total = 0;
  for (int l : pl.load) total += l;
  std::vector<int> nc(ng, 1);
  int left = kNumSMs - ng;
  std::vector<double> want(ng);
  for (int g = 0; g < ng; ++g) want[g] = (double)kNumSMs * pl.load[g] / (double)total;
  for (int g = 0; g < ng; ++g) {
    const int extra = std::min(left, std::max(0, (int)want[g] - 1));
    nc[g] += extra;
    left -= extra;
  }
  while (left > 0) {   // hand the rest to the groups with the most rows per CTA
    int best = 0;
    for (int g = 1; g < ng; ++g)
      if ((double)pl.load[g] / nc[g] > (double)pl.load[best] / nc[best]) best = g;
    ++nc[best];
    --left;
  }
  for (int g = 0; g < ng; ++g)
    for (int c = 0; c < nc[g]; ++c) pl.ctas.push_back(GwCta{g, c, nc[g], 0});
  return pl;
}

// ---- device side (compiled by the translation unit that defines LRVB_GRAM_WIDE_KERNELS) ------
#ifdef LRVB_GRAM_WIDE_KERNELS

__device__ __forceinline__ double2 lds_f64x2(unsigned addr) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];\n" : "=d"(v.x), "=d"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f64x2(unsigned addr, double2 v) {
  asm volatile("st.shared.v2.f64 [%0], {%1, %2};\n" ::"r"(addr), "d"(v.x), "d"(v.y) : "memory");
}

// A thread's walk over the s part of the NEXT stage (pairs of doubles e = tid, tid + 256, ... of the TN x sqh
// array of pairs): squared in place two pairs per k-step, the loads ahead of the k-step's DMMAs and the
// stores behind them, so the pass costs issue slots only.
struct GwSquare {
  unsigned addr;      // shared-memory byte address of the next pair
  int r, c2;          // its row and pair index
  int TN, sqh;        // rows, pairs per row
  unsigned step, wrap;   // address advance per element / correction when c2 wraps into the next row
  int dr, dc;
  __device__ __forceinline__ bool live() const { return r < TN; }
  __device__ __forceinline__ void next() {
    r += dr; c2 += dc; addr += step;
    if (c2 >= sqh) { c2 -= sqh; ++r; addr += wrap; }
  }
};

// (Fetching the fragments of k-step ks + 1 ahead of the DMMAs of k-step ks was measured and is 5 % SLOWER:
// the operand fetch is not what the pipe waits for; profiles/r02_gram_wide.md.)
template <int NI, int NJ, bool STAIR>
__device__ __forceinline__ void gw_ksteps(double (&acc)[5][5][2], unsigned aA, unsigned aB, unsigned aw,
                                          unsigned zstep, int ksteps, GwSquare& sq) {
  for (int ks = 0; ks < ksteps; ++ks) {
    double fa[NI], fb[NJ];
    double2 v0 = make_double2(0.0, 0.0), v1 = make_double2(0.0, 0.0);
    const bool l0 = sq.live();
    const unsigned a0 = sq.addr;
    if (l0) { v0 = lds_f64x2(a0); sq.next(); }
    const bool l1 = sq.live();
    const unsigned a1 = sq.addr;
    if (l1) { v1 = lds_f64x2(a1); sq.next(); }
#pragma unroll
    for (int f = 0; f < NI; ++f) fa[f] = lds_f64(aA + 64u * f);
#pragma unroll
    for (int f = 0; f < NJ; ++f) fb[f] = lds_f64(aB + 64u * f);
    const double w = lds_f64(aw);
#pragma unroll
    for (int f = 0; f < NJ; ++f) fb[f] *= w;
#pragma unroll
    for (int i = 0; i < NI; ++i)
#pragma unroll
      for (int j = 0; j < NJ; ++j)
        if (!STAIR || i <= j) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
    if (l0) { v0.x *= v0.x; v0.y *= v0.y; sts_f64x2(a0, v0); }
    if (l1) { v1.x *= v1.x; v1.y *= v1.y; sts_f64x2(a1, v1); }
    aA += zstep; aB += zstep; aw += 32u;
  }
}

// grid = plan.ctas.size() CTAs of 256 threads; part: (gridDim.x, NT, 64)
__global__ void __launch_bounds__(32 * kGwWarps, 1)
k_gram_wide(const double* __restrict__ X, const double* __restrict__ Wabc, int64_t ldw,
            const GwGroup* __restrict__ groups, const GwCta* __restrict__ ctas,
            double* __restrict__ part, int64_t N, int K, int NT) {
  pdl_sync();
  extern __shared__ __align__(16) double sm[];
  __shared__ GwGroup G;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lr = lane & 3, lc = lane >> 2;
  const GwCta me = ctas[blockIdx.x];
  {
    const int* src = reinterpret_cast<const int*>(groups + me.group);
    int* dst = reinterpret_cast<int*>(&G);
    for (int i = tid; i < (int)(sizeof(GwGroup) / sizeof(int)); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int ZS = G.ZS, TN = G.TN, nblk = G.nblk;
  const int chunk = me.chunk, n_chunk = me.nchunk;
  const size_t z_elems = (size_t)TN * (ZS + 3);
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(sm + kGwBuffers * z_elems);
  const unsigned sm_u = smem_u32(sm), bars_u = smem_u32(bars);
  if (tid == 0) {
#pragma unroll
    for (int b2 = 0; b2 < kGwBuffers; ++b2) mbar_init(bars_u + 8 * b2, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  const GwJob jb = G.job[warp];
  const bool active = jb.ni > 0;

  double acc[5][5][2];
#pragma unroll
  for (int i = 0; i < 5; ++i)
#pragma unroll
    for (int j = 0; j < 5; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  __syncthreads();

  // Stage j of this CTA is global stage chunk + j n_chunk and lives in buffer j % 3: the column blocks of
  // its TN rows (one bulk async copy per row and run of adjacent blocks) and the three weight rows arrive by
  // TMA; the s blocks of stage j + 1 are squared in place DURING the k-steps of stage j; ONE block barrier
  // per stage.
  const int64_t nstage = (N + TN - 1) / TN;
  const int64_t nfull = N / TN;
  const int64_t nmine = (chunk < nstage) ? (nstage - chunk + n_chunk - 1) / n_chunk : 0;
  const unsigned wbytes = (unsigned)(TN * sizeof(double));
  const unsigned stage_bytes = (unsigned)(TN * G.ncols * sizeof(double)) + 3 * wbytes;
  auto arm = [&](int64_t j) {      // thread 0, BEFORE the barrier that precedes issue(j)
    if (j < nmine && chunk + j * n_chunk < nfull)
      mbar_arrive_expect_tx(bars_u + 8 * (unsigned)(j % kGwBuffers), stage_bytes);
  };
  auto issue = [&](int64_t j) {
    const int64_t s = chunk + j * n_chunk;
    if (j < nmine && s < nfull) {
      const unsigned b2 = (unsigned)(j % kGwBuffers);
      const unsigned bar = bars_u + 8 * b2;
      const unsigned dst = sm_u + (unsigned)(b2 * z_elems * sizeof(double));
      const int npiece = TN * G.nrun;
      for (int p = tid; p < npiece + 3; p += blockDim.x) {
        if (p < npiece) {
          const int b = p / TN, r = p - b * TN;
          bulk_g2s(dst + (unsigned)((r * ZS + G.run_off[b]) * sizeof(double)),
                   X + (s * TN + r) * K + G.run_x[b], (unsigned)(G.run_cols[b] * sizeof(double)), bar);
        } else {
          const int f = p - npiece;
          bulk_g2s(dst + (unsigned)((size_t)TN * ZS * sizeof(double)) + f * wbytes,
                   Wabc + (int64_t)f * ldw + s * TN, wbytes, bar);
        }
      }
    }
  };
  // this thread's walk over the s part of a stage
  const int sqh = G.sq_cols >> 1;
  GwSquare sq0;
  sq0.TN = TN; sq0.sqh = sqh;
  sq0.dr = sqh > 0 ? 256 / sqh : 0; sq0.dc = sqh > 0 ? 256 % sqh : 0;
  sq0.r = sqh > 0 ? tid / sqh : TN; sq0.c2 = sqh > 0 ? tid % sqh : 0;
  sq0.step = (unsigned)(8 * (sq0.dr * ZS + 2 * sq0.dc));
  sq0.wrap = (unsigned)(8 * (ZS - 2 * sqh));
  sq0.addr = (unsigned)(8 * (sq0.r * ZS + G.sq_off + 2 * sq0.c2));   // relative to the buffer
  auto wait_stage = [&](int64_t j) {
    mbar_wait(bars_u + 8 * (unsigned)(j % kGwBuffers), (unsigned)(j / kGwBuffers) & 1u);
  };
  auto square_rest = [&](GwSquare& sq) {   // whatever the k-steps did not cover (all of it for stage 0)
    while (sq.live()) {
      double2 v = lds_f64x2(sq.addr);
      v.x *= v.x; v.y *= v.y;
      sts_f64x2(sq.addr, v);
      sq.next();
    }
  };
  auto fill_ragged = [&](int64_t j) {   // ragged last stage of the data: straight from global memory, zero fill
    const int64_t s = chunk + j * n_chunk;
    double* zb = sm + (j % kGwBuffers) * z_elems;
    double* zw = zb + (size_t)TN * ZS;
    const int rows = (int)(N - s * TN);
    for (int b = 0; b < nblk; ++b) {
      const int cols = G.blk_cols[b], sq = G.blk_sq[b];
      for (int r = warp; r < TN; r += kGwWarps)
        for (int c = lane; c < cols; c += 32) {
          const double v = (r < rows) ? X[(s * TN + r) * K + G.blk_x[b] + c] : 0.0;
          zb[(size_t)r * ZS + G.blk_off[b] + c] = sq ? v * v : v;
        }
    }
    for (int e = tid; e < 3 * TN; e += blockDim.x) {
      const int f = e / TN, r = e % TN;
      zw[e] = (r < rows) ? Wabc[(int64_t)f * ldw + s * TN + r] : 0.0;
    }
  };

  if (tid == 0) { arm(0); arm(1); }
  __syncthreads();
  issue(0);
  issue(1);
  if (nmine > 0) {
    if (chunk < nfull) {
      wait_stage(0);
      GwSquare sq = sq0;
      sq.addr += sm_u;
      square_rest(sq);
    } else {
      fill_ragged(0);
    }
  }
  if (tid == 0) arm(2);
  __syncthreads();
  issue(2);
  const unsigned zstep = 32u * (unsigned)ZS;
  for (int64_t j = 0; j < nmine; ++j) {
    const int64_t s = chunk + j * n_chunk;
    const unsigned zb_u = sm_u + (unsigned)((j % kGwBuffers) * z_elems * sizeof(double));
    const int rows = (s < nfull) ? TN : (int)(N - s * TN);
    const int ksteps = (rows + 3) >> 2;
    const bool next_full = (j + 1 < nmine) && (s + n_chunk < nfull);
    GwSquare sq = sq0;
    if (next_full) {
      wait_stage(j + 1);     // its copies were issued two barriers ago
      sq.addr += sm_u + (unsigned)(((j + 1) % kGwBuffers) * z_elems * sizeof(double));
    } else {
      sq.r = TN;
    }
    if (active) {
      const unsigned zu = zb_u + 8u * (unsigned)(lr * ZS + lc);
      const unsigned aA = zu + 8u * (unsigned)jb.offA, aB = zu + 8u * (unsigned)jb.offB;
      const unsigned aw = zb_u + 8u * (unsigned)(TN * ZS + jb.wrow * TN + lr);
#define LRVB_GW(NI, NJ, S) gw_ksteps<NI, NJ, S>(acc, aA, aB, aw, zstep, ksteps, sq)
      if (jb.stair) {
        if (jb.ni == 5) LRVB_GW(5, 5, true); else LRVB_GW(4, 4, true);
      } else if (jb.ni == 5) {
        if (jb.nj == 5) LRVB_GW(5, 5, false); else LRVB_GW(5, 4, false);
      } else {
        if (jb.nj == 5) LRVB_GW(4, 5, false); else LRVB_GW(4, 4, false);
      }
#undef LRVB_GW
    }
    square_rest(sq);
    if (j + 1 < nmine && !next_full) fill_ragged(j + 1);
    if (tid == 0) arm(j + 3);            // buffer j % 3: its phase for stage j completed long ago
    __syncthreads();                     // stage j + 1 complete in shared memory; buffer j % 3 is free
    issue(j + 3);
  }

  if (active) {
    double* out = part + (size_t)blockIdx.x * NT * 64;
    const int crow = lane >> 2, ccol = 2 * (lane & 3);
#pragma unroll
    for (int i = 0; i < 5; ++i)
#pragma unroll
      for (int j = 0; j < 5; ++j)
        if (i < jb.ni && j < jb.nj && (!jb.stair || i <= j)) {
          const int ti = jb.ti0 + i, tj = jb.tj0 + j;
          *reinterpret_cast<double2*>(out + (size_t)(tj * (tj + 1) / 2 + ti) * 64 + crow * 8 + ccol) =
              make_double2(acc[i][j][0], acc[i][j][1]);
        }
  }
}

#endif  // LRVB_GRAM_WIDE_KERNELS

}  // namespace lrvb
