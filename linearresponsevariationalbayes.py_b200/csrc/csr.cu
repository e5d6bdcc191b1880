// Device-side CSR export of the arrowhead Hessian.
//
// Replaces get_sparse_sub_hessian / get_sparse_sub_matrix (SparseObjectives.py:591-619) followed
// by scipy's COO->CSR canonicalisation: entries that are EXACTLY 0.0 are dropped, each
// coordinate appears once, column indices are sorted, indices / indptr are int32.
// Row r of H in the reference layout [globals | u.mean (G) | u.info (G)]:
//   r <  Dg      : A[r,:] , B[g,0,r] for g = 0..G-1 , B[g,1,r] for g = 0..G-1
//   r = Dg+g     : B[g,0,:] , L[g].mm , L[g].mi
//   r = Dg+G+g   : B[g,1,:] , L[g].mi , L[g].ii
// so the column order is already sorted and every kernel only compacts in order.
//
// The global rows are columns of B (group-major in memory), so they are produced by a
// transposing pass: a CTA stages a chunk of kCG groups of B in shared memory (coalesced), then
// each warp takes one (side, global row) column and ballot-compacts its kCG entries into a
// contiguous, coalesced segment of that CSR row.  Per-(chunk, column) counts are scanned over
// chunks to give each segment its offset.  Nothing synchronises with the host: nnz is left in a
// device scalar.
//
// The sparsity pattern is static between evaluations unless an entry becomes (or stops being) exactly
// zero, so the full export also records the ZERO MASK of every structural candidate (one bit each: A,
// then B, then L) and keeps its scan results; lrvb_glmm_hessian_csr_refill then rewrites `data` alone in
// ONE pass with the cached offsets and compares the mask of the new values with the recorded one -- any
// difference raises a device flag, and the caller's conditional full export (run_if) takes over.
#include "common.cuh"
#include "gram_small.cuh"   // mbarrier / bulk-copy helpers

namespace lrvb {

constexpr int kScanChunk = 2048;  // per CTA (256 threads x 8)

// ---- local rows: one warp per row ------------------------------------------------------------
// mask words: [A: Dg rows x WA words | B: 2 G rows x WA words | L: G words (3 bits)], WA = ceil(Dg / 32)
// mismatch: [0] the device flag the conditional export reads, [1] (nullable) its copy in mapped pinned
// host memory, which the host reads after the kernel without a device-to-host copy on the stream
struct MismatchFlag {
  int* dev;
  int* host;
};
template <int FILL>
__device__ __forceinline__ void mask_word(uint32_t* __restrict__ mask, size_t w, unsigned m, const MismatchFlag& mm) {
  if (FILL == 1) mask[w] = m;
  else if (FILL == 2 && mask[w] != m) {
    *mm.dev = 1;
    if (mm.host) *(volatile int*)mm.host = 1;
  }
}

template <int FILL>
__device__ __forceinline__ void csr_local_rows_body(int bid, const double* __restrict__ B, const double* __restrict__ L, int Dg, int G,
                 int32_t* __restrict__ rowcnt, const int32_t* __restrict__ indptr,
                 int32_t* __restrict__ indices, double* __restrict__ data, uint32_t* __restrict__ mask,
                 const MismatchFlag mismatch) {
  const int lane = threadIdx.x & 31;
  const int64_t wg = (int64_t)bid * 8 + (threadIdx.x >> 5);
  if (wg >= 2 * (int64_t)G) return;
  const int which = (wg >= G) ? 1 : 0;
  const int gi = (int)(wg - (which ? G : 0));
  const int64_t row = Dg + wg;
  const double* b = B + (size_t)gi * 2 * Dg + (which ? Dg : 0);
  int64_t base = FILL ? indptr[row] : 0;
  int count = 0;
  const int WA = (Dg + 31) >> 5;
  for (int c0 = 0; c0 < Dg; c0 += 32) {
    const int c = c0 + lane;
    const double v = (c < Dg) ? b[c] : 0.0;
    const bool nz = (v != 0.0);
    const unsigned m = __ballot_sync(0xffffffffu, nz);
    if (FILL && nz) {
      const int off = __popc(m & ((1u << lane) - 1));
      if (FILL == 1) indices[base + off] = c;
      data[base + off] = v;
    }
    // the mask of B is recorded / compared by the local rows (every B entry belongs to exactly one)
    if (FILL && lane == 0) mask_word<FILL>(mask, (size_t)(Dg + wg) * WA + (c0 >> 5), m, mismatch);
    base += __popc(m);
    count += __popc(m);
  }
  if (lane == 0) {
    const double l0 = L[(size_t)gi * 3], l1 = L[(size_t)gi * 3 + 1], l2 = L[(size_t)gi * 3 + 2];
    const double va = which ? l1 : l0;   // column u.mean_g
    const double vb = which ? l2 : l1;   // column u.info_g
    if (va != 0.0) {
      if (FILL == 1) indices[base] = Dg + gi;
      if (FILL) data[base] = va;
      ++base; ++count;
    }
    if (vb != 0.0) {
      if (FILL == 1) indices[base] = Dg + G + gi;
      if (FILL) data[base] = vb;
      ++base; ++count;
    }
    if (!FILL) rowcnt[row] = count;
    if (FILL && which == 0)
      mask_word<FILL>(mask, (size_t)(Dg + 2 * (size_t)G) * WA + gi,
                      (l0 != 0.0 ? 1u : 0u) | (l1 != 0.0 ? 2u : 0u) | (l2 != 0.0 ? 4u : 0u), mismatch);
  }
}

// ---- global rows, part 1: the dense block A (one warp per row) -----------------------------------
template <int FILL>
__device__ __forceinline__ void csr_A_rows_body(int bid, const double* __restrict__ A, int Dg, int32_t* __restrict__ cntA,
             const int32_t* __restrict__ indptr, int32_t* __restrict__ indices,
             double* __restrict__ data, uint32_t* __restrict__ mask, const MismatchFlag mismatch) {
  const int lane = threadIdx.x & 31;
  const int r = bid * 8 + (threadIdx.x >> 5);
  if (r >= Dg) return;
  const double* a = A + (size_t)r * Dg;
  int64_t base = FILL ? indptr[r] : 0;
  int count = 0;
  for (int c0 = 0; c0 < Dg; c0 += 32) {
    const int c = c0 + lane;
    const double v = (c < Dg) ? a[c] : 0.0;
    const bool nz = (v != 0.0);
    const unsigned m = __ballot_sync(0xffffffffu, nz);
    if (FILL && nz) {
      const int off = __popc(m & ((1u << lane) - 1));
      if (FILL == 1) indices[base + off] = c;
      data[base + off] = v;
    }
    if (FILL && lane == 0) mask_word<FILL>(mask, (size_t)r * ((Dg + 31) >> 5) + (c0 >> 5), m, mismatch);
    base += __popc(m);
    count += __popc(m);
  }
  if (!FILL && lane == 0) cntA[r] = count;
}

// ---- global rows, part 2: columns of B, chunked over groups -----------------------------------
// chunkcnt / chunkoff: (nchunk, 2*Dg) int32, column c = side*Dg + r.
template <int FILL>
__device__ __forceinline__ void csr_B_cols_body(int bid, const double* __restrict__ B, int Dg, int G, int CG, int32_t* __restrict__ chunkcnt,
             const int32_t* __restrict__ chunkoff, const int32_t* __restrict__ cntA,
             const int32_t* __restrict__ coltot, const int32_t* __restrict__ indptr,
             int32_t* __restrict__ indices, double* __restrict__ data) {
  extern __shared__ __align__(16) double tile[];   // CG x (2*Dg + 1)  (+1: conflict-free column reads)
  const int ncol = 2 * Dg, ld = ncol + 1;
  const int chunk = bid;
  const int g0 = chunk * CG;
  const int ng = (G - g0 < CG) ? (G - g0) : CG;
  const double* src = B + (size_t)g0 * ncol;
  for (int e = threadIdx.x; e < ng * ncol; e += blockDim.x) {
    const int gl = e / ncol, c = e - gl * ncol;
    tile[gl * ld + c] = src[e];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = warp; c < ncol; c += 8) {
    const int side = (c >= Dg) ? 1 : 0, r = c - side * Dg;
    int64_t base = 0;
    if (FILL)
      base = (int64_t)indptr[r] + cntA[r] + (side ? coltot[r] : 0) + chunkoff[(size_t)chunk * ncol + c];
    // the fill pass records where this (chunk, column) segment starts: the refill then needs ONE index load
    // per segment (chunkcnt is the segment-base array in that launch)
    if (FILL == 1 && lane == 0 && chunkcnt) chunkcnt[(size_t)chunk * ncol + c] = (int32_t)base;
    int count = 0;
    for (int s0 = 0; s0 < ng; s0 += 32) {
      const int gl = s0 + lane;
      const double v = (gl < ng) ? tile[gl * ld + c] : 0.0;
      const bool nz = (v != 0.0);
      const unsigned m = __ballot_sync(0xffffffffu, nz);
      if (FILL && nz) {
        const int off = __popc(m & ((1u << lane) - 1));
        if (FILL == 1) indices[base + off] = Dg + side * G + g0 + gl;
        data[base + off] = v;
      }
      base += __popc(m);
      count += __popc(m);
    }
    if (!FILL && lane == 0) chunkcnt[(size_t)chunk * ncol + c] = count;
  }
}

// ---- refill of one chunk of CG groups: border columns AND local rows from one staged tile -------------
// B is read from HBM once (the full export reads it twice: transposed for the global rows, row-wise for the
// local rows).  The index words the chunk needs are fetched into shared memory BEFORE the tile is awaited,
// so no warp walks a chain of dependent loads per column or row:
//   sseg  (2 Dg)   start of every (chunk, column) segment of a global row (recorded by the fill pass)
//   sbase (2 CG)   indptr of the chunk's local rows
//   sl    (CG x 4) the local 2x2 block | recorded 3-bit mask
//   spos  (2 Dg)   uniform chunks: per side, the recorded-nonzero columns of a local row in order
// Usual case ("uniform"): all local rows of a side have the SAME recorded zero mask in this chunk (the
// structural zeros: d2/d u d mu.info and d2/d u.info d mu.mean) and all 2x2 blocks the same 3-bit mask.
// Then every position is known without looking at the values: a local-row entry sits at base + spos[c], a
// border-column segment holds either all of the chunk's groups in order or none, nothing is compacted, and
// the check is "zero exactly where the record says zero".  Otherwise ballots compact the values and the
// masks are compared word by word.  CG is a power of two <= 32 (a warp packs 32 / CG columns per pass).
// The tile rows are 2 Dg + 2 doubles apart: bulk async copies (TMA) need 16-byte aligned destinations, and the
// even stride costs a two-way bank conflict on the column reads, which is noise next to the copies it saves.
__host__ __device__ inline size_t csr_refill_smem(int Dg, int CG) {
  return sizeof(double) * ((size_t)CG * (2 * Dg + 2) + (size_t)CG * 4 + 1) +
         sizeof(int32_t) * ((size_t)4 * Dg + 2 * CG + 2 * ((Dg + 31) / 32) + 4);
}
__device__ __forceinline__ void csr_refill_chunk_body(int chunk, const double* __restrict__ B, const double* __restrict__ L,
                 int Dg, int G, int CG, const int32_t* __restrict__ segbase, const int32_t* __restrict__ indptr,
                 double* __restrict__ data, const uint32_t* __restrict__ mask, const MismatchFlag mismatch) {
  extern __shared__ __align__(16) double tile[];   // CG x (2*Dg + 2)
  const int ncol = 2 * Dg, ld = ncol + 2;
  const int WA = (Dg + 31) >> 5;
  double* sl = tile + (size_t)CG * ld;
  unsigned long long* mbar = (unsigned long long*)(sl + (size_t)CG * 4);
  int32_t* sseg = (int32_t*)(mbar + 1);
  int32_t* sbase = sseg + ncol;
  int32_t* spos = sbase + 2 * CG;
  uint32_t* spm = (uint32_t*)(spos + ncol);      // [2][WA] mask of the first row of each side | [2*WA + 0] L mask
  const int g0 = chunk * CG;
  const int ng = (G - g0 < CG) ? (G - g0) : CG;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t maskL = ((size_t)Dg + 2 * (size_t)G) * WA;
  // --- tile: one bulk async copy per group row (warp 0 issues them; nobody touches a register for it) ---
  const unsigned bar = smem_u32(mbar);
  if (warp == 0) {
    if (lane == 0) {
      mbar_init(bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
      mbar_arrive_expect_tx(bar, (unsigned)(ng * ncol * sizeof(double)));
    }
    __syncwarp();
    if (lane < ng)
      bulk_g2s(smem_u32(tile + lane * ld), B + ((size_t)g0 + lane) * ncol, (unsigned)(ncol * sizeof(double)), bar);
  }
  // --- metadata (independent of the tile) ---
  bool uniform = true;
  for (int t = tid; t < ncol; t += 256) sseg[t] = segbase[(size_t)chunk * ncol + t];
  {
    // every recorded mask word of the chunk's local rows in ONE round trip (one word per thread at Dg <= 128)
    const uint32_t* mfirst0 = mask + ((size_t)Dg + g0) * WA;                  // first row of side 0 / 1
    const uint32_t* mfirst1 = mask + ((size_t)Dg + (size_t)G + g0) * WA;
    const int nw = ng * WA;                  // words per side (consecutive in memory: rows g0 .. g0 + ng - 1)
    for (int t = tid; t < 2 * nw; t += 256) {
      const int side = t >= nw ? 1 : 0, o = t - side * nw;
      const uint32_t* mf = side ? mfirst1 : mfirst0;
      const uint32_t m = mf[o];
      const int k = o % WA;
      uniform &= (m == mf[k]);
      if (o < WA) spm[side * WA + o] = m;
    }
    const int32_t* ip0 = indptr + (size_t)Dg + g0;
    for (int t = tid; t < 2 * ng; t += 256) sbase[t] = (t >= ng) ? ip0[(size_t)G + t - ng] : ip0[t];
  }
  {
    const uint32_t lm0 = mask[maskL + g0];
    if (tid == 0) spm[2 * WA] = lm0;
    for (int t = tid; t < ng * 4; t += 256) {
      const int gl = t >> 2, k = t & 3;
      double v;
      if (k < 3) v = L[(size_t)(g0 + gl) * 3 + k];
      else {
        const uint32_t lm = mask[maskL + g0 + gl];
        uniform &= (lm == lm0);
        v = (double)lm;
      }
      sl[t] = v;
    }
  }
  uniform = __syncthreads_and(uniform ? 1 : 0) != 0;
  mbar_wait(bar, 0);               // the tile has landed (the barrier above ordered the mbarrier's init)
  bool bad = false;
  const int per = 32 / CG;                       // columns per warp pass
  const int sub = lane / CG, glc = lane - sub * CG;
  if (uniform) {
    // per side: the list of recorded-nonzero columns in order (spos[side * Dg + j] = column of the j-th entry
    // of a local row), and sseg[c] = -1 for a recorded-zero column
    for (int t = tid; t < ncol; t += 256) {
      const int side = t >= Dg ? 1 : 0, c = t - side * Dg;
      const uint32_t* pm = spm + side * WA;
      int p = 0;
      for (int w = 0; w < (c >> 5); ++w) p += __popc(pm[w]);
      const uint32_t mw = pm[c >> 5];
      p += __popc(mw & ((1u << (c & 31)) - 1u));
      if ((mw >> (c & 31)) & 1u) spos[side * Dg + p] = c;
      else sseg[t] = -1;
    }
    __syncthreads();
    // --- border columns: all of the chunk's groups in order, or none; EVERY tile element is checked here ---
    if (glc < ng) {
      const double* tp = tile + glc * ld;
      for (int c = warp * per + sub; c < ncol; c += 8 * per) {
        const double v = tp[c];
        const int sg = sseg[c];
        bad |= ((v != 0.0) != (sg >= 0));
        if (sg >= 0) data[sg + glc] = v;
      }
    }
    // --- local rows: the recorded border entries in order, then the recorded entries of the 2x2 block ---
    const uint32_t lm = spm[2 * WA];
    int nzs[2] = {0, 0};                       // recorded border entries per local row of side 0 / 1
    for (int w = 0; w < WA; ++w) { nzs[0] += __popc(spm[w]); nzs[1] += __popc(spm[WA + w]); }
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const int nz = nzs[side];
      const bool rec = (lm >> (side + (lane & 1))) & 1u;
      const int lpos = nz + ((lane == 1) ? (int)((lm >> side) & 1u) : 0);
      for (int gl = warp; gl < ng; gl += 8) {
        double* d = data + sbase[side * ng + gl];
        const double* b = tile + gl * ld + side * Dg;
        const int32_t* pc = spos + side * Dg;
        for (int j = lane; j < nz; j += 32) d[j] = b[pc[j]];
        if (lane < 2) {
          // side 0: (mm, mi) = bits 0, 1 of the 3-bit mask; side 1: (mi, ii) = bits 1, 2
          const double v = sl[gl * 4 + side + lane];
          bad |= ((v != 0.0) != rec);
          if (rec) d[lpos] = v;
        }
      }
    }
  } else {
    const unsigned cgmask = (CG == 32) ? 0xffffffffu : ((1u << CG) - 1u);
    for (int cb = warp * per; cb < ncol; cb += 8 * per) {
      const int c = cb + sub;
      const bool on = (c < ncol) && (glc < ng);
      const double v = on ? tile[glc * ld + c] : 0.0;
      const bool nz = (v != 0.0);
      const unsigned m = (__ballot_sync(0xffffffffu, nz) >> (sub * CG)) & cgmask;
      if (nz) data[(int64_t)sseg[c] + __popc(m & ((1u << glc) - 1u))] = v;
    }
    for (int rr = warp; rr < 2 * ng; rr += 8) {
      const int side = rr >= ng ? 1 : 0, gl = rr - side * ng;
      const size_t wg = (size_t)side * G + g0 + gl;
      int64_t base = sbase[rr];
      const double* b = tile + gl * ld + side * Dg;
      for (int c0 = 0; c0 < Dg; c0 += 32) {
        const int c = c0 + lane;
        const double v = (c < Dg) ? b[c] : 0.0;
        const bool nz = (v != 0.0);
        const unsigned m = __ballot_sync(0xffffffffu, nz);
        if (nz) data[base + __popc(m & ((1u << lane) - 1u))] = v;
        bad |= (m != mask[((size_t)Dg + wg) * WA + (c0 >> 5)]);
        base += __popc(m);
      }
      if (lane == 0) {
        const double l0 = sl[gl * 4], l1 = sl[gl * 4 + 1], l2 = sl[gl * 4 + 2];
        const double va = side ? l1 : l0, vb = side ? l2 : l1;
        if (va != 0.0) data[base++] = va;
        if (vb != 0.0) data[base] = vb;
        if (side == 0) {
          const unsigned lmc = (l0 != 0.0 ? 1u : 0u) | (l1 != 0.0 ? 2u : 0u) | (l2 != 0.0 ? 4u : 0u);
          bad |= (lmc != (unsigned)sl[gl * 4 + 3]);
        }
      }
    }
  }
  if (bad) {
    *mismatch.dev = 1;
    if (mismatch.host) *(volatile int*)mismatch.host = 1;
  }
}

// The three block-uniform roles of a count (FILL = 0) or fill (FILL = 1) pass, walked with a grid stride (a
// conditional export is launched with a capped grid: its usual fate is an early return).
template <int FILL>
__device__ __forceinline__ void csr_roles(const double* A, const double* B, const double* L, int Dg, int G, int CG, int nA,
           int nB, int32_t* cntA, int32_t* chunkcnt, const int32_t* chunkoff, const int32_t* coltot, int32_t* rowcnt,
           const int32_t* indptr, int32_t* indices, double* data, uint32_t* mask, const MismatchFlag mismatch) {
  const int total = nA + nB + (int)((2 * (int64_t)G + 7) / 8);
  for (int vb = blockIdx.x; vb < total; vb += gridDim.x) {
    if (vb < nA) {
      csr_A_rows_body<FILL>(vb, A, Dg, cntA, indptr, indices, data, mask, mismatch);
    } else if (vb < nA + nB) {
      csr_B_cols_body<FILL>(vb - nA, B, Dg, G, CG, chunkcnt, chunkoff, cntA, coltot, indptr, indices, data);
      __syncthreads();      // the staging tile is reused by the next role of this CTA
    } else {
      csr_local_rows_body<FILL>(vb - nA - nB, B, L, Dg, G, rowcnt, indptr, indices, data, mask, mismatch);
    }
  }
}

// One launch per phase: blocks [0, nA) take the rows of A, the next nB blocks a chunk of B each,
// the rest the local rows (block-uniform roles; only the B role uses the dynamic shared memory).
// FILL = 0 count, 1 fill (and record the zero mask), 2 refill: data only with the cached offsets, the
// zero mask compared with the recorded one.
template <int FILL>
__global__ void __launch_bounds__(256)
k_csr_pass(const double* __restrict__ A, const double* __restrict__ B, const double* __restrict__ L,
           int Dg, int G, int CG, int nA, int nB, int32_t* __restrict__ cntA,
           int32_t* __restrict__ chunkcnt, const int32_t* __restrict__ chunkoff,
           const int32_t* __restrict__ coltot, int32_t* __restrict__ rowcnt,
           const int32_t* __restrict__ indptr, int32_t* __restrict__ indices, double* __restrict__ data,
           uint32_t* __restrict__ mask, const MismatchFlag mismatch) {
  const int bid = blockIdx.x;
  if constexpr (FILL == 2) {
  if (bid >= nA) {
    // Refill: the border columns and the local rows need B and L only.  Those are written by k_finish, and
    // every path to this kernel passes k_global_post (or a kernel launched even later), which signals its
    // dependents after its own wait: B and L are complete when this CTA starts, so it runs ahead of the
    // wait, behind k_global_post (one CTA), which is still finishing A.  Nothing written here is read by
    // a kernel that might still be running in front of this one.
    pdl_launch_dependents();
    if (chunkcnt != nullptr) {
      // merged refill (large G), grid = nA + nB: every chunk block writes its border segments and its local rows (chunkcnt = segment bases)
      csr_refill_chunk_body(bid - nA, B, L, Dg, G, CG, chunkcnt, indptr, data, mask, mismatch);
    } else if (bid < nA + nB) {
      csr_B_cols_body<FILL>(bid - nA, B, Dg, G, CG, chunkcnt, chunkoff, cntA, coltot, indptr, indices, data);
    } else {
      csr_local_rows_body<FILL>(bid - nA - nB, B, L, Dg, G, rowcnt, indptr, indices, data, mask, mismatch);
    }
    pdl_wait();        // completion of this kernel still implies completion of its prerequisite
    return;
  }
  }
  pdl_sync();
  csr_roles<FILL>(A, B, L, Dg, G, CG, nA, nB, cntA, chunkcnt, chunkoff, coltot, rowcnt, indptr, indices, data, mask,
                  mismatch);
}

// exclusive scan of chunkcnt over chunks, one CTA per column; coltot[c] = column total
__device__ __forceinline__ void csr_colscan_body(int c, const int32_t* chunkcnt, int32_t* chunkoff, int32_t* coltot,
                                                 int nchunk, int ncol);
__global__ void __launch_bounds__(256)
k_csr_colscan(const int32_t* __restrict__ chunkcnt, int32_t* __restrict__ chunkoff,
              int32_t* __restrict__ coltot, int nchunk, int ncol) {
  pdl_sync();
  csr_colscan_body(blockIdx.x, chunkcnt, chunkoff, coltot, nchunk, ncol);
}
__device__ __forceinline__ void csr_colscan_body(int c, const int32_t* chunkcnt, int32_t* chunkoff, int32_t* coltot,
                                                 int nchunk, int ncol) {
  __shared__ int wsum[8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int carry = 0;
  for (int s0 = 0; s0 < nchunk; s0 += 256) {
    const int i = s0 + threadIdx.x;
    const int cnt = (i < nchunk) ? chunkcnt[(size_t)i * ncol + c] : 0;
    int v = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    __syncthreads();
    if (lane == 31) wsum[wid] = v;
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      if (w < wid) off += wsum[w];
      tot += wsum[w];
    }
    if (i < nchunk) chunkoff[(size_t)i * ncol + c] = carry + off + v - cnt;
    carry += tot;
  }
  if (threadIdx.x == 0) coltot[c] = carry;
}

// rowcnt[r] for the global rows
__global__ void k_csr_global_rowcnt(const int32_t* __restrict__ cntA,
                                    const int32_t* __restrict__ coltot, int Dg,
                                    int32_t* __restrict__ rowcnt) {
  pdl_sync();
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < Dg) rowcnt[r] = cntA[r] + coltot[r] + coltot[Dg + r];
}

// ---- exclusive scan of rowcnt (n entries) into indptr (n+1 entries), 3 phases --------------------
__device__ __forceinline__ void scan_sum_body(int vb, const int32_t* cnt, int64_t n, int64_t* blk);
__device__ __forceinline__ void scan_apply_body(int vb, int nblk, const int32_t* cnt, int64_t n, const int64_t* blk,
                                                const int64_t* total, int32_t* indptr);
__global__ void __launch_bounds__(256)
k_scan_sum(const int32_t* __restrict__ cnt, int64_t n, int64_t* __restrict__ blk) {
  pdl_sync();
  scan_sum_body(blockIdx.x, cnt, n, blk);
}
__device__ __forceinline__ void scan_sum_body(int vb, const int32_t* cnt, int64_t n, int64_t* blk) {
  __shared__ double red[32];
  const int64_t b0 = (int64_t)vb * kScanChunk;
  long long s = 0;
  for (int i = threadIdx.x; i < kScanChunk; i += blockDim.x)
    if (b0 + i < n) s += cnt[b0 + i];
  // counts < 2^31 each and at most 2048 per chunk: exact in double
  const double t = block_sum((double)s, red);
  if (threadIdx.x == 0) blk[vb] = (int64_t)t;
}

__device__ __forceinline__ void scan_top_body(int64_t* blk, int nblk, int64_t* total, int64_t* nnz_out);
__global__ void k_scan_top(int64_t* __restrict__ blk, int nblk, int64_t* __restrict__ total,
                           int64_t* __restrict__ nnz_out) {
  pdl_sync();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  scan_top_body(blk, nblk, total, nnz_out);
}
__device__ __forceinline__ void scan_top_body(int64_t* blk, int nblk, int64_t* total, int64_t* nnz_out) {
  int64_t run = 0;
  for (int i = 0; i < nblk; ++i) {
    const int64_t c = blk[i];
    blk[i] = run;
    run += c;
  }
  *total = run;
  if (nnz_out) *nnz_out = run;
}

__global__ void __launch_bounds__(256)
k_scan_apply(const int32_t* __restrict__ cnt, int64_t n, const int64_t* __restrict__ blk,
             const int64_t* __restrict__ total, int32_t* __restrict__ indptr) {
  pdl_sync();
  scan_apply_body(blockIdx.x, gridDim.x, cnt, n, blk, total, indptr);
}
__device__ __forceinline__ void scan_apply_body(int vb, int nblk, const int32_t* cnt, int64_t n, const int64_t* blk,
                                                const int64_t* total, int32_t* indptr) {
  __shared__ int wsum[8];
  const int64_t b0 = (int64_t)vb * kScanChunk;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  int64_t carry = blk[vb];
  for (int s0 = 0; s0 < kScanChunk; s0 += 256) {
    const int64_t i = b0 + s0 + threadIdx.x;
    const int c = (i < n) ? cnt[i] : 0;
    int v = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, o);
      if (lane >= o) v += t;
    }
    __syncthreads();
    if (lane == 31) wsum[wid] = v;
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      if (w < wid) off += wsum[w];
      tot += wsum[w];
    }
    if (i < n) indptr[i] = (int32_t)(carry + off + v - c);
    carry += tot;
  }
  if (vb == nblk - 1 && threadIdx.x == 0) indptr[n] = (int32_t)(*total);
}

// ---- the whole export as ONE launch: the conditional export behind a refill ---------------------------
// A refill is followed by a full export that runs only if the refill found the zero pattern changed.  As four
// dependent launches its usual fate -- four early returns -- still costs four launch hops per evaluation; as
// one launch of co-resident CTAs (kCoopCtasPerSM per SM; ensure_csr_scratch checks that they fit) that walk the
// same phases between grid-wide barriers it costs one.  A first export stays the chain of launches: there every
// phase gets a grid of its own size, and the fixed grid of co-resident CTAs is slower (DESIGN.md section 3).
// bar[0]: arrivals (monotonic over the phases of one launch), bar[1]: CTAs that left; the last one resets both.
// A barrier that does not complete within ~2 s gives up (the export is then wrong, which the caller's
// status check reports: mismatch stays raised) instead of hanging the device.
constexpr int kCoopCtasPerSM = 2;
__device__ __forceinline__ bool grid_barrier(unsigned* bar, unsigned target) {
  __shared__ int ok;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(bar, 1u);
    unsigned seen = 0, spins = 0;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(bar) : "memory");
      if (seen >= target) break;
      __nanosleep(100);
    } while (++spins < (1u << 24));
    ok = (seen >= target);
    __threadfence();
  }
  __syncthreads();
  return ok != 0;
}
__global__ void __launch_bounds__(256)
k_csr_export_coop(const double* A, const double* B, const double* L, int Dg, int G, int CG, int nA, int nB,
                  int32_t* cntA, int32_t* chunkcnt, int32_t* chunkoff, int32_t* coltot, int32_t* segbase,
                  int32_t* rowcnt, int64_t D, int64_t* blk, int nblk, int32_t* indptr, int32_t* indices, double* data,
                  int64_t* nnz_out, uint32_t* mask, unsigned* bar, const int* __restrict__ run_if) {
  pdl_sync();
  if (*run_if == 0) return;
  const unsigned nc = gridDim.x;
  unsigned phase = 0;
  const MismatchFlag none{nullptr, nullptr};
  bool ok = true;
  // counts
  csr_roles<0>(A, B, L, Dg, G, CG, nA, nB, cntA, chunkcnt, nullptr, nullptr, rowcnt, nullptr, nullptr, nullptr, nullptr, none);
  ok = ok && grid_barrier(bar, ++phase * nc);
  // column scans (or no groups: zero column totals)
  if (G > 0) {
    for (int c = blockIdx.x; c < 2 * Dg; c += nc) { csr_colscan_body(c, chunkcnt, chunkoff, coltot, nB, 2 * Dg); __syncthreads(); }
  } else if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < 2 * Dg; c += blockDim.x) coltot[c] = 0;
  }
  ok = ok && grid_barrier(bar, ++phase * nc);
  if (blockIdx.x == 0)
    for (int r = threadIdx.x; r < Dg; r += blockDim.x) rowcnt[r] = cntA[r] + coltot[r] + coltot[Dg + r];
  ok = ok && grid_barrier(bar, ++phase * nc);
  for (int vb = blockIdx.x; vb < nblk; vb += nc) { scan_sum_body(vb, rowcnt, D, blk); __syncthreads(); }
  ok = ok && grid_barrier(bar, ++phase * nc);
  if (blockIdx.x == 0 && threadIdx.x == 0) scan_top_body(blk, nblk, blk + nblk, nnz_out);
  ok = ok && grid_barrier(bar, ++phase * nc);
  for (int vb = blockIdx.x; vb < nblk; vb += nc) { scan_apply_body(vb, nblk, rowcnt, D, blk, blk + nblk, indptr); __syncthreads(); }
  ok = ok && grid_barrier(bar, ++phase * nc);
  // fill (records the zero mask and the segment bases for later refills)
  if (ok)
    csr_roles<1>(A, B, L, Dg, G, CG, nA, nB, cntA, segbase, chunkoff, coltot, nullptr, indptr, indices, data, mask, none);
  // leave: the last CTA resets the barrier words for the next launch
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(bar + 1, 1u) == nc - 1) {
      bar[0] = 0;
      bar[1] = 0;
      __threadfence();
    }
  }
}

// Small problems (D <= kIndptrOneCta): row counts of the global rows + exclusive scan + nnz in ONE
// CTA -- replaces k_csr_global_rowcnt, k_scan_sum, k_scan_top, k_scan_apply (four dependent launches,
// each a few microseconds of latency on a 20k-element array).
constexpr int64_t kIndptrOneCta = 262144;
__global__ void __launch_bounds__(1024)
k_csr_indptr_small(const int32_t* __restrict__ cntA, const int32_t* __restrict__ coltot, int Dg,
                   const int32_t* __restrict__ rowcnt, int64_t n, int32_t* __restrict__ indptr,
                   int64_t* __restrict__ nnz_out) {
  pdl_sync();
  __shared__ int wsum[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  long long carry = 0;
  constexpr int U = 8;     // tiles in flight: the loads of U tiles are issued before the first scan
  for (int64_t s0 = 0; s0 < n; s0 += 1024 * U) {
    int cs[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = s0 + (int64_t)u * 1024 + threadIdx.x;
      cs[u] = 0;
      if (i < n) cs[u] = (i < Dg) ? cntA[i] + coltot[i] + coltot[Dg + i] : rowcnt[i];
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = s0 + (int64_t)u * 1024 + threadIdx.x;
      if (s0 + (int64_t)u * 1024 >= n) break;
      const int c = cs[u];
      int v = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
      }
      __syncthreads();
      if (lane == 31) wsum[wid] = v;
      __syncthreads();
      const int ws = wsum[lane];                 // every warp scans the 32 warp totals
      int wv = ws;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, wv, o);
        if (lane >= o) wv += t;
      }
      const int tot = __shfl_sync(0xffffffffu, wv, 31);
      const int off = __shfl_sync(0xffffffffu, wv - ws, wid);
      if (i < n) indptr[i] = (int32_t)(carry + off + v - c);
      carry += tot;
    }
  }
  if (threadIdx.x == 0) {
    indptr[n] = (int32_t)carry;
    if (nnz_out) *nnz_out = carry;
  }
}

static int csr_chunk_groups(int Dg) {
  // stage CG x (2 Dg + 1) doubles in <= 54 KB of shared memory
  // (4 CTAs of 8 warps per SM; a power of two <= 32 -- the refill packs 32 / cg columns per ballot)
  int cg = 32;
  while (cg > 4 && csr_refill_smem(Dg, cg) > 55 * 1024 + 512) cg >>= 1;
  return cg;
}

static int ensure_csr_scratch(lrvb_glmm* h) {
  if (h->rowcnt) return LRVB_OK;
  const int Dg = h->Dg, G = h->G;
  const int64_t D = h->D;
  const int nblk = cdiv(D, kScanChunk);
  const int CG = csr_chunk_groups(Dg);
  const int nchunk = cdiv(G, CG) > 0 ? cdiv(G, CG) : 1;
  // raised first: once h->rowcnt is set, this function returns at its first line
  const size_t smem = sizeof(double) * (size_t)CG * (2 * Dg + 1);
  LRVB_TRY(raise_smem_limit(k_csr_pass<0>, smem));
  LRVB_TRY(raise_smem_limit(k_csr_pass<1>, smem));
  LRVB_TRY(raise_smem_limit(k_csr_pass<2>, csr_refill_smem(Dg, CG)));
  LRVB_TRY(raise_smem_limit(k_csr_export_coop, smem));
  // the grid barriers of the one-launch export wait for every CTA of its grid: all of them must be resident at once
  int fit = 0;
  LRVB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&fit, k_csr_export_coop, 256, smem));
  if (fit < kCoopCtasPerSM) {
    set_error("CSR export: %d CTAs of k_csr_export_coop (%zu B of shared memory) fit per SM, %d needed", fit, smem,
              kCoopCtasPerSM);
    return LRVB_ECUDA;
  }
  h->csr_cg = CG;
  h->csr_nchunk = nchunk;
  LRVB_CUDA(cudaMalloc((void**)&h->rowcnt, sizeof(int32_t) * (size_t)(D + 1)));
  LRVB_CUDA(cudaMalloc((void**)&h->scanblk, sizeof(int64_t) * ((size_t)nblk + 2)));
  // cntA (Dg) | coltot (2Dg) | chunkcnt (nchunk*2Dg) | chunkoff (nchunk*2Dg) | segbase (nchunk*2Dg)
  LRVB_CUDA(cudaMalloc((void**)&h->csrwork,
                       sizeof(int32_t) * ((size_t)3 * Dg + (size_t)6 * Dg * nchunk + 4)));
  // zero mask of the last full export: A (Dg x WA) | B (2G x WA) | L (G) words
  const size_t WA = ((size_t)Dg + 31) / 32;
  LRVB_CUDA(cudaMalloc((void**)&h->csrmask, sizeof(uint32_t) * ((size_t)(Dg + 2 * (size_t)G) * WA + (size_t)G + 1)));
  // the grid-barrier words of the one-launch export (the four spare words behind the scan scratch)
  LRVB_CUDA(cudaMemset(h->csrwork + (size_t)3 * Dg + (size_t)6 * Dg * nchunk, 0, sizeof(int32_t) * 4));
  return LRVB_OK;
}

}  // namespace lrvb

using namespace lrvb;

extern "C" {

int lrvb_glmm_hessian_csr_capacity(const lrvb_glmm* h, int64_t* capacity) {
  LRVB_REQUIRE(h != nullptr && capacity != nullptr, "lrvb_glmm_hessian_csr_capacity: NULL argument");
  *capacity = (int64_t)h->Dg * h->Dg + 4 * (int64_t)h->Dg * h->G + 4 * (int64_t)h->G;
  return LRVB_OK;
}

static int csr_full_export(lrvb_glmm* h, int32_t* indptr_dev, int32_t* indices_dev, double* data_dev,
                           int64_t capacity, int64_t* nnz_dev, const int* run_if, const char* who, void* stream) {
  LRVB_REQUIRE(h != nullptr && indptr_dev && indices_dev && data_dev && nnz_dev, "%s: NULL argument", who);
  if (!h->hess_valid) {
    set_error("%s: no Hessian cached (call lrvb_glmm_eval with order 2)", who);
    return LRVB_ESTATE;
  }
  int64_t cap = 0;
  lrvb_glmm_hessian_csr_capacity(h, &cap);
  LRVB_REQUIRE(capacity >= cap, "%s: capacity %lld < structural bound %lld", who, (long long)capacity, (long long)cap);
  LRVB_REQUIRE(cap < (int64_t)2147483647, "Hessian may have %lld nonzeros: exceeds int32 CSR indices",
               (long long)cap);
  LRVB_TRY(ensure_csr_scratch(h));
  cudaStream_t st = (cudaStream_t)stream;
  const int Dg = h->Dg, G = h->G, CG = h->csr_cg, nchunk = h->csr_nchunk;
  const int64_t D = h->D;
  const int nblk = cdiv(D, kScanChunk);
  int32_t* cntA = h->csrwork;
  int32_t* coltot = cntA + Dg;
  int32_t* chunkcnt = coltot + 2 * Dg;
  int32_t* chunkoff = chunkcnt + (size_t)2 * Dg * nchunk;
  int64_t* blk = (int64_t*)h->scanblk;
  const size_t smem = sizeof(double) * (size_t)CG * (2 * Dg + 1);

  const int nA = cdiv(Dg, 8), nB = (G > 0) ? nchunk : 0, nL = (G > 0) ? cdiv(2 * (int64_t)G, 8) : 0;
  if (run_if) {
    // the conditional export behind a refill: one launch of co-resident CTAs
    int32_t* segb = chunkoff + (size_t)2 * Dg * nchunk;
    unsigned* bar = (unsigned*)(segb + (size_t)2 * Dg * nchunk);
    LRVB_CUDA(launch_pdl(k_csr_export_coop, dim3(kCoopCtasPerSM * kNumSMs), dim3(256), smem, st, (const double*)h->A,
                         (const double*)h->B, (const double*)h->L, Dg, G, CG, nA, nB, cntA, chunkcnt, chunkoff, coltot,
                         segb, h->rowcnt, (int64_t)D, blk, nblk, indptr_dev, indices_dev, data_dev, (int64_t*)nnz_dev,
                         h->csrmask, bar, run_if));
    LRVB_CHECK_LAUNCH();
    h->csr_pattern_valid = 1;
    return LRVB_OK;
  }
  // ---- counts: rows of A, columns of B (per chunk) and local rows in one launch ----
  const int pass_grid = nA + nB + nL;
  LRVB_CUDA(launch_pdl(k_csr_pass<0>, dim3(pass_grid), dim3(256), smem, st, h->A, h->B, h->L, Dg, G,
                       CG, nA, nB, cntA, chunkcnt, nullptr, nullptr, h->rowcnt, nullptr, nullptr, nullptr,
                       (uint32_t*)nullptr, MismatchFlag{nullptr, nullptr}));
  LRVB_CHECK_LAUNCH();
  if (G > 0) {
    LRVB_CUDA(launch_pdl(k_csr_colscan, dim3(2 * Dg), dim3(256), 0, st, chunkcnt, chunkoff, coltot, nchunk, 2 * Dg));
    LRVB_CHECK_LAUNCH();
  } else {
    LRVB_CUDA(cudaMemsetAsync(coltot, 0, sizeof(int32_t) * 2 * Dg, st));
  }
  // ---- indptr ----
  if (D <= kIndptrOneCta) {
    LRVB_CUDA(launch_pdl(k_csr_indptr_small, dim3(1), dim3(1024), 0, st, cntA, coltot, Dg, h->rowcnt, D,
                         indptr_dev, (int64_t*)nnz_dev));
    LRVB_CHECK_LAUNCH();
  } else {
    LRVB_CUDA(launch_pdl(k_csr_global_rowcnt, dim3(cdiv(Dg, 256)), dim3(256), 0, st, cntA, coltot, Dg, h->rowcnt));
    LRVB_CHECK_LAUNCH();
    LRVB_CUDA(launch_pdl(k_scan_sum, dim3(nblk), dim3(256), 0, st, h->rowcnt, D, blk));
    LRVB_CHECK_LAUNCH();
    LRVB_CUDA(launch_pdl(k_scan_top, dim3(1), dim3(32), 0, st, blk, nblk, blk + nblk, nnz_dev));
    LRVB_CHECK_LAUNCH();
    LRVB_CUDA(launch_pdl(k_scan_apply, dim3(nblk), dim3(256), 0, st, h->rowcnt, D, blk, blk + nblk, indptr_dev));
    LRVB_CHECK_LAUNCH();
  }
  // ---- fill: the same three roles, one launch; records the zero mask for later refills ----
  int32_t* segbase = chunkoff + (size_t)2 * Dg * nchunk;
  LRVB_CUDA(launch_pdl(k_csr_pass<1>, dim3(pass_grid), dim3(256), smem, st, h->A, h->B, h->L, Dg, G, CG,
                       nA, nB, cntA, segbase, chunkoff, coltot, nullptr, indptr_dev, indices_dev, data_dev,
                       h->csrmask, MismatchFlag{nullptr, nullptr}));
  LRVB_CHECK_LAUNCH();
  h->csr_pattern_valid = 1;
  return LRVB_OK;
}

int lrvb_glmm_hessian_csr(lrvb_glmm* h, int32_t* indptr_dev, int32_t* indices_dev,
                          double* data_dev, int64_t capacity, int64_t* nnz_dev, void* stream) {
  return csr_full_export(h, indptr_dev, indices_dev, data_dev, capacity, nnz_dev, nullptr, "lrvb_glmm_hessian_csr",
                         stream);
}

int lrvb_glmm_hessian_csr_if(lrvb_glmm* h, const int32_t* run_if_dev, int32_t* indptr_dev, int32_t* indices_dev,
                             double* data_dev, int64_t capacity, int64_t* nnz_dev, void* stream) {
  LRVB_REQUIRE(run_if_dev != nullptr, "lrvb_glmm_hessian_csr_if: run_if is NULL");
  return csr_full_export(h, indptr_dev, indices_dev, data_dev, capacity, nnz_dev, (const int*)run_if_dev,
                         "lrvb_glmm_hessian_csr_if", stream);
}

int lrvb_glmm_hessian_csr_refill(lrvb_glmm* h, const int32_t* indptr_dev, double* data_dev, int32_t* mismatch_dev,
                                 int32_t* mismatch_host_mapped, void* stream) {
  LRVB_REQUIRE(h != nullptr && indptr_dev && data_dev && mismatch_dev, "lrvb_glmm_hessian_csr_refill: NULL argument");
  if (!h->hess_valid) {
    set_error("lrvb_glmm_hessian_csr_refill: no Hessian cached (call lrvb_glmm_eval with order 2)");
    return LRVB_ESTATE;
  }
  if (!h->csr_pattern_valid || !h->rowcnt) {
    set_error("lrvb_glmm_hessian_csr_refill: no pattern recorded (call lrvb_glmm_hessian_csr first)");
    return LRVB_ESTATE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int Dg = h->Dg, G = h->G, CG = h->csr_cg, nchunk = h->csr_nchunk;
  int32_t* cntA = h->csrwork;
  int32_t* coltot = cntA + Dg;
  int32_t* chunkcnt = coltot + 2 * Dg;
  int32_t* chunkoff = chunkcnt + (size_t)2 * Dg * nchunk;
  const size_t smem = csr_refill_smem(Dg, CG);
  const int nA = cdiv(Dg, 8), nB = (G > 0) ? nchunk : 0, nL = (G > 0) ? cdiv(2 * (int64_t)G, 8) : 0;
  int32_t* segbase = chunkoff + (size_t)2 * Dg * nchunk;
  // large G: one block per chunk writes border segments and local rows from one staged tile (B read once);
  // small G is launch- and latency-bound, where the many short blocks of the separate roles finish sooner
  const bool merged = G >= 32768;
  LRVB_CUDA(launch_pdl(k_csr_pass<2>, dim3(nA + nB + (merged ? 0 : nL)), dim3(256), smem, st, h->A, h->B, h->L, Dg, G, CG,
                       nA, nB, cntA, merged ? segbase : nullptr, chunkoff, coltot, nullptr, indptr_dev, (int32_t*)nullptr, data_dev,
                       h->csrmask, MismatchFlag{(int*)mismatch_dev, (int*)mismatch_host_mapped}));
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

}  // extern "C"
