// Arrowhead Hessian-vector product, conjugate gradient, Schur complement and the direct
// block-elimination solve behind the LRVB covariance.  fp64, sm_100a, no atomics.
//
// Replaces Objective.fun_free_hvp (SparseObjectives.py:183-187), ConjugateGradientSolver
// .get_hinv_vec (ConjugateGradient.py:81-85 -> scipy.sparse.linalg.cg) and the dense
// cho_factor / cho_solve of ModelSensitivity.py:594-602 for the GLMM Hessian
//      H = [[A, B^T], [B, L]],   A (Dg,Dg) dense, B (G,2,Dg), L = G independent 2x2 blocks.
#include <stdlib.h>
#include <mutex>
#include "common.cuh"

namespace lrvb {

// ---- H v -------------------------------------------------------------------------------------
// One warp per group (grid-stride): local rows of H v, and per-CTA partials of B^T v_l.
// flags[0] != 0 (CG converged) turns the kernel into a no-op.
__global__ void __launch_bounds__(256)
k_hvp_groups(const double* __restrict__ B, const double* __restrict__ L,
             const double* __restrict__ v, double* __restrict__ out,
             double* __restrict__ hvppart, const int* __restrict__ flags, int Dg, int G) {
  pdl_sync();
  if (flags && flags[0]) return;
  extern __shared__ double sm[];
  double* vg = sm;             // Dg
  double* acc = sm + Dg;       // 8 * Dg
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = threadIdx.x; c < Dg; c += blockDim.x) vg[c] = v[c];
  for (int c = threadIdx.x; c < 8 * Dg; c += blockDim.x) acc[c] = 0.0;
  __syncthreads();
  double* my = acc + (size_t)warp * Dg;
  for (int gi = blockIdx.x * 8 + warp; gi < G; gi += gridDim.x * 8) {
    const double vm = v[Dg + gi], vi = v[Dg + G + gi];
    const double* b0 = B + (size_t)gi * 2 * Dg;
    const double* b1 = b0 + Dg;
    double d0 = 0.0, d1 = 0.0;
    for (int c = lane; c < Dg; c += 32) {
      const double x0 = b0[c], x1 = b1[c], vc = vg[c];
      d0 = fma(x0, vc, d0);
      d1 = fma(x1, vc, d1);
      my[c] += x0 * vm + x1 * vi;
    }
    d0 = warp_sum(d0);
    d1 = warp_sum(d1);
    if (lane == 0) {
      const double l0 = L[(size_t)gi * 3], l1 = L[(size_t)gi * 3 + 1], l2 = L[(size_t)gi * 3 + 2];
      out[Dg + gi] = d0 + l0 * vm + l1 * vi;
      out[Dg + G + gi] = d1 + l1 * vm + l2 * vi;
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < Dg; c += blockDim.x) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += acc[(size_t)w * Dg + c];
    hvppart[(size_t)blockIdx.x * Dg + c] = s;
  }
}

// One warp per global row: (A v_g)[r] (optional) + fixed-order sum of the CTA partials.
__global__ void __launch_bounds__(256)
k_hvp_global(const double* __restrict__ A, const double* __restrict__ v,
             const double* __restrict__ hvppart, int npart, double* __restrict__ out,
             const int* __restrict__ flags, int Dg, int include_A) {
  pdl_sync();
  if (flags && flags[0]) return;
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= Dg) return;
  double s = 0.0;
  if (include_A) {
    const double* a = A + (size_t)r * Dg;
    for (int c = lane; c < Dg; c += 32) s = fma(a[c], v[c], s);
  }
  double t = 0.0;
  for (int p = lane; p < npart; p += 32) t += hvppart[(size_t)p * Dg + r];
  s = warp_sum(s);
  t = warp_sum(t);
  if (lane == 0) out[r] = s + t;
}

int launch_hvp(lrvb_glmm* h, const double* v, double* out, int include_A, const int* flags,
               cudaStream_t st) {
  const int Dg = h->Dg, G = h->G;
  const size_t smem = sizeof(double) * 9 * (size_t)Dg;
  LRVB_CUDA(launch_pdl(k_hvp_groups, dim3(h->hvp_grid), dim3(256), smem, st, h->B, h->L, v, out, h->hvppart, flags, Dg, G));
  LRVB_CHECK_LAUNCH();
  LRVB_CUDA(launch_pdl(k_hvp_global, dim3(cdiv(Dg, 8)), dim3(256), 0, st, h->A, v, h->hvppart, h->hvp_grid, out, flags, Dg,
                                             include_A));
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

int ensure_solver_scratch(lrvb_glmm* h) {
  if (h->cgbuf) return LRVB_OK;
  const int Dg = h->Dg, G = h->G;
  h->hvp_grid = cdiv(G, 8 * 4);
  if (h->hvp_grid > 8 * kNumSMs) h->hvp_grid = 8 * kNumSMs;   // latency-bound streaming: 64 warps per SM
  if (h->hvp_grid < 1) h->hvp_grid = 1;
  h->dot_grid = cdiv(h->D, 256 * 8);
  if (h->dot_grid > 2 * kNumSMs) h->dot_grid = 2 * kNumSMs;
  if (h->dot_grid < 1) h->dot_grid = 1;
  LRVB_CUDA(cudaMalloc((void**)&h->hvppart, sizeof(double) * (size_t)h->hvp_grid * Dg));
  LRVB_CUDA(cudaMalloc((void**)&h->dotpart, sizeof(double) * (size_t)h->dot_grid * 4 * 3));
  LRVB_CUDA(cudaMalloc((void**)&h->Linv, sizeof(double) * ((size_t)G * 3 + 1)));
  LRVB_CUDA(cudaMalloc((void**)&h->cgbuf, sizeof(double) * 6 * (size_t)h->D));
  return LRVB_OK;
}

// ---- conjugate gradient ------------------------------------------------------------------------
// Mirrors scipy.sparse.linalg.cg (scipy 1.18 _isolve/iterative.py): atol = rtol * ||b||,
// loop { if ||r|| < atol: done; z = M r; rho = r.z; p = z + (rho/rho_prev) p; q = H p;
//        alpha = rho / p.q; x += alpha p; r -= alpha q }.
// Scalars never visit the host: every CTA re-reduces the per-CTA dot partials in the same fixed
// order, so all CTAs agree bitwise.  flags[0] = converged, flags[1] = completed iterations.
// scal: [0],[1] rho ping-pong, [2] atol, [3] ||r|| at exit.

__device__ __forceinline__ double reduce_parts(const double* __restrict__ part, int n, int stride,
                                               double* red) {
  double v = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) v += part[(size_t)i * stride];
  v = block_sum(v, red);
  __shared__ double bc;
  if (threadIdx.x == 0) bc = v;
  __syncthreads();
  v = bc;
  __syncthreads();
  return v;
}

// partial dot products a.b (slot 0) and c.d (slot 1, optional)
__global__ void __launch_bounds__(256)
k_dot(const double* __restrict__ a, const double* __restrict__ b, const double* __restrict__ c,
      const double* __restrict__ d, int64_t n, double* __restrict__ part,
      const int* __restrict__ flags) {
  pdl_sync();
  if (flags && flags[0]) return;
  __shared__ double red[32];
  double s0 = 0.0, s1 = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    s0 = fma(a[i], b[i], s0);
    if (c) s1 = fma(c[i], d[i], s1);
  }
  s0 = block_sum(s0, red);
  s1 = block_sum(s1, red);
  if (threadIdx.x == 0) {
    part[blockIdx.x * 2] = s0;
    part[blockIdx.x * 2 + 1] = s1;
  }
}

// atol = rtol * ||b||; flags: done if ||b|| == 0
__global__ void k_cg_init(const double* __restrict__ bbpart, int npart, double rtol,
                          double* __restrict__ scal, int* __restrict__ flags) {
  pdl_sync();
  __shared__ double red[32];
  const double bb = reduce_parts(bbpart, npart, 2, red);
  if (threadIdx.x == 0) {
    scal[2] = rtol * sqrt(bb);
    scal[0] = scal[1] = 0.0;
    flags[0] = (bb == 0.0) ? 1 : 0;
    flags[1] = 0;
  }
}

// Top of iteration `it`: convergence test on ||r|| (partials in rrpart slot 0), then z = M r
// and partials of rho = r.z.   precond 0: z = r.  1: block-Jacobi (1/A_ii, inverse 2x2 blocks).
__global__ void __launch_bounds__(256)
k_cg_precond(const double* __restrict__ r, double* __restrict__ z, const double* __restrict__ A,
             const double* __restrict__ Linv, const double* __restrict__ rrpart, int npart,
             double* __restrict__ rzpart, double* __restrict__ scal, int* __restrict__ flags,
             int Dg, int G, int precond) {
  pdl_sync();
  if (flags[0]) return;
  __shared__ double red[32];
  const double rr = reduce_parts(rrpart, npart, 2, red);
  const double rn = sqrt(rr);
  if (rn < scal[2]) {
    // every CTA takes the same branch; the flag is only read by LATER kernels
    if (blockIdx.x == 0 && threadIdx.x == 0) { flags[2] = 1; scal[3] = rn; }
    return;
  }
  const int64_t D = Dg + 2 * (int64_t)G;
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < D;
       i += (int64_t)gridDim.x * blockDim.x) {
    double zi;
    const double ri = r[i];
    if (!precond) zi = ri;
    else if (precond == 2) zi = z[i];        // z = M r was formed by the caller's operator
    else if (i < Dg) zi = ri / A[(size_t)i * Dg + i];
    else if (i < Dg + G) {
      const int64_t gi = i - Dg;
      zi = Linv[gi * 3] * ri + Linv[gi * 3 + 1] * r[i + G];
    } else {
      const int64_t gi = i - Dg - G;
      zi = Linv[gi * 3 + 1] * r[i - G] + Linv[gi * 3 + 2] * ri;
    }
    if (precond != 2) z[i] = zi;
    s = fma(ri, zi, s);
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) {
    rzpart[blockIdx.x * 2] = s;
    rzpart[blockIdx.x * 2 + 1] = 0.0;
  }
}

// z = M r for a caller-supplied preconditioner matrix: CSR (one warp per row) or dense row-major
__global__ void __launch_bounds__(256)
k_cg_m_csr(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
           const double* __restrict__ data, const double* __restrict__ r, double* __restrict__ z, int64_t D,
           const int* __restrict__ flags) {
  pdl_sync();
  if (flags[0]) return;
  const int lane = threadIdx.x & 31;
  for (int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); row < D; row += (int64_t)gridDim.x * 8) {
    double s = 0.0;
    for (int32_t e = indptr[row] + lane; e < indptr[row + 1]; e += 32) s = fma(data[e], r[indices[e]], s);
    s = warp_sum(s);
    if (lane == 0) z[row] = s;
  }
}
__global__ void __launch_bounds__(256)
k_cg_m_dense(const double* __restrict__ M, const double* __restrict__ r, double* __restrict__ z, int64_t D,
             const int* __restrict__ flags) {
  pdl_sync();
  if (flags[0]) return;
  const int lane = threadIdx.x & 31;
  for (int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); row < D; row += (int64_t)gridDim.x * 8) {
    const double* m = M + (size_t)row * D;
    double s = 0.0;
    for (int64_t c = lane; c < D; c += 32) s = fma(m[c], r[c], s);
    s = warp_sum(s);
    if (lane == 0) z[row] = s;
  }
}

// flags[2] (set by k_cg_precond of this iteration) -> flags[0]; separate tiny kernel so that no
// CTA of k_cg_precond can observe the flag it is about to set.
__global__ void k_cg_latch(int* flags) {
  pdl_sync();
  if (flags[2]) flags[0] = 1;
}

// p = z + (rho/rho_prev) p   (p = z on the first iteration); stores rho in scal[it & 1]
__global__ void __launch_bounds__(256)
k_cg_dir(const double* __restrict__ z, double* __restrict__ p, const double* __restrict__ rzpart,
         int npart, double* __restrict__ scal, const int* __restrict__ flags, int64_t D, int it) {
  pdl_sync();
  if (flags[0]) return;
  __shared__ double red[32];
  const double rho = reduce_parts(rzpart, npart, 2, red);
  const double beta = (it > 0) ? rho / scal[(it - 1) & 1] : 0.0;
  if (blockIdx.x == 0 && threadIdx.x == 0) scal[it & 1] = rho;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < D;
       i += (int64_t)gridDim.x * blockDim.x)
    p[i] = (it > 0) ? fma(beta, p[i], z[i]) : z[i];
}

// alpha = rho / p.q ; x += alpha p ; r -= alpha q ; partials of r.r
__global__ void __launch_bounds__(256)
k_cg_update(double* __restrict__ x, double* __restrict__ r, const double* __restrict__ p,
            const double* __restrict__ q, const double* __restrict__ pqpart, int npart,
            double* __restrict__ rrpart, const double* __restrict__ scal, int* __restrict__ flags,
            int64_t D, int it) {
  pdl_sync();
  if (flags[0]) return;
  __shared__ double red[32];
  const double pq = reduce_parts(pqpart, npart, 2, red);
  const double alpha = scal[it & 1] / pq;
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < D;
       i += (int64_t)gridDim.x * blockDim.x) {
    x[i] = fma(alpha, p[i], x[i]);
    const double ri = fma(-alpha, q[i], r[i]);
    r[i] = ri;
    s = fma(ri, ri, s);
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) {
    rrpart[blockIdx.x * 2] = s;
    rrpart[blockIdx.x * 2 + 1] = 0.0;
    if (blockIdx.x == 0) flags[1] = it + 1;
  }
}

// ---- sharded variants (lrvb_glmm_cg_sharded) ---------------------------------------------------------
// z = M r and the partials of r.r (slot 0) and r.z (slot 1) over the entries [lo, D) this rank counts
__global__ void __launch_bounds__(256)
k_cg_precond2(const double* __restrict__ r, double* __restrict__ z, const double* __restrict__ A,
              const double* __restrict__ Linv, double* __restrict__ part, const int* __restrict__ flags,
              int Dg, int G, int precond, int64_t lo) {
  pdl_sync();
  if (flags[0]) return;
  __shared__ double red[32];
  const int64_t D = Dg + 2 * (int64_t)G;
  double s0 = 0.0, s1 = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < D;
       i += (int64_t)gridDim.x * blockDim.x) {
    double zi;
    const double ri = r[i];
    if (!precond) zi = ri;
    else if (i < Dg) zi = ri / A[(size_t)i * Dg + i];
    else if (i < Dg + G) {
      const int64_t gi = i - Dg;
      zi = Linv[gi * 3] * ri + Linv[gi * 3 + 1] * r[i + G];
    } else {
      const int64_t gi = i - Dg - G;
      zi = Linv[gi * 3 + 1] * r[i - G] + Linv[gi * 3 + 2] * ri;
    }
    z[i] = zi;
    if (i >= lo) {
      s0 = fma(ri, ri, s0);
      s1 = fma(ri, zi, s1);
    }
  }
  s0 = block_sum(s0, red);
  s1 = block_sum(s1, red);
  if (threadIdx.x == 0) {
    part[blockIdx.x * 2] = s0;
    part[blockIdx.x * 2 + 1] = s1;
  }
}

// per-CTA partials (npart, 2) -> the two scalars of this rank's message
__global__ void __launch_bounds__(256)
k_cg_fold(const double* __restrict__ part, int npart, double* __restrict__ sc, const int* __restrict__ flags) {
  pdl_sync();
  if (flags && flags[0]) return;
  __shared__ double red[32];
  const double a = reduce_parts(part, npart, 2, red);
  const double b = reduce_parts(part + 1, npart, 2, red);
  if (threadIdx.x == 0) { sc[0] = a; sc[1] = b; }
}

// convergence test on the summed r.r, then p = z + (rho / rho_prev) p with the summed rho = r.z
__global__ void __launch_bounds__(256)
k_cg_dir2(const double* __restrict__ z, double* __restrict__ p, const double* __restrict__ sc,
          double* __restrict__ scal, int* __restrict__ flags, int64_t D, int it) {
  pdl_sync();
  if (flags[0]) return;
  const double rn = sqrt(sc[0]);
  if (rn < scal[2]) {
    // identical on every CTA and every rank: a CTA that starts late and already sees the flag
    // returns at the top, which is the same decision
    if (blockIdx.x == 0 && threadIdx.x == 0) { flags[0] = 1; scal[3] = rn; }
    return;
  }
  const double rho = sc[1];
  const double beta = (it > 0) ? rho / scal[4 + ((it - 1) & 1)] : 0.0;
  if (blockIdx.x == 0 && threadIdx.x == 0) scal[4 + (it & 1)] = rho;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < D;
       i += (int64_t)gridDim.x * blockDim.x)
    p[i] = (it > 0) ? fma(beta, p[i], z[i]) : z[i];
}

// message of the second collective: [q_g (Dg) | sum of the local p.q partials]
__global__ void __launch_bounds__(256)
k_cg_pack(const double* __restrict__ q, const double* __restrict__ part, int npart, double* __restrict__ msg,
          int Dg, const int* __restrict__ flags) {
  pdl_sync();
  if (flags[0]) return;
  __shared__ double red[32];
  for (int i = threadIdx.x; i < Dg; i += blockDim.x) msg[i] = q[i];
  const double s = reduce_parts(part, npart, 2, red);
  if (threadIdx.x == 0) msg[Dg] = s;
}

// q_g <- summed global rows; alpha = rho / (p_g.q_g + summed local part); x += alpha p; r -= alpha q
__global__ void __launch_bounds__(256)
k_cg_update2(double* __restrict__ x, double* __restrict__ r, const double* __restrict__ p,
             double* __restrict__ q, const double* __restrict__ msg, const double* __restrict__ scal,
             int* __restrict__ flags, int64_t D, int Dg, int it) {
  pdl_sync();
  if (flags[0]) return;
  __shared__ double red[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < Dg; i += blockDim.x) s = fma(p[i], msg[i], s);
  s = block_sum(s, red);
  __shared__ double bc;
  if (threadIdx.x == 0) bc = s + msg[Dg];
  __syncthreads();
  const double alpha = scal[4 + (it & 1)] / bc;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < D;
       i += (int64_t)gridDim.x * blockDim.x) {
    const double qi = (i < Dg) ? msg[i] : q[i];
    if (i < Dg) q[i] = qi;
    x[i] = fma(alpha, p[i], x[i]);
    r[i] = fma(-alpha, qi, r[i]);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) flags[1] = it + 1;
}

__global__ void k_axpby(double* __restrict__ out, const double* __restrict__ a, double alpha,
                        const double* __restrict__ b, double beta, int64_t n) {
  pdl_sync();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = alpha * (a ? a[i] : 0.0) + beta * (b ? b[i] : 0.0);
}

// inverse of the local 2x2 blocks, (G,3) as (mm, mi, ii)
__global__ void k_linv(const double* __restrict__ L, double* __restrict__ Linv, int G) {
  pdl_sync();
  const int gi = blockIdx.x * blockDim.x + threadIdx.x;
  if (gi >= G) return;
  const double l0 = L[(size_t)gi * 3], l1 = L[(size_t)gi * 3 + 1], l2 = L[(size_t)gi * 3 + 2];
  const double det = l0 * l2 - l1 * l1;
  Linv[(size_t)gi * 3] = l2 / det;
  Linv[(size_t)gi * 3 + 1] = -l1 / det;
  Linv[(size_t)gi * 3 + 2] = l0 / det;
}

// ---- Schur complement on the FP64 tensor cores ----------------------------------------------------
// S = [A] - sum_g B_g^T L_g^-1 B_g  =  [A] - P^T Q  with P = B as a (2G, Dg) matrix and
// Q = blockdiag(L_g^-1) P.  A warp owns a kRT x kRT rectangle (ri <= rj, the result is symmetric)
// of 8x8 tiles for a chunk of groups; a k-step is 4 rows = 2 groups.
template <int NI, int NJ, bool TRI>
__device__ __forceinline__ void schur_ksteps(double (&acc)[kRT][kRT][2],
                                             const double* __restrict__ B,
                                             const double* __restrict__ Linv, int Dg, int G,
                                             const int (&cola)[kRT], const int (&colb)[kRT],
                                             int k0, int k1, int lr) {
  const int which = lr & 1;
  for (int ks = k0; ks < k1; ++ks) {
    const int gi = 2 * ks + (lr >> 1);
    const bool ok = gi < G;
    const double* b0 = B + (size_t)(ok ? gi : 0) * 2 * Dg;
    const double* b1 = b0 + Dg;
    double w0 = 0.0, w1 = 0.0;
    if (ok) {
      const double* li = Linv + (size_t)gi * 3;
      w0 = which ? li[1] : li[0];
      w1 = which ? li[2] : li[1];
    }
    double fa[kRT], fb[kRT];
#pragma unroll
    for (int i = 0; i < kRT; ++i) {
      if (i < NI) fa[i] = (ok && cola[i] < Dg) ? (which ? b1[cola[i]] : b0[cola[i]]) : 0.0;
      if (i < NJ) fb[i] = (ok && colb[i] < Dg) ? (w0 * b0[colb[i]] + w1 * b1[colb[i]]) : 0.0;
    }
#pragma unroll
    for (int i = 0; i < kRT; ++i)
#pragma unroll
      for (int j = 0; j < kRT; ++j)
        if (i < NI && j < NJ && (!TRI || i <= j)) dmma884(acc[i][j][0], acc[i][j][1], fa[i], fb[j]);
  }
}

__global__ void __launch_bounds__(256)
k_schur(const double* __restrict__ B, const double* __restrict__ Linv, double* __restrict__ part,
        int Dg, int G, int R, int n_jobs, int n_chunk) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  const int wg = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int job = wg % n_jobs, chunk = wg / n_jobs;
  if (chunk >= n_chunk) return;
  // decode job -> (ri, rj), ri <= rj
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
  const int ksteps = (G + 1) / 2;
  const int per = (ksteps + n_chunk - 1) / n_chunk;
  const int k0 = chunk * per, k1 = (k0 + per < ksteps) ? k0 + per : ksteps;
  int ni = DT - kRT * ri, nj = DT - kRT * rj;
  ni = ni > kRT ? kRT : ni;
  nj = nj > kRT ? kRT : nj;
  // compile-time specialised on the live tiles: a predicated-off DMMA still occupies the pipe
#define LRVB_S(NI, NJ, T) schur_ksteps<NI, NJ, T>(acc, B, Linv, Dg, G, cola, colb, k0, k1, lr)
  if (ri == rj) {
    switch (ni) {
      case 1: LRVB_S(1, 1, true); break;
      case 2: LRVB_S(2, 2, true); break;
      case 3: LRVB_S(3, 3, true); break;
      default: LRVB_S(4, 4, true); break;
    }
  } else {
    switch (nj) {   // ri < rj: the row rectangle is always full (ni == kRT)
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
        *reinterpret_cast<double2*>(out + (i * kRT + j) * 64 + crow * 8 + ccol) =
            make_double2(acc[i][j][0], acc[i][j][1]);
}

__global__ void __launch_bounds__(256)
k_schur_finish(const double* __restrict__ part, const double* __restrict__ A,
               double* __restrict__ S, int Dg, int R, int n_jobs, int n_chunk, int include_A) {
  pdl_sync();
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
  for (int p = ps; p < n_chunk; p += 4) s += src[(size_t)p * stride];
  red[ps][e] = s;
  __syncthreads();
  if (ps != 0) return;
  s = (red[0][e] + red[1][e]) + (red[2][e] + red[3][e]);
  const int p = 8 * it + (e >> 3), q = 8 * jt + (e & 7);
  if (p >= Dg || q >= Dg) return;
  if (it == jt && p > q) return;
  const double base = include_A ? A[(size_t)p * Dg + q] : 0.0;
  const double v = base - s;
  S[(size_t)p * Dg + q] = v;
  S[(size_t)q * Dg + p] = v;
}

// ---- in-place inverse of a small SPD matrix, n <= 128: register-resident Gauss-Jordan ----------
// Thread (i, jj) = (tid / 8, tid % 8) keeps the entries j = jj, jj + 8, ... of row i in registers.
// Per pivot k: the (unscaled) pivot row comes from a double-buffered shared row, the pivot-column
// entry of a row from a shuffle inside the 8 lanes that hold the row; one block barrier per pivot.
template <int NQ>   // NQ = ceil(n / 8) register entries per thread
__global__ void __launch_bounds__(1024)
k_spd_inverse_reg(double* __restrict__ S, int n, int* __restrict__ info) {
  pdl_sync();
  __shared__ double rowbuf[2][128];
  const int tid = threadIdx.x, lane = tid & 31;
  const int i = tid >> 3, jj = tid & 7;
  double m[NQ];
#pragma unroll
  for (int q = 0; q < NQ; ++q) {
    const int j = jj + 8 * q;
    m[q] = (i < n && j < n) ? S[(size_t)i * n + j] : 0.0;
  }
  if (i == 0) {
#pragma unroll
    for (int q = 0; q < NQ; ++q)
      if (jj + 8 * q < n) rowbuf[0][jj + 8 * q] = m[q];
  }
  __syncthreads();
  int bad = 0;
#pragma unroll
  for (int kq = 0; kq < NQ; ++kq) {
    for (int kr = 0; kr < 8; ++kr) {
      const int k = 8 * kq + kr;
      if (k >= n || bad) break;
      const double* row = rowbuf[k & 1];
      const double d = row[k];
      if (!(d > 0.0)) {      // the same value in every thread: uniform exit
        bad = k + 1;
        break;
      }
      const double pinv = 1.0 / d;
      const double ci = __shfl_sync(0xffffffffu, m[kq], (lane & ~7) | kr);   // M[i][k]
      const bool piv = (i == k);
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const int j = jj + 8 * q;
        if (j < n) {
          const double rj = row[j] * pinv;
          double v;
          if (j == k) v = piv ? pinv : -ci * pinv;
          else v = piv ? rj : fma(-ci, rj, m[q]);
          m[q] = v;
        }
      }
      if (i == k + 1) {      // the next pivot row, already updated
#pragma unroll
        for (int q = 0; q < NQ; ++q)
          if (jj + 8 * q < n) rowbuf[(k + 1) & 1][jj + 8 * q] = m[q];
      }
      __syncthreads();
    }
  }
  if (!bad && i < n) {
#pragma unroll
    for (int q = 0; q < NQ; ++q)
      if (jj + 8 * q < n) S[(size_t)i * n + jj + 8 * q] = m[q];
  }
  if (tid == 0) *info = bad;
}

// ---- SPD inverse on many CTAs: blocked Gauss-Jordan sweeps (n > kSpdBlockedMin) ------------------------
// (profiles/r02_spd_inverse_blocked.log)
// A one-CTA inverse is bound by one SM (its registers up to n = 128, its shared memory up to 234, global
// memory beyond: 5.5 ms at n = 264, ~20 ms at n = 404 = the LRVB covariance of K = 200).  Here the
// matrix is cut into 32 x 32 tiles and pivot block kb is swept by ONE launch of T x T CTAs, out of place
// (X -> Y, two buffers in turn; the matrix is at most 2 MB, so it lives in the L2):
//     Y_kk = P^-1        Y_kj = P^-1 X_kj        Y_ik = -X_ik P^-1        Y_ij = X_ij - X_ik P^-1 X_kj
// with P = X_kk inverted by one warp of every CTA (lane = row, the block in registers: redundant, but a
// launch round trip cheaper than publishing it).  After the T sweeps the buffer holds X^-1 (the sweep
// operator); a last launch symmetrises it into the caller's matrix.  The scalar pivots are those of the
// unblocked elimination, so "info = k: leading minor k not positive" keeps its meaning.  Indices >= n are
// padded with the identity.
constexpr int kSpdBlockedMin = 104;     // measured: equal at n = 104 (158 us), 1.5x at 128, 3.6x at 204, 44x at 404
__device__ __forceinline__ int gj_invert_block(double (&r)[32], int lane) {
  int bad = 0;
#pragma unroll
  for (int p = 0; p < 32; ++p) {
    const double d = __shfl_sync(0xffffffffu, r[p], p);
    if (!(d > 0.0) && !bad) bad = p + 1;      // the same value in every lane
    const double ip = 1.0 / d;
    const double f = r[p];                    // a_ip of this lane's row
    const bool me = (lane == p);
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (j == p) continue;
      const double rj = __shfl_sync(0xffffffffu, r[j], p) * ip;     // scaled pivot row
      r[j] = me ? rj : fma(-f, rj, r[j]);
    }
    r[p] = me ? ip : -f * ip;
  }
  return bad;
}

__global__ void __launch_bounds__(256)
k_spd_gj_step(const double* __restrict__ X, double* __restrict__ Y, int n, int kb, int* __restrict__ info) {
  pdl_sync();
  __shared__ double sP[32][33], sA[32][33], sR[32][33], sM[32][33];
  const int bi = blockIdx.y, bj = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int k0 = kb * 32, i0 = bi * 32, j0 = bj * 32;
  auto ldx = [&](int i, int j) { return (i < n && j < n) ? X[(size_t)i * n + j] : (i == j ? 1.0 : 0.0); };
  double c[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int r = warp * 4 + q;
    sP[r][lane] = ldx(k0 + r, k0 + lane);
    sA[r][lane] = ldx(i0 + r, k0 + lane);     // X_ik
    sR[r][lane] = ldx(k0 + r, j0 + lane);     // X_kj
    c[q] = ldx(i0 + r, j0 + lane);            // X_ij
  }
  __syncthreads();
  if (warp == 0) {
    double r[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) r[j] = sP[lane][j];
    const int bad = gj_invert_block(r, lane);
#pragma unroll
    for (int j = 0; j < 32; ++j) sP[lane][j] = r[j];
    if (bad && bi == 0 && bj == 0 && lane == 0 && k0 + bad <= n) atomicCAS(info, 0, k0 + bad);
  }
  __syncthreads();
  double o[4];
  if (bi == kb && bj == kb) {
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q] = sP[warp * 4 + q][lane];
  } else if (bi == kb) {            // P^-1 X_kj
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q] = 0.0;
#pragma unroll 8
    for (int t = 0; t < 32; ++t) {
      const double b = sR[t][lane];
#pragma unroll
      for (int q = 0; q < 4; ++q) o[q] = fma(sP[warp * 4 + q][t], b, o[q]);
    }
  } else {
    double m[4] = {0.0, 0.0, 0.0, 0.0};       // M = X_ik P^-1
#pragma unroll 8
    for (int t = 0; t < 32; ++t) {
      const double b = sP[t][lane];
#pragma unroll
      for (int q = 0; q < 4; ++q) m[q] = fma(sA[warp * 4 + q][t], b, m[q]);
    }
    if (bj == kb) {
#pragma unroll
      for (int q = 0; q < 4; ++q) o[q] = -m[q];
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) sM[warp * 4 + q][lane] = m[q];
      __syncthreads();
#pragma unroll
      for (int q = 0; q < 4; ++q) o[q] = c[q];
#pragma unroll 8
      for (int t = 0; t < 32; ++t) {
        const double b = sR[t][lane];
#pragma unroll
        for (int q = 0; q < 4; ++q) o[q] = fma(-sM[warp * 4 + q][t], b, o[q]);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int i = i0 + warp * 4 + q, j = j0 + lane;
    if (i < n && j < n) Y[(size_t)i * n + j] = o[q];
  }
}

// S = (Z + Z^T) / 2, one thread per pair i <= j (works in place: a pair is read and written by one thread)
__global__ void __launch_bounds__(256)
k_spd_gj_finish(const double* Z, double* S, int n) {
  pdl_sync();
  const int i = blockIdx.y * 16 + (threadIdx.x >> 4), j = blockIdx.x * 16 + (threadIdx.x & 15);
  if (i >= n || j >= n || i > j) return;
  const double v = 0.5 * (Z[(size_t)i * n + j] + Z[(size_t)j * n + i]);
  S[(size_t)i * n + j] = v;
  S[(size_t)j * n + i] = v;
}

// ---- direct solve by block elimination -----------------------------------------------------------
// rhs_g = [b_g] - sum_g B_g^T L_g^-1 b_l,g     (per right-hand side; per-CTA partials)
__global__ void __launch_bounds__(256)
k_solve_reduce(const double* __restrict__ B, const double* __restrict__ Linv,
               const double* __restrict__ b, double* __restrict__ part, int Dg, int G) {
  pdl_sync();
  extern __shared__ double acc[];  // 8 * Dg
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = threadIdx.x; c < 8 * Dg; c += blockDim.x) acc[c] = 0.0;
  __syncthreads();
  double* my = acc + (size_t)warp * Dg;
  for (int gi = blockIdx.x * 8 + warp; gi < G; gi += gridDim.x * 8) {
    const double bm = b[Dg + gi], bi = b[Dg + G + gi];
    const double* li = Linv + (size_t)gi * 3;
    const double t0 = li[0] * bm + li[1] * bi, t1 = li[1] * bm + li[2] * bi;
    const double* b0 = B + (size_t)gi * 2 * Dg;
    const double* b1 = b0 + Dg;
    for (int c = lane; c < Dg; c += 32) my[c] += b0[c] * t0 + b1[c] * t1;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < Dg; c += blockDim.x) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += acc[(size_t)w * Dg + c];
    part[(size_t)blockIdx.x * Dg + c] = s;
  }
}

__global__ void __launch_bounds__(256)
k_solve_reduce_finish(const double* __restrict__ part, int npart, const double* __restrict__ b,
                      double* __restrict__ rhs, int Dg, int include_bg) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= Dg) return;
  double t = 0.0;
  for (int p = lane; p < npart; p += 32) t += part[(size_t)p * Dg + r];
  t = warp_sum(t);
  if (lane == 0) rhs[r] = (include_bg ? b[r] : 0.0) - t;
}

// x_g = Sinv rhs_g  (one warp per row)
__global__ void __launch_bounds__(256)
k_solve_global(const double* __restrict__ Sinv, const double* __restrict__ rhs,
               double* __restrict__ x, int Dg) {
  pdl_sync();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= Dg) return;
  const double* a = Sinv + (size_t)r * Dg;
  double s = 0.0;
  for (int c = lane; c < Dg; c += 32) s = fma(a[c], rhs[c], s);
  s = warp_sum(s);
  if (lane == 0) x[r] = s;
}

// x_l,g = L_g^-1 (b_l,g - B_g x_g)   (one warp per group)
__global__ void __launch_bounds__(256)
k_solve_local(const double* __restrict__ B, const double* __restrict__ Linv,
              const double* __restrict__ b, double* __restrict__ x, int Dg, int G) {
  pdl_sync();
  extern __shared__ double xg[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c = threadIdx.x; c < Dg; c += blockDim.x) xg[c] = x[c];
  __syncthreads();
  for (int gi = blockIdx.x * 8 + warp; gi < G; gi += gridDim.x * 8) {
    const double* b0 = B + (size_t)gi * 2 * Dg;
    const double* b1 = b0 + Dg;
    double d0 = 0.0, d1 = 0.0;
    for (int c = lane; c < Dg; c += 32) {
      d0 = fma(b0[c], xg[c], d0);
      d1 = fma(b1[c], xg[c], d1);
    }
    d0 = warp_sum(d0);
    d1 = warp_sum(d1);
    if (lane == 0) {
      const double r0 = b[Dg + gi] - d0, r1 = b[Dg + G + gi] - d1;
      const double* li = Linv + (size_t)gi * 3;
      x[Dg + gi] = li[0] * r0 + li[1] * r1;
      x[Dg + G + gi] = li[1] * r0 + li[2] * r1;
    }
  }
}

// cov_g = L_g^-1 + T_g Sinv T_g^T with T_g = L_g^-1 B_g (2 x Dg): one warp per group,
// Sinv staged in shared memory when it fits, else read through L2.
__global__ void __launch_bounds__(256)
k_local_cov(const double* __restrict__ B, const double* __restrict__ Linv,
            const double* __restrict__ Sinv, double* __restrict__ cov, int Dg, int G) {
  pdl_sync();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int gi = blockIdx.x * 8 + warp; gi < G; gi += gridDim.x * 8) {
    const double* b0 = B + (size_t)gi * 2 * Dg;
    const double* b1 = b0 + Dg;
    // q00 = b0 Sinv b0^T, q01 = b0 Sinv b1^T, q11 = b1 Sinv b1^T
    double q00 = 0.0, q01 = 0.0, q11 = 0.0;
    for (int r = 0; r < Dg; ++r) {
      const double* s = Sinv + (size_t)r * Dg;
      double u0 = 0.0, u1 = 0.0;
      for (int c = lane; c < Dg; c += 32) {
        u0 = fma(s[c], b0[c], u0);
        u1 = fma(s[c], b1[c], u1);
      }
      u0 = warp_sum(u0);
      u1 = warp_sum(u1);
      const double x0 = b0[r], x1 = b1[r];
      q00 = fma(x0, u0, q00);
      q01 = fma(x0, u1, q01);
      q11 = fma(x1, u1, q11);
    }
    if (lane == 0) {
      const double* li = Linv + (size_t)gi * 3;
      const double i0 = li[0], i1 = li[1], i2 = li[2];
      // Linv * Q * Linv
      const double m00 = i0 * q00 + i1 * q01, m01 = i0 * q01 + i1 * q11;
      const double m10 = i1 * q00 + i2 * q01, m11 = i1 * q01 + i2 * q11;
      cov[(size_t)gi * 3] = i0 + m00 * i0 + m01 * i1;
      cov[(size_t)gi * 3 + 1] = i1 + m00 * i1 + m01 * i2;
      cov[(size_t)gi * 3 + 2] = i2 + m10 * i1 + m11 * i2;
    }
  }
}

static int require_hess(lrvb_glmm* h, const char* who) {
  LRVB_REQUIRE(h != nullptr, "%s: NULL handle", who);
  if (!h->hess_valid) {
    set_error("%s: no Hessian cached (call lrvb_glmm_eval with order 2 first)", who);
    return LRVB_ESTATE;
  }
  return ensure_solver_scratch(h);
}

static int prepare_linv(lrvb_glmm* h, cudaStream_t st) {
  if (h->G > 0) {
    LRVB_CUDA(launch_pdl(k_linv, dim3(cdiv(h->G, 256)), dim3(256), 0, st, h->L, h->Linv, h->G));
    LRVB_CHECK_LAUNCH();
  }
  return LRVB_OK;
}

}  // namespace lrvb

using namespace lrvb;

extern "C" {

int lrvb_glmm_hvp(lrvb_glmm* h, const double* v_dev, double* out_dev, int32_t include_A,
                  void* stream) {
  LRVB_TRY(require_hess(h, "lrvb_glmm_hvp"));
  LRVB_REQUIRE(v_dev && out_dev, "lrvb_glmm_hvp: NULL vector");
  LRVB_REQUIRE(v_dev != out_dev, "lrvb_glmm_hvp: in-place product not supported");
  return launch_hvp(h, v_dev, out_dev, include_A, nullptr, (cudaStream_t)stream);
}

static int cg_run(lrvb_glmm* h, const double* b_dev, const double* x0_dev, const lrvb_cg_precond* M,
                  double rtol, int32_t maxiter, double* x_dev, int32_t* info, int32_t* iters, void* stream) {
  LRVB_TRY(require_hess(h, "lrvb_glmm_cg"));
  LRVB_REQUIRE(b_dev && x_dev && info, "lrvb_glmm_cg: NULL argument");
  const int kind = M ? M->kind : 0;
  LRVB_REQUIRE(kind >= 0 && kind <= 4, "lrvb_glmm_cg: preconditioner kind = %d not in 0..4", kind);
  LRVB_REQUIRE(kind != LRVB_PRECOND_SCHUR || M->Sinv_dev, "lrvb_glmm_cg: Schur preconditioner needs Sinv_dev");
  LRVB_REQUIRE(kind != LRVB_PRECOND_CSR || (M->indptr_dev && M->indices_dev && M->data_dev),
               "lrvb_glmm_cg: CSR preconditioner needs indptr / indices / data");
  LRVB_REQUIRE(kind != LRVB_PRECOND_DENSE || M->dense_dev, "lrvb_glmm_cg: dense preconditioner needs dense_dev");
  const int precond = kind >= 2 ? 2 : kind;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t D = h->D;
  const int Dg = h->Dg, G = h->G;
  if (maxiter <= 0) maxiter = (int)(D * 10 < 2000000000 ? D * 10 : 2000000000);  // scipy: n * 10
  double* r = h->cgbuf;
  double* z = r + D;
  double* p = z + D;
  double* q = p + D;
  double* x = x_dev;
  double* rrpart = h->dotpart;
  double* rzpart = rrpart + 2 * (size_t)h->dot_grid;
  double* pqpart = rzpart + 2 * (size_t)h->dot_grid;
  int* flags = h->flags;
  const int vgrid = h->dot_grid;
  LRVB_CUDA(cudaMemsetAsync(flags, 0, sizeof(int) * 8, st));
  if (kind == LRVB_PRECOND_BLOCK_JACOBI || kind == LRVB_PRECOND_SCHUR) LRVB_TRY(prepare_linv(h, st));
  double* rhs_g = h->cgbuf + 4 * D;        // Dg doubles of scratch (Schur preconditioner)
  // ||b||, x, r
  LRVB_CUDA(launch_pdl(k_dot, dim3(vgrid), dim3(256), 0, st, b_dev, b_dev, nullptr, nullptr, D, pqpart, nullptr));
  LRVB_CHECK_LAUNCH();
  LRVB_CUDA(launch_pdl(k_cg_init, dim3(1), dim3(256), 0, st, pqpart, vgrid, rtol, h->scal, flags));
  LRVB_CHECK_LAUNCH();
  if (x0_dev) {
    if (x0_dev != x) LRVB_CUDA(cudaMemcpyAsync(x, x0_dev, sizeof(double) * D, cudaMemcpyDeviceToDevice, st));
    LRVB_TRY(launch_hvp(h, x, q, 1, nullptr, st));
    LRVB_CUDA(launch_pdl(k_axpby, dim3(vgrid), dim3(256), 0, st, r, b_dev, 1.0, q, -1.0, D));
  } else {
    LRVB_CUDA(cudaMemsetAsync(x, 0, sizeof(double) * D, st));
    LRVB_CUDA(launch_pdl(k_axpby, dim3(vgrid), dim3(256), 0, st, r, b_dev, 1.0, nullptr, 0.0, D));
  }
  LRVB_CHECK_LAUNCH();
  LRVB_CUDA(launch_pdl(k_dot, dim3(vgrid), dim3(256), 0, st, r, r, nullptr, nullptr, D, rrpart, nullptr));
  LRVB_CHECK_LAUNCH();

  int hflags[4] = {0, 0, 0, 0};
  int it = 0;
  const int batch = 8;
  while (it < maxiter) {
    const int end = (it + batch < maxiter) ? it + batch : maxiter;
    for (; it < end; ++it) {
      if (kind == LRVB_PRECOND_SCHUR) {
        // z = H^-1 r by block elimination with the caller's S^-1: M is the exact inverse
        LRVB_CUDA(launch_pdl(k_solve_reduce, dim3(h->hvp_grid), dim3(256), sizeof(double) * 8 * (size_t)Dg, st, h->B,
                             h->Linv, (const double*)r, h->hvppart, Dg, G));
        LRVB_CUDA(launch_pdl(k_solve_reduce_finish, dim3(cdiv(Dg, 8)), dim3(256), 0, st, h->hvppart, h->hvp_grid,
                             (const double*)r, rhs_g, Dg, 1));
        LRVB_CUDA(launch_pdl(k_solve_global, dim3(cdiv(Dg, 8)), dim3(256), 0, st, M->Sinv_dev, (const double*)rhs_g, z, Dg));
        g_launches += 3;
        if (G > 0) {
          LRVB_CUDA(launch_pdl(k_solve_local, dim3(h->hvp_grid), dim3(256), sizeof(double) * (size_t)Dg, st, h->B, h->Linv,
                               (const double*)r, z, Dg, G));
          ++g_launches;
        }
      } else if (kind == LRVB_PRECOND_CSR) {
        LRVB_CUDA(launch_pdl(k_cg_m_csr, dim3(vgrid), dim3(256), 0, st, M->indptr_dev, M->indices_dev, M->data_dev,
                             (const double*)r, z, D, (const int*)flags));
        ++g_launches;
      } else if (kind == LRVB_PRECOND_DENSE) {
        LRVB_CUDA(launch_pdl(k_cg_m_dense, dim3(vgrid), dim3(256), 0, st, M->dense_dev, (const double*)r, z, D,
                             (const int*)flags));
        ++g_launches;
      }
      LRVB_CUDA(launch_pdl(k_cg_precond, dim3(vgrid), dim3(256), 0, st, r, z, h->A, h->Linv, rrpart, vgrid, rzpart, h->scal, flags,
                                          Dg, G, precond));
      LRVB_CUDA(launch_pdl(k_cg_latch, dim3(1), dim3(1), 0, st, flags));
      LRVB_CUDA(launch_pdl(k_cg_dir, dim3(vgrid), dim3(256), 0, st, z, p, rzpart, vgrid, h->scal, flags, D, it));
      LRVB_TRY(launch_hvp(h, p, q, 1, flags, st));
      LRVB_CUDA(launch_pdl(k_dot, dim3(vgrid), dim3(256), 0, st, p, q, nullptr, nullptr, D, pqpart, flags));
      LRVB_CUDA(launch_pdl(k_cg_update, dim3(vgrid), dim3(256), 0, st, x, r, p, q, pqpart, vgrid, rrpart, h->scal, flags, D, it));
      g_launches += 4;  // precond, latch, dir, dot share the check below
      LRVB_CHECK_LAUNCH();
    }
    LRVB_CUDA(cudaMemcpyAsync(hflags, flags, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
    LRVB_CUDA(cudaStreamSynchronize(st));
    if (hflags[0]) break;
  }
  if (!hflags[0]) {
    // scipy tests convergence at the top of the next iteration only inside the loop: after
    // maxiter updates it reports maxiter without another test.
    *info = maxiter;
  } else {
    *info = 0;
  }
  if (iters) *iters = hflags[1];
  return LRVB_OK;
}

int lrvb_glmm_cg(lrvb_glmm* h, const double* b_dev, const double* x0_dev, int32_t precond,
                 double rtol, int32_t maxiter, double* x_dev, int32_t* info, int32_t* iters,
                 void* stream) {
  LRVB_REQUIRE(precond == 0 || precond == 1, "lrvb_glmm_cg: precond = %d not in {0,1}", precond);
  lrvb_cg_precond M = {};
  M.kind = precond;
  return cg_run(h, b_dev, x0_dev, &M, rtol, maxiter, x_dev, info, iters, stream);
}

int lrvb_glmm_cg_m(lrvb_glmm* h, const double* b_dev, const double* x0_dev, const lrvb_cg_precond* M,
                   double rtol, int32_t maxiter, double* x_dev, int32_t* info, int32_t* iters,
                   void* stream) {
  return cg_run(h, b_dev, x0_dev, M, rtol, maxiter, x_dev, info, iters, stream);
}

// ---- conjugate gradient over the shards of one job ------------------------------------------------
// Same iteration as lrvb_glmm_cg on vectors in the shard's local layout [globals | u.mean | u.info of
// the shard's groups]: the global entries are replicated on every rank (bitwise: they evolve from
// all-reduced quantities only), the local ones are private.  Per iteration TWO collectives over the
// NVLink peer windows (csrc/p2p.cu), both folded messages:
//   [r.r, r.z]                          after the preconditioner (2 doubles)
//   [(H p)_g (Dg doubles), p_l.q_l]     after the Hessian-vector product (Dg + 1 doubles)
// Dot products count the global entries once (`root` = the rank that owns them).  As in the single-GPU
// solver no scalar visits the host; the converged flag is read back every 8 iterations.
int lrvb_glmm_cg_sharded(lrvb_glmm* h, lrvb_p2p* comm_h, const double* b_dev, const double* x0_dev,
                         int32_t precond, double rtol, int32_t maxiter, int32_t root, double* x_dev,
                         int32_t* info, int32_t* iters, void* stream) {
  LRVB_TRY(require_hess(h, "lrvb_glmm_cg_sharded"));
  LRVB_REQUIRE(comm_h != nullptr, "lrvb_glmm_cg_sharded: the peer all-reduce handle is NULL");
  LRVB_REQUIRE(b_dev && x_dev && info, "lrvb_glmm_cg_sharded: NULL argument");
  LRVB_REQUIRE(precond == 0 || precond == 1, "lrvb_glmm_cg_sharded: precond = %d not in {0,1}", precond);
  LRVB_REQUIRE(maxiter > 0, "lrvb_glmm_cg_sharded: maxiter must be positive (10 x the JOB's dimension in scipy)");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t D = h->D;
  const int Dg = h->Dg, G = h->G;
  double* r = h->cgbuf;
  double* z = r + D;
  double* p = z + D;
  double* q = p + D;
  double* msg = q + D;            // Dg + 1
  double* sc = msg + D;           // 2 scalars
  double* x = x_dev;
  double* part = h->dotpart;      // (dot_grid, 2)
  int* flags = h->flags;
  const int vgrid = h->dot_grid;
  const int64_t lo = root ? 0 : Dg;      // first entry this rank counts in dot products
  LRVB_CUDA(cudaMemsetAsync(flags, 0, sizeof(int) * 8, st));
  if (precond) LRVB_TRY(prepare_linv(h, st));
#define LRVB_AR(buf, n) LRVB_TRY(lrvb_p2p_allreduce_sum(comm_h, (buf), (n), stream))
  // atol = rtol ||b||
  LRVB_CUDA(launch_pdl(k_dot, dim3(vgrid), dim3(256), 0, st, b_dev + lo, b_dev + lo, nullptr, nullptr, D - lo, part, nullptr));
  LRVB_CHECK_LAUNCH();
  LRVB_CUDA(launch_pdl(k_cg_fold, dim3(1), dim3(256), 0, st, part, vgrid, sc, nullptr));
  LRVB_CHECK_LAUNCH();
  LRVB_AR(sc, 2);
  LRVB_CUDA(launch_pdl(k_cg_init, dim3(1), dim3(256), 0, st, sc, 1, rtol, h->scal, flags));
  LRVB_CHECK_LAUNCH();
  if (x0_dev) {
    if (x0_dev != x) LRVB_CUDA(cudaMemcpyAsync(x, x0_dev, sizeof(double) * D, cudaMemcpyDeviceToDevice, st));
    LRVB_TRY(launch_hvp(h, x, q, root ? 1 : 0, nullptr, st));
    LRVB_AR(q, Dg);
    LRVB_CUDA(launch_pdl(k_axpby, dim3(vgrid), dim3(256), 0, st, r, b_dev, 1.0, q, -1.0, D));
  } else {
    LRVB_CUDA(cudaMemsetAsync(x, 0, sizeof(double) * D, st));
    LRVB_CUDA(launch_pdl(k_axpby, dim3(vgrid), dim3(256), 0, st, r, b_dev, 1.0, nullptr, 0.0, D));
  }
  LRVB_CHECK_LAUNCH();

  int hflags[4] = {0, 0, 0, 0};
  int it = 0;
  const int batch = 8;
  while (it < maxiter) {
    const int end = (it + batch < maxiter) ? it + batch : maxiter;
    for (; it < end; ++it) {
      LRVB_CUDA(launch_pdl(k_cg_precond2, dim3(vgrid), dim3(256), 0, st, r, z, h->A, h->Linv, part, flags, Dg, G,
                           precond, lo));
      LRVB_CUDA(launch_pdl(k_cg_fold, dim3(1), dim3(256), 0, st, part, vgrid, sc, flags));
      g_launches += 2;
      LRVB_AR(sc, 2);
      LRVB_CUDA(launch_pdl(k_cg_dir2, dim3(vgrid), dim3(256), 0, st, z, p, sc, h->scal, flags, D, it));
      LRVB_TRY(launch_hvp(h, p, q, root ? 1 : 0, flags, st));
      LRVB_CUDA(launch_pdl(k_dot, dim3(vgrid), dim3(256), 0, st, p + Dg, q + Dg, nullptr, nullptr, D - Dg, part, flags));
      LRVB_CUDA(launch_pdl(k_cg_pack, dim3(1), dim3(256), 0, st, q, part, vgrid, msg, Dg, flags));
      g_launches += 3;
      LRVB_AR(msg, (int64_t)Dg + 1);
      LRVB_CUDA(launch_pdl(k_cg_update2, dim3(vgrid), dim3(256), 0, st, x, r, p, q, msg, h->scal, flags, D, Dg, it));
      LRVB_CHECK_LAUNCH();
    }
    LRVB_CUDA(cudaMemcpyAsync(hflags, flags, sizeof(int) * 4, cudaMemcpyDeviceToHost, st));
    LRVB_CUDA(cudaStreamSynchronize(st));
    if (hflags[0]) break;
  }
#undef LRVB_AR
  if (!hflags[0]) {
    // one more convergence test would need another collective: scipy reports maxiter here as well
    *info = maxiter;
  } else {
    *info = 0;
  }
  if (iters) *iters = hflags[1];
  return LRVB_OK;
}

int lrvb_glmm_schur(lrvb_glmm* h, double* S_dev, int32_t include_A, void* stream) {
  LRVB_TRY(require_hess(h, "lrvb_glmm_schur"));
  LRVB_REQUIRE(S_dev != nullptr, "lrvb_glmm_schur: S is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  const int Dg = h->Dg, G = h->G;
  LRVB_TRY(prepare_linv(h, st));
  const int DT = (Dg + 7) / 8, R = (DT + kRT - 1) / kRT;
  const int n_jobs = R * (R + 1) / 2;
  int n_chunk = (8 * 2 * kNumSMs) / n_jobs;
  if (n_chunk < 1) n_chunk = 1;
  const int ksteps = (G + 1) / 2;
  if (n_chunk > ksteps) n_chunk = ksteps > 0 ? ksteps : 1;
  if (n_chunk > 512) n_chunk = 512;
  const size_t need = (size_t)n_chunk * n_jobs * kRT * kRT * 64;
  if (!h->schurpart || h->schur_grid != n_chunk) {
    if (h->schurpart) cudaFree(h->schurpart);
    h->schurpart = nullptr;
    LRVB_CUDA(cudaMalloc((void**)&h->schurpart, sizeof(double) * need));
    h->schur_grid = n_chunk;
  }
  LRVB_CUDA(launch_pdl(k_schur, dim3(cdiv((int64_t)n_jobs * n_chunk, 8)), dim3(256), 0, st, h->B, h->Linv, h->schurpart, Dg, G, R,
                                                              n_jobs, n_chunk));
  LRVB_CHECK_LAUNCH();
  LRVB_CUDA(launch_pdl(k_schur_finish, dim3(n_jobs * kRT * kRT), dim3(256), 0, st, h->schurpart, h->A, S_dev, Dg, R, n_jobs,
                                                     n_chunk, include_A));
  LRVB_CHECK_LAUNCH();
  return LRVB_OK;
}

int lrvb_spd_inverse(double* S_dev, int32_t n, int32_t* info_host, void* stream) {
  LRVB_REQUIRE(S_dev && info_host, "lrvb_spd_inverse: NULL argument");
  LRVB_REQUIRE(n >= 1 && n <= 4 + 2 * kMaxK, "lrvb_spd_inverse: n = %d out of range", n);
  cudaStream_t st = (cudaStream_t)stream;
  // the status word: one of 64 words of the CURRENT device, handed out round-robin (thread-safe), so that
  // calls on different devices, streams or threads never share a word -- and no allocation per call
  // (a stream-ordered cudaMallocAsync / cudaFreeAsync pair costs ~0.4 ms here: the default pool returns its
  // memory at every synchronisation)
  int* dinfo = nullptr;
  double* scratch = nullptr;        // second matrix buffer of the blocked sweeps: 8 per device, round-robin
  const bool blocked = n > kSpdBlockedMin;
  {
    static std::mutex mu;
    static int* words[64] = {nullptr};          // per device: 64 ints
    static unsigned next[64] = {0};
    static double* bufs[64] = {nullptr};        // per device: 8 matrices of the largest n
    int dev = 0;
    LRVB_CUDA(cudaGetDevice(&dev));
    LRVB_REQUIRE(dev >= 0 && dev < 64, "lrvb_spd_inverse: device ordinal %d not supported", dev);
    std::lock_guard<std::mutex> lock(mu);
    if (!words[dev]) LRVB_CUDA(cudaMalloc((void**)&words[dev], sizeof(int) * 64));
    const unsigned slot = next[dev]++;
    dinfo = words[dev] + (slot & 63u);
    if (blocked) {
      const size_t nmax = 4 + 2 * (size_t)kMaxK;
      if (!bufs[dev]) LRVB_CUDA(cudaMalloc((void**)&bufs[dev], sizeof(double) * 8 * nmax * nmax));
      scratch = bufs[dev] + (size_t)(slot & 7u) * nmax * nmax;
    }
  }
  if (blocked) {
    const int T = (n + 31) / 32;
    LRVB_CUDA(cudaMemsetAsync(dinfo, 0, sizeof(int), st));
    double* cur = S_dev;
    double* oth = scratch;
    for (int kb = 0; kb < T; ++kb) {
      LRVB_CUDA(launch_pdl(k_spd_gj_step, dim3(T, T), dim3(256), 0, st, (const double*)cur, oth, (int)n, kb, dinfo));
      double* t = cur; cur = oth; oth = t;
    }
    LRVB_CUDA(launch_pdl(k_spd_gj_finish, dim3((n + 15) / 16, (n + 15) / 16), dim3(256), 0, st, (const double*)cur,
                         S_dev, (int)n));
  } else {
    const int threads = 8 * ((n + 3) / 4 * 4);     // whole warps: 4 rows of 8 lanes each
    const int nq = (n + 7) / 8;
    cudaError_t le;
#define LRVB_SPD(Q) le = launch_pdl(k_spd_inverse_reg<Q>, dim3(1), dim3(threads), 0, st, S_dev, (int)n, dinfo)
    if (nq <= 2) LRVB_SPD(2);
    else if (nq <= 4) LRVB_SPD(4);
    else if (nq <= 6) LRVB_SPD(6);
    else if (nq <= 8) LRVB_SPD(8);
    else LRVB_SPD(16);
#undef LRVB_SPD
    LRVB_CUDA(le);
  }
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(info_host, dinfo, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    set_error("lrvb_spd_inverse failed: %s", cudaGetErrorString(e));
    return LRVB_ECUDA;
  }
  return LRVB_OK;
}

int lrvb_glmm_solve_reduce_rhs(lrvb_glmm* h, const double* b_dev, int32_t nrhs,
                               double* rhs_g_dev, int32_t include_bg, void* stream) {
  LRVB_TRY(require_hess(h, "lrvb_glmm_solve_reduce_rhs"));
  LRVB_REQUIRE(b_dev && rhs_g_dev && nrhs >= 1, "lrvb_glmm_solve_reduce_rhs: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int Dg = h->Dg, G = h->G;
  LRVB_TRY(prepare_linv(h, st));
  for (int j = 0; j < nrhs; ++j) {
    const double* b = b_dev + (size_t)j * h->D;
    LRVB_CUDA(launch_pdl(k_solve_reduce, dim3(h->hvp_grid), dim3(256), sizeof(double) * 8 * (size_t)Dg, st, h->B, h->Linv, b,
                                                                              h->hvppart, Dg, G));
    LRVB_CUDA(launch_pdl(k_solve_reduce_finish, dim3(cdiv(Dg, 8)), dim3(256), 0, st, h->hvppart, h->hvp_grid, b,
                                                       rhs_g_dev + (size_t)j * Dg, Dg, include_bg));
    LRVB_CHECK_LAUNCH();
  }
  return LRVB_OK;
}

int lrvb_glmm_solve_finish(lrvb_glmm* h, const double* Sinv_dev, const double* rhs_g_dev,
                           const double* b_dev, int32_t nrhs, double* x_dev, void* stream) {
  LRVB_TRY(require_hess(h, "lrvb_glmm_solve_finish"));
  LRVB_REQUIRE(Sinv_dev && rhs_g_dev && b_dev && x_dev && nrhs >= 1,
               "lrvb_glmm_solve_finish: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int Dg = h->Dg, G = h->G;
  for (int j = 0; j < nrhs; ++j) {
    double* x = x_dev + (size_t)j * h->D;
    LRVB_CUDA(launch_pdl(k_solve_global, dim3(cdiv(Dg, 8)), dim3(256), 0, st, Sinv_dev, rhs_g_dev + (size_t)j * Dg, x, Dg));
    if (G > 0)
      LRVB_CUDA(launch_pdl(k_solve_local, dim3(h->hvp_grid), dim3(256), sizeof(double) * (size_t)Dg, st, 
          h->B, h->Linv, b_dev + (size_t)j * h->D, x, Dg, G));
    LRVB_CHECK_LAUNCH();
  }
  return LRVB_OK;
}

int lrvb_glmm_local_cov(lrvb_glmm* h, const double* Sinv_dev, double* cov_dev, void* stream) {
  LRVB_TRY(require_hess(h, "lrvb_glmm_local_cov"));
  LRVB_REQUIRE(Sinv_dev && cov_dev, "lrvb_glmm_local_cov: NULL argument");
  cudaStream_t st = (cudaStream_t)stream;
  LRVB_TRY(prepare_linv(h, st));
  if (h->G > 0) {
    int grid = cdiv(h->G, 8);
    if (grid > 8 * kNumSMs) grid = 8 * kNumSMs;
    LRVB_CUDA(launch_pdl(k_local_cov, dim3(grid), dim3(256), 0, st, h->B, h->Linv, Sinv_dev, cov_dev, h->Dg, h->G));
    LRVB_CHECK_LAUNCH();
  }
  return LRVB_OK;
}

}  // extern "C"
