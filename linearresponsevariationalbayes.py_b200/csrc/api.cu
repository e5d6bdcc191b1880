// C-ABI entry points: handle life-cycle and evaluation (see include/lrvb_b200.h).
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <new>
#include <vector>
#include "common.cuh"
#include "gram_small.cuh"
#include "obs_fused.cuh"
#include "gram_mid.cuh"
#include "gram_big.cuh"
#include "gram_wide.cuh"
#include "fused.cuh"

namespace lrvb {

static thread_local char g_err[1024] = "";
long long g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Validate group ids (range, sortedness) and build gptr (G+1): first observation of each group.
__global__ void k_gptr(const int32_t* __restrict__ g, int32_t* __restrict__ gptr, int* flags,
                       int64_t N, int G) {
  const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n > N) return;
  int prev = (n == 0) ? -1 : g[n - 1];
  int cur = (n == N) ? G : g[n];
  if (n < N && (cur < 0 || cur >= G)) { atomicOr(flags, 1); return; }
  if (n > 0 && (prev < 0 || prev >= G)) { atomicOr(flags, 1); return; }
  if (n > 0 && n < N && cur < prev) { atomicOr(flags, 2); return; }
  for (int gg = prev + 1; gg <= cur; ++gg) gptr[gg] = (int32_t)n;
}

template <typename T>
static int dev_alloc(T** p, size_t n) {
  *p = nullptr;
  if (n == 0) n = 1;
  LRVB_CUDA(cudaMalloc((void**)p, n * sizeof(T)));
  return LRVB_OK;
}

// kernels defined in glmm_eval.cu whose attributes must be raised for > 48 KB dynamic smem
void configure_kernels(size_t obs_smem, size_t gram_smem);
void configure_obs_fused(size_t smem);

}  // namespace lrvb

using namespace lrvb;

extern "C" {

const char* lrvb_last_error(void) { return g_err; }
int lrvb_version(void) { return 100; }

int lrvb_glmm_destroy(lrvb_glmm* h) {
  if (!h) return LRVB_OK;
  void* ptrs[] = {h->gh, h->gptr, h->vec, h->W, h->klpart, h->gradpart, h->gsc, h->BR, h->locpart, h->fin_counter, h->fin_pre,
                  h->jobs, h->gslots, h->grampart, h->bval, h->wc_scratch, h->B, h->L, h->gradl, h->outg, h->rowcnt, h->scanblk, h->csrwork, h->csrmask,
                  h->cgbuf, h->hvppart, h->dotpart, h->scal, h->flags, h->Linv, h->T,
                  h->schurpart, h->pred_B, h->logo_V};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  for (cudaEvent_t e : h->ev)
    if (e) cudaEventDestroy(e);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->side) cudaStreamDestroy(h->side);
  delete h;
  return LRVB_OK;
}

int lrvb_glmm_create(lrvb_glmm** out, int64_t N, int32_t K, int32_t G, int32_t Q,
                     const double* X_dev, const double* y_dev, const int32_t* g_dev,
                     const double* w_dev, const double* gh_x_host, const double* gh_w_host,
                     const lrvb_glmm_prior* prior, const lrvb_glmm_bounds* bounds,
                     int32_t include_global_terms, void* stream) {
  LRVB_REQUIRE(out != nullptr, "lrvb_glmm_create: out is NULL");
  *out = nullptr;
  LRVB_REQUIRE(N >= 0 && N < (int64_t)2147483000, "lrvb_glmm_create: N = %lld out of range",
               (long long)N);
  LRVB_REQUIRE(K >= 1 && K <= kMaxK, "lrvb_glmm_create: K = %d not in [1, %d]", K, kMaxK);
  LRVB_REQUIRE(G >= 0, "lrvb_glmm_create: G = %d negative", G);
  LRVB_REQUIRE(Q >= 1 && Q <= kMaxQ, "lrvb_glmm_create: Q = %d not in [1, %d]", Q, kMaxQ);
  LRVB_REQUIRE(N == 0 || (X_dev && y_dev && g_dev), "lrvb_glmm_create: X, y, g must be non-NULL");
  LRVB_REQUIRE(N == 0 || G >= 1, "lrvb_glmm_create: observations but no groups");
  LRVB_REQUIRE(gh_x_host && gh_w_host && prior && bounds, "lrvb_glmm_create: NULL argument");
  LRVB_REQUIRE((((uintptr_t)X_dev) & 15) == 0, "lrvb_glmm_create: X not 16-byte aligned");
  LRVB_REQUIRE(N == 0 || (((((uintptr_t)y_dev) | ((uintptr_t)g_dev) | ((uintptr_t)w_dev)) & 15) == 0),
               "lrvb_glmm_create: y, g, w must be 16-byte aligned (bulk async copies)");
  cudaStream_t st = (cudaStream_t)stream;

  lrvb_glmm* h = new (std::nothrow) lrvb_glmm();
  LRVB_REQUIRE(h != nullptr, "out of host memory");
  h->N = N; h->K = K; h->G = G; h->Q = Q;
  h->Dg = 4 + 2 * K;
  h->D = h->Dg + 2 * (int64_t)G;
  h->KT = (K + 7) / 8;
  h->include_global = include_global_terms ? 1 : 0;
  h->X = X_dev; h->y = y_dev; h->g = g_dev; h->w = w_dev;
  h->prior = *prior;
  h->bounds = *bounds;
  const int Dg = h->Dg;

#define CREATE_TRY(expr)                         \
  do {                                           \
    int rc__ = (expr);                           \
    if (rc__ != LRVB_OK) { lrvb_glmm_destroy(h); return rc__; } \
  } while (0)
#define CREATE_CUDA(call)                                                      \
  do {                                                                         \
    cudaError_t e__ = (call);                                                  \
    if (e__ != cudaSuccess) {                                                  \
      set_error("%s failed: %s", #call, cudaGetErrorString(e__));              \
      lrvb_glmm_destroy(h);                                                    \
      return LRVB_ECUDA;                                                       \
    }                                                                          \
  } while (0)

  // quadrature constants: c_q = sqrt(2) x_q, what_q = w_q / sqrt(pi)   (Modeling.py:41-48)
  std::vector<double> ghh(2 * Q);
  for (int q = 0; q < Q; ++q) {
    ghh[q] = sqrt(2.0) * gh_x_host[q];
    ghh[Q + q] = gh_w_host[q] / sqrt(M_PI);
  }
  CREATE_TRY(dev_alloc(&h->gh, 2 * Q));
  CREATE_CUDA(cudaMemcpyAsync(h->gh, ghh.data(), sizeof(double) * 2 * Q, cudaMemcpyHostToDevice, st));
  CREATE_CUDA(cudaStreamSynchronize(st));  // ghh goes out of scope

  CREATE_TRY(dev_alloc(&h->flags, 8));
  CREATE_CUDA(cudaMemsetAsync(h->flags, 0, sizeof(int) * 8, st));
  CREATE_TRY(dev_alloc(&h->gptr, (size_t)G + 1));
  k_gptr<<<cdiv(N + 1, 256), 256, 0, st>>>(g_dev, h->gptr, h->flags, N, G);
  CREATE_CUDA(cudaGetLastError());
  int hflag = 0;
  CREATE_CUDA(cudaMemcpyAsync(&hflag, h->flags, sizeof(int), cudaMemcpyDeviceToHost, st));
  CREATE_CUDA(cudaStreamSynchronize(st));
  if (hflag) {
    set_error(hflag & 1 ? "lrvb_glmm_create: group id outside [0, G)"
                        : "lrvb_glmm_create: group ids must be non-decreasing (group-sorted)");
    lrvb_glmm_destroy(h);
    return LRVB_EINVAL;
  }

  CREATE_TRY(dev_alloc(&h->vec, (size_t)h->D + 8 + (size_t)K + (size_t)G));   // + k_prep's derived factors (prep_aux)
  h->ldw = (N + 7) / 8 * 8;
  CREATE_TRY(dev_alloc(&h->W, 5 * (size_t)h->ldw));

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
    // fused observation + group pass: every warp owns a contiguous multiple-of-32 range of rows
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
      // one-slot rings when they buy at least three more warps per SM (K >= ~36)
      const int w1 = obs_fused_warps(K, 1);
      if (w1 >= h->of_warps + 3) {
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
      if (tt > nrec) nrec = tt;
    }
    CREATE_TRY(dev_alloc(&h->bval, (size_t)nrec * 2 * (5 + 4 * (size_t)K)));
    configure_obs_fused(h->of_smem > h->of1_smem ? h->of_smem : h->of1_smem);
    if (h->obs_grid < h->of_grid) h->obs_grid = h->of_grid;
    if (h->obs_grid < h->fu_grid) h->obs_grid = h->fu_grid;     // klpart / gradpart are sized by obs_grid
  }
  CREATE_TRY(dev_alloc(&h->klpart, (size_t)h->obs_grid));
  CREATE_TRY(dev_alloc(&h->gradpart, (size_t)h->obs_grid * 2 * K));

  CREATE_TRY(dev_alloc(&h->gsc, (size_t)G * 5));
  CREATE_TRY(dev_alloc(&h->BR, (size_t)G * 4 * K));
  h->loc_grid = cdiv(G, 256);
  if (h->loc_grid > 2 * kNumSMs) h->loc_grid = 2 * kNumSMs;
  if (h->loc_grid < 1) h->loc_grid = 1;
  CREATE_TRY(dev_alloc(&h->locpart, (size_t)h->loc_grid * 4));
  CREATE_TRY(dev_alloc(&h->fin_counter, 1));
  CREATE_TRY(dev_alloc(&h->fin_pre, 8 + 2 * (size_t)K));
  CREATE_CUDA(cudaMemsetAsync(h->fin_counter, 0, sizeof(unsigned int), st));

  // Gram geometry
  {
    size_t npart;
    if (h->fused2) {
      // no Gram kernel: the one-pass kernel (fused.cuh) writes the packed partials, one slab per CTA
      npart = (size_t)h->fu_grid * gram_small_shape(K).NT * 64;
    } else if (K <= kGmMaxK) {
      // 24 < K <= 104: one warp or a team of warps = the whole packed triangle (gram_mid.cuh)
      h->gram_mid = 1;
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
      CREATE_TRY(dev_alloc((char**)&h->jobs, sizeof(GwGroup) * pl.groups.size()));
      CREATE_TRY(dev_alloc((char**)&h->gslots, sizeof(GwCta) * pl.ctas.size()));
      CREATE_CUDA(cudaMemcpyAsync(h->jobs, pl.groups.data(), sizeof(GwGroup) * pl.groups.size(),
                                  cudaMemcpyHostToDevice, st));
      CREATE_CUDA(cudaMemcpyAsync(h->gslots, pl.ctas.data(), sizeof(GwCta) * pl.ctas.size(),
                                  cudaMemcpyHostToDevice, st));
      CREATE_CUDA(cudaStreamSynchronize(st));   // pl goes out of scope
      npart = (size_t)h->gram_grid_x * gram_small_shape(K).NT * 64;
    } else {
      // rectangles of the packed triangle dealt to 16-warp CTAs (gram_big.cuh)
      const GbPlan pl = gram_big_plan(K);
      h->gram_jobs = (int)pl.jobs.size();
      h->gram_grid_y = pl.n_groups;
      h->gram_tn = pl.TN;
      h->gram_smem = pl.smem;
      int64_t nst = (N + pl.TN - 1) / pl.TN;
      int64_t nchunk = (kNumSMs * kGbCtasPerSM) / pl.n_groups;
      if (nchunk > nst) nchunk = nst;
      if (nchunk < 1) nchunk = 1;
      h->gram_grid_x = (int)nchunk * pl.n_groups;
      CREATE_TRY(dev_alloc((char**)&h->jobs, sizeof(GbJob) * pl.jobs.size()));
      CREATE_TRY(dev_alloc((char**)&h->gslots, sizeof(GbSlot) * pl.slots.size()));
      CREATE_CUDA(cudaMemcpyAsync(h->jobs, pl.jobs.data(), sizeof(GbJob) * pl.jobs.size(),
                                  cudaMemcpyHostToDevice, st));
      CREATE_CUDA(cudaMemcpyAsync(h->gslots, pl.slots.data(), sizeof(GbSlot) * pl.slots.size(),
                                  cudaMemcpyHostToDevice, st));
      CREATE_CUDA(cudaStreamSynchronize(st));   // pl goes out of scope
      npart = (size_t)nchunk * pl.n_groups * kGbWarps * 16 * 64;
    }
    CREATE_TRY(dev_alloc(&h->grampart, npart));
    CREATE_CUDA(cudaMemsetAsync(h->grampart, 0, sizeof(double) * npart, st));
  }
  configure_kernels(h->obs_smem, h->gram_smem);

  CREATE_TRY(dev_alloc(&h->B, (size_t)G * 2 * Dg));
  CREATE_TRY(dev_alloc(&h->L, (size_t)G * 3));
  CREATE_TRY(dev_alloc(&h->gradl, 2 * (size_t)G));
  CREATE_TRY(dev_alloc(&h->outg, 1 + (size_t)Dg + (size_t)Dg * Dg));
  h->A = h->outg + 1 + Dg;
  CREATE_TRY(dev_alloc(&h->scal, 32));
  CREATE_CUDA(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
  CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
  CREATE_CUDA(cudaStreamSynchronize(st));
#undef CREATE_TRY
#undef CREATE_CUDA
  *out = h;
  return LRVB_OK;
}

long long lrvb_launch_count(void) { return g_launches; }

int lrvb_glmm_set_timing(lrvb_glmm* h, int32_t enable) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_set_timing: NULL handle");
  if (enable && !h->ev[0])
    for (int i = 0; i < 6; ++i) LRVB_CUDA(cudaEventCreate(&h->ev[i]));
  h->timing = enable ? 1 : 0;
  h->ev_order = -1;
  return LRVB_OK;
}

int lrvb_glmm_last_timing(lrvb_glmm* h, float* ms3) {
  LRVB_REQUIRE(h != nullptr && ms3 != nullptr, "lrvb_glmm_last_timing: NULL argument");
  if (!h->timing || h->ev_order < 0) {
    set_error("lrvb_glmm_last_timing: timing not enabled or no evaluation since it was enabled");
    return LRVB_ESTATE;
  }
  LRVB_CUDA(cudaEventSynchronize(h->ev[5]));
  ms3[0] = ms3[1] = ms3[2] = 0.f;
  LRVB_CUDA(cudaEventElapsedTime(&ms3[0], h->ev[4], h->ev[5]));
  if (h->N > 0) {
    LRVB_CUDA(cudaEventElapsedTime(&ms3[1], h->ev[0], h->ev[1]));
    // with the one-pass kernel (fused.cuh) there is no separate Gram launch: ms3[2] stays 0
    if (h->ev_order >= 2 && h->ev_gram) LRVB_CUDA(cudaEventElapsedTime(&ms3[2], h->ev[2], h->ev[3]));
  }
  return LRVB_OK;
}

int lrvb_glmm_set_coords(lrvb_glmm* h, int32_t vector_coords) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_set_coords: NULL handle");
  if (h->vecmode != (vector_coords ? 1 : 0)) {
    h->vecmode = vector_coords ? 1 : 0;
    h->hess_valid = 0;
    h->grad_valid = 0;
    h->point_valid = 0;
  }
  return LRVB_OK;
}

int lrvb_glmm_set_shard(lrvb_glmm* h, int64_t g0, int64_t G_total) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_set_shard: NULL handle");
  LRVB_REQUIRE(G_total == 0 || (g0 >= 0 && g0 + h->G <= G_total),
               "lrvb_glmm_set_shard: groups [%lld, %lld) are not inside [0, %lld)", (long long)g0,
               (long long)(g0 + h->G), (long long)G_total);
  h->shard_g0 = G_total > 0 ? g0 : 0;
  h->shard_G = G_total;
  h->point_valid = 0;
  return LRVB_OK;
}

int lrvb_glmm_dims(const lrvb_glmm* h, int64_t* D, int32_t* Dg) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_dims: NULL handle");
  if (D) *D = h->D;
  if (Dg) *Dg = h->Dg;
  return LRVB_OK;
}

int lrvb_glmm_eval(lrvb_glmm* h, const double* free_dev, int32_t order, double* out_global_dev,
                   double* grad_local_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_eval: NULL handle");
  LRVB_REQUIRE(free_dev != nullptr, "lrvb_glmm_eval: free is NULL");
  LRVB_REQUIRE(order >= 0 && order <= 2, "lrvb_glmm_eval: order = %d not in {0,1,2}", order);
  return launch_eval(h, free_dev, order, out_global_dev, grad_local_dev, (cudaStream_t)stream);
}

int lrvb_glmm_result_buffers(lrvb_glmm* h, double** out_global_dev, double** grad_local_dev) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_result_buffers: NULL handle");
  if (out_global_dev) *out_global_dev = h->outg;
  if (grad_local_dev) *grad_local_dev = h->gradl;
  return LRVB_OK;
}

int lrvb_glmm_blocks(lrvb_glmm* h, double** A_dev, double** B_dev, double** L_dev) {
  LRVB_REQUIRE(h != nullptr, "lrvb_glmm_blocks: NULL handle");
  if (!h->hess_valid) {
    set_error("lrvb_glmm_blocks: no Hessian cached (call lrvb_glmm_eval with order 2 first)");
    return LRVB_ESTATE;
  }
  if (A_dev) *A_dev = h->A;
  if (B_dev) *B_dev = h->B;
  if (L_dev) *L_dev = h->L;
  return LRVB_OK;
}

int lrvb_glmm_set_global_block(lrvb_glmm* h, const double* A_dev, void* stream) {
  LRVB_REQUIRE(h != nullptr && A_dev != nullptr, "lrvb_glmm_set_global_block: NULL argument");
  if (!h->hess_valid) {
    set_error("lrvb_glmm_set_global_block: no Hessian cached");
    return LRVB_ESTATE;
  }
  if (A_dev != h->A)
    LRVB_CUDA(cudaMemcpyAsync(h->A, A_dev, sizeof(double) * (size_t)h->Dg * h->Dg,
                              cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return LRVB_OK;
}

int lrvb_glmm_obs_weights(lrvb_glmm* h, double** W_dev, int64_t* ld) {
  LRVB_REQUIRE(h != nullptr && W_dev != nullptr, "lrvb_glmm_obs_weights: NULL argument");
  if (!h->grad_valid) {
    set_error("lrvb_glmm_obs_weights: no evaluation of order >= 1 cached");
    return LRVB_ESTATE;
  }
  *W_dev = h->W;
  if (ld) *ld = h->ldw;
  return LRVB_OK;
}

}  // extern "C"
