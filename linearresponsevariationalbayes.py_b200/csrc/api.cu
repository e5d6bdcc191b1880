// C-ABI entry points: handle life-cycle and evaluation (see include/lrvb_b200.h).
#include <stdarg.h>
#include <string.h>
#include <new>
#include <vector>
#include "common.cuh"

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

// Poisson data checks beside k_gptr's, on the same flags word: 4 = a y that is negative or not finite, 8 = an
// offset that is not finite.  Per-CTA partials of c = sum_n w_n lgamma(y_n + 1) (grid fixed by N: a fixed order).
constexpr int kPoisConstCtas = 1024;
__global__ void __launch_bounds__(256)
k_pois_check(const double* __restrict__ y, const double* __restrict__ w, const double* __restrict__ off, int64_t N,
             int* flags, double* __restrict__ part) {
  __shared__ double red[32];
  int bad = 0;
  double c = 0.0;
  for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
    const double yn = y[n];
    if (!(yn >= 0.0) || !isfinite(yn)) bad |= 4;
    else c += (w ? w[n] : 1.0) * lgamma(yn + 1.0);
    if (off && !isfinite(off[n])) bad |= 8;
  }
  if (bad) atomicOr(flags, bad);
  c = block_sum(c, red);
  if (threadIdx.x == 0) part[blockIdx.x] = c;
}
__global__ void __launch_bounds__(256) k_pois_const(const double* __restrict__ part, int n, double* __restrict__ c) {
  __shared__ double red[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += part[i];
  s = block_sum(s, red);
  if (threadIdx.x == 0) *c = s;
}

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
                  h->schurpart, h->pred_B, h->logo_V, h->amip_work, h->ij_work, h->pois_work};
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

  CREATE_TRY(plan_eval(h, st));

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

int lrvb_glmm_create_poisson(lrvb_glmm** out, int64_t N, int32_t K, int32_t G, const double* X_dev,
                             const double* y_dev, const int32_t* g_dev, const double* w_dev, const double* offset_dev,
                             const lrvb_glmm_prior* prior, const lrvb_glmm_bounds* bounds,
                             int32_t include_global_terms, void* stream) {
  LRVB_REQUIRE(out != nullptr, "lrvb_glmm_create_poisson: out is NULL");
  *out = nullptr;
  LRVB_REQUIRE(N >= 0 && N < (int64_t)2147483000, "lrvb_glmm_create_poisson: N = %lld out of range", (long long)N);
  LRVB_REQUIRE(K >= 1 && K <= kMaxK, "lrvb_glmm_create_poisson: K = %d not in [1, %d]", K, kMaxK);
  LRVB_REQUIRE(G >= 0, "lrvb_glmm_create_poisson: G = %d negative", G);
  LRVB_REQUIRE(N == 0 || (X_dev && y_dev && g_dev), "lrvb_glmm_create_poisson: X, y, g must be non-NULL");
  LRVB_REQUIRE(N == 0 || G >= 1, "lrvb_glmm_create_poisson: observations but no groups");
  LRVB_REQUIRE(prior && bounds, "lrvb_glmm_create_poisson: NULL argument");
  LRVB_REQUIRE((((uintptr_t)X_dev) & 15) == 0, "lrvb_glmm_create_poisson: X not 16-byte aligned");
  LRVB_REQUIRE(N == 0 || ((((uintptr_t)y_dev) | ((uintptr_t)g_dev) | ((uintptr_t)w_dev) | ((uintptr_t)offset_dev)) &
                          15) == 0,
               "lrvb_glmm_create_poisson: y, g, w, offset must be 16-byte aligned (bulk async copies)");
  cudaStream_t st = (cudaStream_t)stream;

  lrvb_glmm* h = new (std::nothrow) lrvb_glmm();
  LRVB_REQUIRE(h != nullptr, "out of host memory");
  h->family = kFamilyPoisson;
  h->N = N; h->K = K; h->G = G; h->Q = 0;
  h->Dg = 4 + 2 * K;
  h->D = h->Dg + 2 * (int64_t)G;
  h->KT = (K + 7) / 8;
  h->include_global = include_global_terms ? 1 : 0;
  h->X = X_dev; h->y = y_dev; h->g = g_dev; h->w = w_dev; h->offset = N > 0 ? offset_dev : nullptr;
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

  CREATE_TRY(dev_alloc(&h->flags, 8));
  CREATE_CUDA(cudaMemsetAsync(h->flags, 0, sizeof(int) * 8, st));
  CREATE_TRY(dev_alloc(&h->gptr, (size_t)G + 1));
  k_gptr<<<cdiv(N + 1, 256), 256, 0, st>>>(g_dev, h->gptr, h->flags, N, G);
  CREATE_CUDA(cudaGetLastError());
  // c = sum_n w_n lgamma(y_n + 1), the part of the log-likelihood that does not depend on the parameters
  const int nc = N == 0 ? 1 : (cdiv(N, 256) < kPoisConstCtas ? cdiv(N, 256) : kPoisConstCtas);
  CREATE_TRY(dev_alloc(&h->pois_work, 1 + (size_t)nc));
  CREATE_CUDA(cudaMemsetAsync(h->pois_work, 0, sizeof(double) * (1 + (size_t)nc), st));
  if (N > 0) {
    k_pois_check<<<nc, 256, 0, st>>>(y_dev, w_dev, h->offset, N, h->flags, h->pois_work + 1);
    CREATE_CUDA(cudaGetLastError());
    k_pois_const<<<1, 256, 0, st>>>(h->pois_work + 1, nc, h->pois_work);
    CREATE_CUDA(cudaGetLastError());
  }
  int hflag = 0;
  CREATE_CUDA(cudaMemcpyAsync(&hflag, h->flags, sizeof(int), cudaMemcpyDeviceToHost, st));
  CREATE_CUDA(cudaStreamSynchronize(st));
  if (hflag) {
    set_error(hflag & 1 ? "lrvb_glmm_create_poisson: group id outside [0, G)"
              : hflag & 2 ? "lrvb_glmm_create_poisson: group ids must be non-decreasing (group-sorted)"
              : hflag & 4 ? "lrvb_glmm_create_poisson: y must be finite and >= 0 (counts)"
                          : "lrvb_glmm_create_poisson: the offset must be finite");
    lrvb_glmm_destroy(h);
    return LRVB_EINVAL;
  }

  CREATE_TRY(dev_alloc(&h->vec, (size_t)h->D + 8 + (size_t)K + (size_t)G));   // + k_prep's derived factors (prep_aux)
  h->ldw = (N + 7) / 8 * 8;
  CREATE_TRY(dev_alloc(&h->W, 5 * (size_t)h->ldw));

  CREATE_TRY(plan_eval(h, st));

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
