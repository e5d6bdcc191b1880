// Shared declarations of the lrvb_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/lrvb_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "lrvb_b200 is written for sm_100a (B200) only"
#endif

namespace lrvb {

void set_error(const char* fmt, ...);

#define LRVB_CUDA(call)                                                              \
  do {                                                                               \
    cudaError_t e__ = (call);                                                        \
    if (e__ != cudaSuccess) {                                                        \
      lrvb::set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,           \
                      cudaGetErrorString(e__));                                      \
      return LRVB_ECUDA;                                                             \
    }                                                                                \
  } while (0)

// every kernel launch of the library is followed by exactly one LRVB_CHECK_LAUNCH (or adds the
// extra launches to g_launches by hand), so lrvb_launch_count() is the number of OUR kernels
extern long long g_launches;
#define LRVB_CHECK_LAUNCH()          \
  do {                               \
    ++lrvb::g_launches;              \
    LRVB_CUDA(cudaGetLastError());   \
  } while (0)

#define LRVB_REQUIRE(cond, ...)                                                      \
  do {                                                                               \
    if (!(cond)) {                                                                   \
      lrvb::set_error(__VA_ARGS__);                                                  \
      return LRVB_EINVAL;                                                            \
    }                                                                                \
  } while (0)

#define LRVB_TRY(expr)                                                               \
  do {                                                                               \
    int rc__ = (expr);                                                               \
    if (rc__ != LRVB_OK) return rc__;                                                \
  } while (0)

constexpr int kMaxQ = 64;
constexpr int kMaxK = 256;
constexpr int kNumSMs = 148;  // B200
constexpr int kRT = 4;        // Schur warp job = kRT x kRT output tiles of 8x8 (solve.cu)

static inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

template <typename T>
static int dev_alloc(T** p, size_t n) {
  *p = nullptr;
  if (n == 0) n = 1;
  LRVB_CUDA(cudaMalloc((void**)p, n * sizeof(T)));
  return LRVB_OK;
}

// Let `kernel` use `bytes` of dynamic shared memory on the current device.  The limit is an attribute of the
// kernel on a device, shared by every handle there, so it is only ever raised: lowering it to one handle's
// need would make another handle's launches fail.
template <typename... KArgs>
static int raise_smem_limit(void (*kernel)(KArgs...), size_t bytes) {
  cudaFuncAttributes fa;
  LRVB_CUDA(cudaFuncGetAttributes(&fa, kernel));
  if (bytes > (size_t)fa.maxDynamicSharedSizeBytes)
    LRVB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return LRVB_OK;
}

// ---- fp64 special functions the CUDA math library lacks -------------------------------
// digamma / trigamma / tetragamma for x > 0: upward recurrence to x >= 16, then the
// asymptotic (Bernoulli) series; truncation < 1e-17 relative there.
__host__ __device__ inline double digamma_pos(double x) {
  double acc = 0.0;
  while (x < 16.0) { acc -= 1.0 / x; x += 1.0; }
  const double r = 1.0 / x, r2 = r * r;
  double s = r2 * (1.0 / 12.0 - r2 * (1.0 / 120.0 - r2 * (1.0 / 252.0 - r2 * (1.0 / 240.0 -
             r2 * (1.0 / 132.0 - r2 * (691.0 / 32760.0 - r2 * (1.0 / 12.0)))))));
  return acc + log(x) - 0.5 * r - s;
}
__host__ __device__ inline double trigamma_pos(double x) {
  double acc = 0.0;
  while (x < 16.0) { acc += 1.0 / (x * x); x += 1.0; }
  const double r = 1.0 / x, r2 = r * r;
  double s = r * r2 * (1.0 / 6.0 - r2 * (1.0 / 30.0 - r2 * (1.0 / 42.0 - r2 * (1.0 / 30.0 -
             r2 * (5.0 / 66.0 - r2 * (691.0 / 2730.0 - r2 * (7.0 / 6.0)))))));
  return acc + r + 0.5 * r2 + s;
}
__host__ __device__ inline double tetragamma_pos(double x) {
  double acc = 0.0;
  while (x < 16.0) { acc -= 2.0 / (x * x * x); x += 1.0; }
  const double r = 1.0 / x, r2 = r * r;
  double s = r2 * r2 * (0.5 - r2 * (1.0 / 6.0 - r2 * (1.0 / 6.0 - r2 * (3.0 / 10.0 -
             r2 * (5.0 / 6.0 - r2 * (691.0 / 210.0 - r2 * (35.0 / 2.0)))))));
  return acc - r2 - r * r2 - s;
}

// Branch-free digamma and log-gamma for the batched exponential-family kernels (x > 0): shift by EIGHT with
// the product P(x) = x (x+1) ... (x+7) and its derivative (psi(x) = psi(x+8) - P'(x)/P(x): one division
// instead of up to sixteen dependent ones; lgamma(x) = lgamma(x+8) - log P(x)), then the asymptotic series
// at y = x + 8 >= 8 through y^-16 (psi) / y^-15 (lgamma): truncation < 2e-16 / 1e-16.  Both share y, 1/y,
// log y and P.  Huge arguments (P would overflow) take the series directly.
struct PsiLg {
  double psi, lg;
};
__host__ __device__ inline PsiLg digamma_lgamma_pos(double x, bool want_lg) {
  PsiLg o;
  double p = x, dp = 1.0;
#pragma unroll
  for (int k = 1; k < 8; ++k) {
    const double t = x + (double)k;
    dp = fma(dp, t, p);
    p *= t;
  }
  const bool huge = x > 1e15;
  const double y = huge ? x : x + 8.0;
  const double ly = log(y);
  const double r = 1.0 / y, r2 = r * r;
  const double sp = r2 * (1.0 / 12.0 - r2 * (1.0 / 120.0 - r2 * (1.0 / 252.0 - r2 * (1.0 / 240.0 -
                    r2 * (1.0 / 132.0 - r2 * (691.0 / 32760.0 - r2 * (1.0 / 12.0 - r2 * (3617.0 / 8160.0))))))));
  o.psi = ly - 0.5 * r - sp - (huge ? 0.0 : dp / p);
  o.lg = 0.0;
  if (want_lg) {
    const double sl = r * (1.0 / 12.0 - r2 * (1.0 / 360.0 - r2 * (1.0 / 1260.0 - r2 * (1.0 / 1680.0 -
                      r2 * (1.0 / 1188.0 - r2 * (691.0 / 360360.0 - r2 * (1.0 / 156.0 - r2 * (3617.0 / 122400.0))))))));
    o.lg = (y - 0.5) * ly - y + 0.91893853320467274178 + sl - (huge ? 0.0 : log(p));
  }
  return o;
}

// psi', psi'' and psi''' for x > 0, branch-free like digamma_lgamma_pos (the third derivative of the gamma entropy
// and of E log tau, amip.cu): shift by eight (psi^(n)(x) = psi^(n)(x+8) + (-1)^(n+1) n! sum_{k<8} (x+k)^-(n+1)),
// then the asymptotic series at y = x + 8 >= 8 through the Bernoulli number B_20: the first omitted term is
// below 1e-16 (psi'), 3e-15 (psi''), 3e-14 (psi''') relative.
struct Psi123 {
  double p1, p2, p3;
};
__host__ __device__ inline Psi123 polygamma123_pos(double x) {
  double s2 = 0.0, s3 = 0.0, s4 = 0.0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const double r = 1.0 / (x + (double)k), rr = r * r;
    s2 += rr;
    s3 = fma(rr, r, s3);
    s4 = fma(rr, rr, s4);
  }
  const double y = x + 8.0, r = 1.0 / y, r2 = r * r;
  const double b1 = 1.0 / 6.0 + r2 * (-1.0 / 30.0 + r2 * (1.0 / 42.0 + r2 * (-1.0 / 30.0 + r2 * (5.0 / 66.0 +
                    r2 * (-691.0 / 2730.0 + r2 * (7.0 / 6.0 + r2 * (-3617.0 / 510.0 + r2 * (43867.0 / 798.0 +
                    r2 * (-174611.0 / 330.0)))))))));
  const double b2 = 0.5 + r2 * (-1.0 / 6.0 + r2 * (1.0 / 6.0 + r2 * (-3.0 / 10.0 + r2 * (5.0 / 6.0 +
                    r2 * (-691.0 / 210.0 + r2 * (35.0 / 2.0 + r2 * (-3617.0 / 30.0 + r2 * (43867.0 / 42.0 +
                    r2 * (-1222277.0 / 110.0)))))))));
  const double b3 = 2.0 + r2 * (-1.0 + r2 * (4.0 / 3.0 + r2 * (-3.0 + r2 * (10.0 +
                    r2 * (-691.0 / 15.0 + r2 * (280.0 + r2 * (-10851.0 / 5.0 + r2 * (438670.0 / 21.0 +
                    r2 * (-1222277.0 / 5.0)))))))));
  Psi123 o;
  o.p1 = r + 0.5 * r2 + r * r2 * b1 + s2;
  o.p2 = -r2 - r * r2 - r2 * r2 * b2 - 2.0 * s3;
  o.p3 = 2.0 * r * r2 + 3.0 * r2 * r2 + r * r2 * r2 * b3 + 6.0 * s4;
  return o;
}

#ifdef __CUDACC__
// ---- programmatic dependent launch (PDL) ------------------------------------------------------
// Every kernel of the evaluation / CSR chain starts with pdl_sync(): it lets the NEXT kernel of the
// stream be scheduled right away (its CTAs start as soon as SM resources free up instead of after
// a full launch round trip) and then waits until the PREVIOUS kernel has completed and flushed its
// memory.  Launched without the attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_sync() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
// The two halves separately.  A kernel that calls pdl_wait() BEFORE pdl_launch_dependents() lets its
// dependent start only once this kernel's own prerequisite has completed: the dependent may then read,
// ahead of its own wait, everything written by kernels EARLIER than this one (k_finish -> k_global).
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- warp / block helpers ----------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum with a fixed (deterministic) tree; result valid in thread 0.
// `red` is shared scratch of >= 32 doubles.  All threads must call.
__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  double r = 0.0;
  if (wid == 0) {
    r = (lane < nw) ? red[lane] : 0.0;
    r = warp_sum(r);
  }
  return r;
}

// FP64 tensor-core MMA, D(8x8) += A(8x4, row) * B(4x8, col).  SASS: DMMA.8x8x4.
//   a : A[lane>>2][lane&3]      b : B[lane&3][lane>>2]      c0,c1 : C[lane>>2][2*(lane&3)+{0,1}]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// Copy `n` contiguous doubles global -> shared with cp.async (16 B chunks when both sides are
// 16-B aligned, 8 B otherwise).  All threads of the CTA call; caller commits / waits / syncs.
__device__ __forceinline__ void tile_load_async(double* dst, const double* src, int64_t n) {
  const bool al16 = ((((uintptr_t)src) | ((uintptr_t)dst)) & 15) == 0;
  if (al16) {
    const int64_t n2 = n >> 1;
    for (int64_t i = threadIdx.x; i < n2; i += blockDim.x) cp_async16(dst + 2 * i, src + 2 * i);
    if ((n & 1) && threadIdx.x == 0) cp_async8(dst + n - 1, src + n - 1);
  } else {
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) cp_async8(dst + i, src + i);
  }
}
#endif  // __CUDACC__

struct FusedArgs;   // fused.cuh

}  // namespace lrvb

// ---- the model handle --------------------------------------------------------------------
struct lrvb_glmm {
  int64_t N = 0, D = 0;
  int64_t ldw = 0;            // row stride of W (N rounded up to 8: 16-B aligned rows for TMA)
  int K = 0, G = 0, Q = 0, Dg = 0, KT = 0;  // KT = ceil(K/8) feature tiles
  int include_global = 1;
  int vecmode = 0;            // 1: evaluate in the constrained ("vector") parameterisation
  int64_t shard_g0 = 0, shard_G = 0;   // shard_G > 0: eval reads the FULL layout of a job with shard_G groups
  const double *X = nullptr, *y = nullptr, *w = nullptr;
  const int32_t* g = nullptr;
  lrvb_glmm_prior prior;
  lrvb_glmm_bounds bounds;
  // ---- device-owned ----
  double* gh = nullptr;       // [2][Q]: c_q = sqrt(2) x_q ; what_q = w_q / sqrt(pi)
  int32_t* gptr = nullptr;    // (G+1) first observation of each group
  double* vec = nullptr;      // (D) constrained values
  double* W = nullptr;        // (5, ldw) per-observation derivative weights
  // observation pass
  int obs_nbuf = 0, obs_grid = 0;   // k_obs (K > 62): number of tile buffers, CTAs
  size_t obs_smem = 0;
  double* klpart = nullptr;   // (obs_grid) per-CTA partials of sum w*l
  double* gradpart = nullptr; // (obs_grid, 2, K) per-CTA partials of X^T l_m , S^T l_v
  // fused observation + group pass (K <= 62, obs_fused.cuh)
  int gram_mid = 0;           // 24 < K <= 104: a warp or team of warps owns the packed triangle (gram_mid.cuh)
  int obs_fused = 0, of_grid = 0, of_warps = 0;
  size_t of_smem = 0;
  int64_t of_rows_per_warp = 0;
  double* bval = nullptr;     // (of_grid * of_warps, 2, 5 + 4K) head / tail pieces of straddling groups
  double* wc_scratch = nullptr;   // (2, ldw) l_m, l_v of a weight-cross-Hessian pass for K > 62 (allocated on first use)
  // one-slot variant of the fused observation pass, which the evaluation runs (more warps per SM than two slots)
  int of1_grid = 0, of1_warps = 0;
  size_t of1_smem = 0;
  int64_t of1_rows_per_warp = 0;
  // order-2 evaluation in one pass (fused.cuh, K <= 24): teams of warps do quadrature, group sums and Gram per stage
  int fused2 = 0, fu_grid = 0, fu_teams = 0, fu_warps = 0;
  int64_t fu_rows_per_team = 0;
  size_t fu_smem = 0;
  void (*fu_kernel)(lrvb::FusedArgs) = nullptr;   // the instantiation for K
  int ev_gram = 0;            // the last timed evaluation ran a separate Gram kernel
  // group pass
  double* gsc = nullptr;      // (G, 5) per-group sums of l_m, l_v, a, b, c
  double* BR = nullptr;       // (G, 4, K) raw borders: sum a x, sum b x, sum b s, sum c s
  int loc_grid = 0;
  double* locpart = nullptr;  // (loc_grid, 4) partials of sum dm, sum Sg, sum log u_info, -
  double* fin_pre = nullptr;         // (8 + 2K) results of k_finish's block 0 for its last block
  unsigned int* fin_counter = nullptr;   // finished work blocks of the running k_finish (reset by its global block)
  // Gram
  int gram_tn = 0, gram_grid_x = 0, gram_grid_y = 0, gram_jobs = 0;   // grid_y = job groups
  size_t gram_smem = 0;
  // gram_mid: the instantiation for K and its CTA size
  void (*gm_kernel)(const double*, const double*, double*, int64_t, int64_t, int) = nullptr;
  int gm_warps = 0;
  int group_overlap = 1;      // k_group on the side stream behind k_gram_wide (LRVB_GROUP_OVERLAP=0: serial)
  int gram_wide = 0;          // K = 176 .. 240, K % 8 == 0: block jobs of 4-5 tiles, 8 warps x 255 registers (gram_wide.cuh);
                              // jobs = GwGroup[], gslots = GwCta[gram_grid_x]
  void* jobs = nullptr;            // device GbJob[gram_jobs]   (gram_big.cuh, K > 20)
  void* gslots = nullptr;          // device GbSlot[gram_grid_y * 16]
  double* grampart = nullptr;      // per-CTA partial tiles of the Gram kernel
  // results
  double *A = nullptr, *B = nullptr, *L = nullptr;  // cached Hessian blocks (free coords)
  double* gradl = nullptr;    // (2G) local gradient of the last eval
  double* outg = nullptr;     // (1 + Dg + Dg*Dg) packed [KL, grad_g, A] of the last eval
  int hess_valid = 0;
  int grad_valid = 0;
  int point_valid = 0;        // vec holds the constrained parameters of the last evaluation
  // optional per-kernel timing (bench): events around the whole eval, k_obs and k_gram
  // side stream: the HBM-bound per-group pass runs beside the FP64-bound Gram kernel
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int timing = 0;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int ev_order = -1;
  // CSR
  int32_t* rowcnt = nullptr;  // (D+1)
  int32_t* scanblk = nullptr; // scan scratch
  int32_t* csrwork = nullptr; // cntA | coltot | chunkcnt | chunkoff
  int csr_cg = 0, csr_nchunk = 0;
  uint32_t* csrmask = nullptr;   // zero mask of the last full export (refill compares against it)
  int csr_pattern_valid = 0;     // csrwork / csrmask describe the pattern of the last full export
  int64_t csr_nnz = -1;
  // solver scratch
  double* cgbuf = nullptr;    // 6*D
  int hvp_grid = 0;
  double* hvppart = nullptr;  // (hvp_grid, Dg)
  int dot_grid = 0;
  double* dotpart = nullptr;  // (dot_grid, 4)
  double* scal = nullptr;     // device scalars (32)
  int* flags = nullptr;       // device ints (8)
  double* Linv = nullptr;     // (G,3) inverse local blocks (Schur / precond)
  double* T = nullptr;        // (G,2,Dg) L^-1 B for the Schur path
  int schur_grid = 0;
  double* schurpart = nullptr;
  double* pred_B = nullptr;   // (3 Kp8, Kp4) scaled beta block of S^-1 for lrvb_glmm_predict_lr (predict.cu)
  double* logo_V = nullptr;   // (G, Dg) per-group gradients of lrvb_glmm_logo, then its (G, K) Cook's products (logo.cu)
  double* amip_work = nullptr;   // row coefficients, per-CTA and per-group partials of lrvb_glmm_third_contract (amip.cu)
};

namespace lrvb {
// glmm_eval.cu entry points used by api.cu (all enqueue on `st`)
// Plan the evaluation of a new handle: kernels, launch geometries, their scratch buffers and shared-memory limits.
int plan_eval(lrvb_glmm* h, cudaStream_t st);
int launch_eval(lrvb_glmm* h, const double* free_dev, int order, double* out_global,
                double* grad_local, cudaStream_t st);
}  // namespace lrvb
