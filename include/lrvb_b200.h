/*
 * lrvb_b200.h -- C ABI of the B200-native logistic-GLMM LRVB hot path.
 *
 * Drop-in boundary for rgiordan/LinearResponseVariationalBayes.py (reference paths are
 * relative to /root/reference/LinearResponseVariationalBayes/).  The reference has no FFI:
 * its "operator interface" for this path is the Python class Objective
 * (SparseObjectives.py:95-240), the sparse-Hessian helpers (SparseObjectives.py:581-657),
 * ConjugateGradientSolver (ConjugateGradient.py:63-105) and the closed-form terms in
 * Modeling.py:35-52 / ExponentialFamilies.py:5-120.  Every entry point below names the
 * reference call it replaces.  INTEGRATION.md shows the ctypes stub a maintainer adds.
 *
 * Conventions
 *  - plain C types only; every `const double*` / `double*` / `int32_t*` named "dev" is a
 *    CUDA device pointer on the current device, borrowed for the duration of the call
 *    (X, y, g, w are borrowed for the lifetime of the handle);
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is
 *    enqueued on it, nothing synchronises unless the comment says "syncs";
 *  - every function returns 0 on success; otherwise a negative code and
 *    lrvb_last_error() holds a message (thread-local).
 *      LRVB_EINVAL (-1): bad size / shape / argument  -> ValueError in the reference
 *      LRVB_ECUDA  (-2): CUDA runtime failure         -> RuntimeError
 *      LRVB_ESTATE (-3): call order (e.g. HVP before a Hessian was evaluated)
 *  - all floating point is IEEE fp64.
 *
 * Flat parameter layout (ParameterDictionary.py:39-46, 64-65; SURVEY.md A.3), D = Dg + 2G,
 * Dg = 4 + 2K:   [mu.mean, mu.info, tau.shape, tau.rate, beta.mean[K], beta.info[K],
 *                 u.mean[G], u.info[G]]
 * "free" coordinates are the reference's unconstrained ones (Parameters.py:31-61):
 * identity for means, log(value - lb) for info / shape / rate.
 */
#ifndef LRVB_B200_H
#define LRVB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRVB_OK 0
#define LRVB_EINVAL (-1)
#define LRVB_ECUDA (-2)
#define LRVB_ESTATE (-3)

typedef struct lrvb_glmm lrvb_glmm;

/* Priors: mu ~ N(mu_mean, 1/mu_info), beta_k ~ N(beta_mean, 1/beta_info), tau ~ Gamma(shape, rate)
 * (ExponentialFamilies.py:191-195 uvn_prior / gamma_prior). */
typedef struct {
  double mu_mean, mu_info, beta_mean, beta_info, tau_shape, tau_rate;
} lrvb_glmm_prior;

/* Lower bounds of the constrained sub-parameters (NormalParams.py:29,56 min_info;
 * GammaParams.py:7-8 min_shape / min_rate). */
typedef struct {
  double mu_info, tau_shape, tau_rate, beta_info, u_info;
} lrvb_glmm_bounds;

const char* lrvb_last_error(void);
int lrvb_version(void);

/* ---- model handle ---------------------------------------------------------------------
 * Binds the data the reference's objective closure would capture (the zero-argument `fun`
 * handed to Objective(par, fun), SparseObjectives.py:95-100).
 *  X  dev (N,K) row-major fp64 (the reference's C-order ndarray), y dev (N,) fp64 in {0,1},
 *  g  dev (N,) int32 group id in [0,G), NON-DECREASING (group-sorted); w dev (N,) or NULL.
 *  gh_x, gh_w HOST (Q,) numpy.polynomial.hermite.hermgauss(Q) nodes / weights
 *  (Modeling.py:35-37 takes them from the caller), Q <= 64.
 *  include_global_terms: 1 = this handle also owns the terms that do not depend on any
 *  group (priors and entropies of mu, beta, tau); ranks > 0 of an observation-sharded job
 *  pass 0 so that the all-reduced sum counts them once.
 * Validates sizes and the sortedness / range of g (syncs). */
int lrvb_glmm_create(lrvb_glmm** out, int64_t N, int32_t K, int32_t G, int32_t Q,
                     const double* X_dev, const double* y_dev, const int32_t* g_dev,
                     const double* w_dev, const double* gh_x_host, const double* gh_w_host,
                     const lrvb_glmm_prior* prior, const lrvb_glmm_bounds* bounds,
                     int32_t include_global_terms, void* stream);
/* The Poisson log-link GLMM for counts (R's glmer(..., family = poisson) with offset(log(exposure))): the same
 * variational family, layout, priors and calls as above with the observation term
 *   E_q log p(y_n | eta_n) = w_n (y_n m_n - exp(m_n + v_n / 2) - lgamma(y_n + 1)),
 * m_n = x_n . E[beta] + E[u_g] + offset_n, v_n = x_n^2 . Var[beta] + Var[u_g], exact under q (no quadrature, no Q).
 *  y dev (N,) fp64 counts, finite and >= 0 (non-integer values are accepted); offset dev (N,) fp64 or NULL, finite,
 *  16-byte aligned like y.  Validates on the device (syncs) and computes sum_n w_n lgamma(y_n + 1) once.
 * lrvb_glmm_predict, _predict_lr, _loo, _logo and _third_contract evaluate the logistic likelihood and return
 * LRVB_EINVAL on a Poisson handle; every other call works unchanged. */
int lrvb_glmm_create_poisson(lrvb_glmm** out, int64_t N, int32_t K, int32_t G, const double* X_dev,
                             const double* y_dev, const int32_t* g_dev, const double* w_dev, const double* offset_dev,
                             const lrvb_glmm_prior* prior, const lrvb_glmm_bounds* bounds,
                             int32_t include_global_terms, void* stream);
int lrvb_glmm_destroy(lrvb_glmm* h);
/* Number of CUDA kernels this library has launched in this process (bench.py gpu_launches). */
long long lrvb_launch_count(void);
/* Optional instrumentation for bench.py's roofline: when enabled, lrvb_glmm_eval records CUDA
 * events on the launching stream around the whole evaluation, the per-observation kernel and the
 * DMMA Gram kernel; lrvb_glmm_last_timing syncs on the last one and returns
 * ms3 = {whole eval, k_obs, k_gram} (HOST floats). */
int lrvb_glmm_set_timing(lrvb_glmm* h, int32_t enable);
int lrvb_glmm_last_timing(lrvb_glmm* h, float* ms3_host);
/* Coordinates of the evaluation point and of every derivative returned afterwards:
 * 0 (default) = free / unconstrained (Objective.fun_free*, SparseObjectives.py:120-158),
 * 1 = constrained "vector" coordinates (Objective.fun_vector*, :127-181).  Invalidates the
 * cached Hessian. */
int lrvb_glmm_set_coords(lrvb_glmm* h, int32_t vector_coords);
/* Observation-sharded jobs (SURVEY.md 8e): this handle owns groups [g0, g0 + G) of a job with
 * G_total groups.  Afterwards lrvb_glmm_eval's free_dev is the job's FULL flat vector
 * (4 + 2K + 2 G_total entries, layout above) and the handle reads its own entries out of it;
 * every output stays in the handle's local layout.  G_total = 0 restores the default. */
int lrvb_glmm_set_shard(lrvb_glmm* h, int64_t g0, int64_t G_total);
/* D = 4 + 2K + 2G, Dg = 4 + 2K. */
int lrvb_glmm_dims(const lrvb_glmm* h, int64_t* D, int32_t* Dg);

/* ---- value / gradient / Hessian ---------------------------------------------------------
 * Replaces Objective.fun_free, fun_free_grad, fun_free_hessian (SparseObjectives.py:120-158)
 * for the composed GLMM KL (SURVEY.md A.1).  order 0: KL; 1: + gradient; 2: + Hessian blocks.
 *  free_dev      (D,)  evaluation point in free coordinates
 *  out_global    dev, 1 + Dg + Dg*Dg doubles: [KL, grad[0:Dg], A (Dg,Dg) row-major]; only the
 *                parts `order` asks for are written.  This packed buffer is exactly what an
 *                observation-sharded job all-reduces (sum) across ranks.
 *  grad_local    dev (2G,) = grad[Dg:D] (u.mean then u.info) or NULL; written when order >= 1.
 * With order 2 the Hessian is kept inside the handle as arrowhead blocks
 * (A (Dg,Dg); B (G,2,Dg): rows u.mean_g / u.info_g against the globals; L (G,3): the 2x2
 * local block as (mm, mi, ii)) for the calls below. */
int lrvb_glmm_eval(lrvb_glmm* h, const double* free_dev, int32_t order, double* out_global_dev,
                   double* grad_local_dev, void* stream);
/* The handle's own result buffers (borrowed, fixed for the handle's lifetime): out_global
 * [KL, grad_g (Dg), A (Dg*Dg)] and grad_local (2G).  lrvb_glmm_eval with NULL output pointers
 * writes there and nowhere else (no device-to-device copy at the end of an evaluation); a sharded
 * job all-reduces out_global in place, which also updates the cached global block A. */
int lrvb_glmm_result_buffers(lrvb_glmm* h, double** out_global_dev, double** grad_local_dev);
/* Device pointers of the cached blocks (borrowed; valid until the next eval / destroy). */
int lrvb_glmm_blocks(lrvb_glmm* h, double** A_dev, double** B_dev, double** L_dev);
/* Overwrite the cached global block (after the all-reduce of out_global in a sharded job). */
int lrvb_glmm_set_global_block(lrvb_glmm* h, const double* A_dev, void* stream);
/* Per-observation derivative weights of the last eval: dev (5, *ld) rows
 * [dl/dz_mean, dl/dz_var, d2l/dz_mean2, d2l/dz_mean dz_var, d2l/dz_var2] (SURVEY.md A.2), the
 * first N entries of each row are the observations (row stride *ld >= N keeps rows 16-byte
 * aligned); rows 2-4 only after order 2.  Borrowed pointer. */
int lrvb_glmm_obs_weights(lrvb_glmm* h, double** W_dev, int64_t* ld);

/* ---- cross-Hessian with the observation weights ------------------------------------------
 * Replaces TwoParameterObjective.fun_hessian_free1_vector2 (SparseObjectives.py:429-438) as used
 * by ParametricSensitivityLinearApproximation (ModelSensitivity.py:555-612) when the
 * hyperparameter is the vector of observation weights: C = d^2 KL / d free d w is (D x N) with
 * column n = -grad_free l_n; it is applied, never formed.  Both calls work at the point (and in the
 * coordinates) of the last lrvb_glmm_eval, for K <= 62.  dw: dev (N) 16-byte aligned, in the
 * handle's (group-sorted) observation order; v: dev (D). */
int lrvb_glmm_weight_cross_matvec(lrvb_glmm* h, const double* dw_dev, double* out_dev /* D */, void* stream);
int lrvb_glmm_weight_cross_rmatvec(lrvb_glmm* h, const double* v_dev, double* out_dev /* N */, void* stream);

/* ---- sparse Hessian export ------------------------------------------------------------
 * Replaces get_sparse_sub_hessian + csr_matrix summation (SparseObjectives.py:591-619):
 * exact zeros dropped, columns sorted, int32 indices, one entry per coordinate.
 * _capacity returns the structural upper bound Dg^2 + 4 Dg G + 4 G on nnz (no device work).
 * lrvb_glmm_hessian_csr writes indptr (D+1,), indices and data (first nnz of `capacity` entries)
 * and the actual nnz into the DEVICE scalar nnz_dev; it never synchronises, the caller reads
 * nnz_dev when it needs the size.  capacity must be >= the structural bound. */
int lrvb_glmm_hessian_csr_capacity(const lrvb_glmm* h, int64_t* capacity);
int lrvb_glmm_hessian_csr(lrvb_glmm* h, int32_t* indptr_dev, int32_t* indices_dev,
                          double* data_dev, int64_t capacity, int64_t* nnz_dev, void* stream);

/* The pattern of an arrowhead Hessian is static between evaluations unless an entry becomes (or stops
 * being) exactly zero.  After one full export on this handle, lrvb_glmm_hessian_csr_refill rewrites `data`
 * ALONE (one pass, offsets cached in the handle) for the pattern `indptr_dev` of that export and compares the
 * zero mask of the new values with the recorded one: *mismatch_dev (int32, caller zeroes it) becomes 1 when
 * the pattern changed, in which case `data` is unusable and a full export is needed.  mismatch_host_mapped
 * (nullable) is a device-accessible pointer to pinned HOST memory that receives the same flag, so the host
 * can read it once the kernel has completed without queueing a copy on the stream.
 * lrvb_glmm_hessian_csr_if is that full export made conditional ON THE DEVICE: every kernel is a no-op unless
 * *run_if_dev != 0, so "refill, then csr_if(mismatch)" never synchronises with the host and is always right. */
int lrvb_glmm_hessian_csr_refill(lrvb_glmm* h, const int32_t* indptr_dev, double* data_dev,
                                 int32_t* mismatch_dev, int32_t* mismatch_host_mapped, void* stream);
int lrvb_glmm_hessian_csr_if(lrvb_glmm* h, const int32_t* run_if_dev, int32_t* indptr_dev, int32_t* indices_dev,
                             double* data_dev, int64_t capacity, int64_t* nnz_dev, void* stream);

/* ---- Hessian-vector product -------------------------------------------------------------
 * Replaces Objective.fun_free_hvp (SparseObjectives.py:183-187) at the point of the last
 * order-2 eval.  v_dev, out_dev (D,).  include_A = 0 leaves the A v_g term out of out[0:Dg]
 * (ranks > 0 of a sharded job, whose A is a replica). */
int lrvb_glmm_hvp(lrvb_glmm* h, const double* v_dev, double* out_dev, int32_t include_A,
                  void* stream);

/* ---- conjugate gradient -----------------------------------------------------------------
 * Replaces ConjugateGradientSolver.get_hinv_vec (ConjugateGradient.py:81-85), i.e.
 * scipy.sparse.linalg.cg(A, b, x0, rtol, atol=0, M): stops when ||r|| <= rtol * ||b||.
 *  precond: 0 = none, 1 = M = inverse of the block-diagonal of H (diag of A, 2x2 local blocks).
 *  x0_dev NULL = zeros.  info: 0 converged, >0 = maxiter reached (scipy convention).
 * Single-GPU handle only.  Syncs. */
int lrvb_glmm_cg(lrvb_glmm* h, const double* b_dev, const double* x0_dev, int32_t precond,
                 double rtol, int32_t maxiter, double* x_dev, int32_t* info, int32_t* iters,
                 void* stream);

/* The same solve with any preconditioner M (the `M=` argument of scipy.sparse.linalg.cg that
 * ConjugateGradientSolver.preconditioner feeds, ConjugateGradient.py:84):
 *   LRVB_PRECOND_NONE / _BLOCK_JACOBI as above;
 *   LRVB_PRECOND_SCHUR: M = H^-1 applied exactly by block elimination with Sinv_dev = S^-1 (Dg,Dg) from
 *     lrvb_glmm_schur + lrvb_spd_inverse (SURVEY.md A.4: "use as preconditioner and as the cross-check");
 *   LRVB_PRECOND_CSR:   M a (D,D) device CSR matrix (int32 indptr / indices, fp64 data), z = M r by SpMV;
 *   LRVB_PRECOND_DENSE: M a dense row-major (D,D) device matrix.
 * M must be symmetric positive definite, as scipy requires. */
#define LRVB_PRECOND_NONE 0
#define LRVB_PRECOND_BLOCK_JACOBI 1
#define LRVB_PRECOND_SCHUR 2
#define LRVB_PRECOND_CSR 3
#define LRVB_PRECOND_DENSE 4
typedef struct {
  int32_t kind;
  const double* Sinv_dev;
  const int32_t* indptr_dev;
  const int32_t* indices_dev;
  const double* data_dev;
  const double* dense_dev;
} lrvb_cg_precond;
int lrvb_glmm_cg_m(lrvb_glmm* h, const double* b_dev, const double* x0_dev, const lrvb_cg_precond* M,
                   double rtol, int32_t maxiter, double* x_dev, int32_t* info, int32_t* iters,
                   void* stream);

/* ---- direct arrowhead solve / LRVB covariance -------------------------------------------
 * Schur complement of the local blocks (SURVEY.md A.4):
 *   S = [include_A ? A : 0] - sum_g B_g^T L_g^{-1} B_g     (Dg,Dg) row-major, dev.
 * A sharded job all-reduces S.  lrvb_spd_inverse then gives (H^{-1})_gg = S^{-1}, the
 * linear-response covariance of the global parameters (the role of
 * -cho_solve(cho_factor(H), .) in ModelSensitivity.py:594-602). */
int lrvb_glmm_schur(lrvb_glmm* h, double* S_dev, int32_t include_A, void* stream);
/* In-place Cholesky inverse of an SPD (n,n) matrix on the device.  info_host: 0 ok,
 * k>0 = leading minor k not positive.  Syncs. */
int lrvb_spd_inverse(double* S_dev, int32_t n, int32_t* info_host, void* stream);
/* x = H^{-1} b for nrhs right-hand sides (row-major (nrhs, D), dev) by block elimination,
 * given Sinv = S^{-1} from above.  The local part uses this handle's groups; a sharded job
 * first all-reduces rhs_g = b_g - sum_g B_g^T L_g^{-1} b_l (lrvb_glmm_solve_reduce_rhs). */
int lrvb_glmm_solve_reduce_rhs(lrvb_glmm* h, const double* b_dev, int32_t nrhs,
                               double* rhs_g_dev, int32_t include_bg, void* stream);
int lrvb_glmm_solve_finish(lrvb_glmm* h, const double* Sinv_dev, const double* rhs_g_dev,
                           const double* b_dev, int32_t nrhs, double* x_dev, void* stream);
/* Marginal LRVB covariance of every group's (u.mean_g, u.info_g): (G,3) as (mm, mi, ii):
 *   L_g^{-1} + L_g^{-1} B_g S^{-1} B_g^T L_g^{-1}. */
int lrvb_glmm_local_cov(lrvb_glmm* h, const double* Sinv_dev, double* cov_dev, void* stream);

/* ---- prediction on new rows ---------------------------------------------------------------
 * At the free point free_dev (D,) (free coordinates; no evaluation over the training rows is needed), for M
 * new rows X_dev (M,K) row-major fp64 (16-byte aligned,
 * K must equal the handle's K) with group ids g_dev (M,) int32 in [-1, G) (-1 = population level: mu in
 * place of u_g).  order_dev (M,) int64 or NULL: the order in which the rows are visited, a permutation of
 * [0, M) (e.g. a stable sort by group, so that rows of one group read its blocks from cache); every row is
 * read from and written to its own place, so the result does not depend on it.  Output:
 *   out_dev (4, M) row-major = [eta_mean, eta_var_mfvb, prob, prob_var_mfvb]
 * with eta = u_g + x.beta under q and prob = E_q[sigma(eta)] by the model's Gauss-Hermite rule.
 * A row whose group id is outside [-1, G) gets NaN.  LRVB_EINVAL for a K other than the handle's, M < 0,
 * NULL pointers or an X that is not 16-byte aligned. */
int lrvb_glmm_predict(lrvb_glmm* h, const double* free_dev, const double* X_dev, int32_t K, const int32_t* g_dev, const int64_t* order_dev,
                      int64_t M, double* out_dev, void* stream);
/* The block of H^-1 between beta and every group's (u.mean_g, u.info_g), cross_dev (G, 2, 2K):
 * cross[g][r][j] = (H^-1)[4 + j, (u.mean_g, u.info_g)_r] = -(S^-1 B_g^T L_g^-1)[4 + j, r], given
 * Sinv_dev = S^-1 (lrvb_glmm_schur + lrvb_spd_inverse).  Once per optimum.  Needs a cached Hessian in
 * free coordinates (LRVB_ESTATE otherwise). */
int lrvb_glmm_predict_cross(lrvb_glmm* h, const double* Sinv_dev, double* cross_dev, void* stream);
/* lrvb_glmm_predict plus the linear-response variances j H^-1 j^T of prob and eta (j = their gradient
 * with respect to the free parameters) from the arrowhead pieces Sinv_dev (Dg,Dg), cross_dev (above) and
 * localcov_dev (G,3) (lrvb_glmm_local_cov): out_dev (6, M) = [eta_mean, eta_var_mfvb, prob,
 * prob_var_mfvb, prob_var_lr, eta_var_lr].  The quadratic forms run on the FP64 tensor cores.  Needs a
 * cached Hessian in free coordinates (LRVB_ESTATE otherwise); allocates a (3K x K) scratch in the
 * handle on first use. */
int lrvb_glmm_predict_lr(lrvb_glmm* h, const double* Sinv_dev, const double* cross_dev, const double* localcov_dev,
                         const double* X_dev, int32_t K, const int32_t* g_dev, const int64_t* order_dev, int64_t M,
                         double* out_dev, void* stream);
/* Approximate leave-one-out cross-validation of the handle's own N training rows by the infinitesimal jackknife,
 * at the cached Hessian (an order-2 evaluation in free coordinates, normally at the optimum; LRVB_ESTATE
 * otherwise), from the same arrowhead pieces as lrvb_glmm_predict_lr.  For row n, with z = u_g + x.beta under q,
 * Q_n = [j_m; j_v] H^-1 [j_m; j_v]^T (j_m, j_v = d E[z] / d free, d Var[z] / d free) and W_m, W_v = rows 0, 1 of
 * lrvb_glmm_obs_weights (w_n dl_n/dz_m, w_n dl_n/dz_v of the same evaluation), dropping the row shifts its
 * moments by (dz_m, dz_v) = -Q_n (W_m, W_v).  Output, in the handle's (group-sorted) row order:
 *   out_dev (4, N) row-major = [lpd, lpd_loo, eta_mean_loo, eta_var_loo]
 * with lpd = log E_q[p(y_n | z)] by the model's Gauss-Hermite rule (y = 0 as log E[sigma(-z)]), lpd_loo the
 * same at the shifted moments, eta_*_loo = the shifted moments.  A row whose shifted variance is <= 0 gets NaN
 * in lpd_loo and eta_var_loo.  y must be 0 or 1 (any y != 0 counts as 1).  No atomics: repeated calls are
 * bitwise equal.  LRVB_EINVAL for NULL pointers; uses the scratch of lrvb_glmm_predict_lr. */
int lrvb_glmm_loo(lrvb_glmm* h, const double* Sinv_dev, const double* cross_dev, const double* localcov_dev,
                  double* out_dev, void* stream);
/* Approximate leave-one-group-out cross-validation and group influence by the infinitesimal jackknife, at the cached
 * Hessian (an order-2 evaluation in free coordinates, normally at the optimum; LRVB_ESTATE otherwise).  Dropping
 * group g (w_n -> 0 on its rows) shifts the globals by delta_g = -S^-1 (v_glob - B_g^T L_g^-1 v_loc), v = the group's
 * data gradient from W rows 0, 1 (lrvb_glmm_obs_weights).  Sinv_dev = S^-1 (Dg,Dg), Pinv_dev = the inverse of its
 * (K,K) block on E[beta].  Output:
 *   delta_dev     (G, Dg) row-major: delta_g
 *   group_out_dev (2, G)  row-major: [cook_g = delta_beta,g^T P^-1 delta_beta,g / K, elpd_logo_group]
 *   row_out_dev   (3, N)  row-major, the handle's (group-sorted) row order: [lpd_logo, eta_mean_logo, eta_var_logo]
 * with the globals at theta + delta_g mapped exactly to constrained values, q(u_g) at its optimum without the group's
 * rows (mean E[mu]', info max(E[tau]', lb_u)), eta = u_g + x.beta under that q and lpd_logo = log E_q[p(y_n | eta)]
 * by the model's Gauss-Hermite rule (y = 0 as log E[sigma(-eta)]).  An empty group gets delta = 0, cook = 0 and
 * elpd_logo_group = 0.  No atomics: repeated calls are bitwise equal.  LRVB_EINVAL for NULL pointers; allocates a
 * (G, Dg) scratch in the handle on first use. */
int lrvb_glmm_logo(lrvb_glmm* h, const double* Sinv_dev, const double* Pinv_dev, double* delta_dev,
                   double* group_out_dev, double* row_out_dev, void* stream);
/* The third derivative of the KL along a_dev (D), at the point of the last evaluation (free coordinates;
 * LRVB_ESTATE otherwise): t_dev (D) = D^3 KL[a, a, .] and q_dev (N) = a^T (grad^2 l_n) a, the unweighted per-row
 * quadratic form, in the handle's (group-sorted) row order.  With a = H^-1 c it gives how the LRVB variance
 * c^T H^-1 c moves with the observation weights: d/dw_n = q_n - grad l_n . (H^-1 t).  No atomics: repeated calls are
 * bitwise equal.  LRVB_EINVAL for NULL pointers; allocates a (2N + 5G + O(K)) scratch in the handle on first use. */
int lrvb_glmm_third_contract(lrvb_glmm* h, const double* a_dev, double* t_dev, double* q_dev, void* stream);
/* The "meat" of the infinitesimal-jackknife (IJ) bootstrap covariance of the global parameters, at the cached Hessian
 * (an order-2 evaluation in free coordinates, normally at the optimum; LRVB_ESTATE otherwise).  The IJ influence of
 * a unit u (a row, unit = 0, or a whole group, unit = 1) on the globals is S^-1 V_u with V_u = v_glob - B_g^T L_g^-1
 * v_loc, v = the unit's data gradient from W rows 0, 1 (lrvb_glmm_obs_weights), as in lrvb_glmm_logo.  Output:
 *   meat_dev (Dg, Dg) row-major: sum_u V_u V_u^T, exactly symmetric
 *   sum_dev  (Dg):               s = sum_u V_u (the same for both units: the column sums of the groups' V)
 * so that the IJ covariance of the globals is S^-1 (meat - s s^T / U) S^-1 with U = the units of non-zero weight.
 * Rows of weight 0 have V_u = 0 exactly.  No atomics: repeated calls are bitwise equal; nothing a later evaluation,
 * solve or IJ call reads is changed.  LRVB_EINVAL for NULL pointers or a unit other than 0 or 1; allocates a scratch
 * of about 5 N + G (4K + 3 Dg) doubles in the handle on first use. */
int lrvb_glmm_ij_meat(lrvb_glmm* h, int32_t unit, double* meat_dev, double* sum_dev, void* stream);

/* ---- batched exponential-family terms (ExponentialFamilies.py) --------------------------
 * All pointers dev; M = number of factors. */
/* :33-35 gamma_entropy per factor, out (M,). */
int lrvb_ef_gamma_entropy(const double* shape, const double* rate, int64_t M, double* out,
                          void* stream);
/* :111-112 get_e_log_gamma, out (M,). */
int lrvb_ef_e_log_gamma(const double* shape, const double* rate, int64_t M, double* out,
                        void* stream);
/* :33-35 and :111-112 in one pass over (shape, rate) -- they share digamma(shape) and log(rate):
 * entropy (M,) and / or e_log (M,); either may be NULL. */
int lrvb_ef_gamma_terms(const double* shape, const double* rate, int64_t M, double* entropy,
                        double* e_log, void* stream);
/* :43-52 and :118-120 in one pass over alpha (d, M): entropy (M,) and / or e_log (d, M); either may be NULL. */
int lrvb_ef_dirichlet_terms(const double* alpha, int32_t d, int64_t M, double* entropy, double* e_log,
                            void* stream);
/* :23-25 univariate_normal_entropy per factor (the reference sums them), out (M,). */
int lrvb_ef_uvn_entropy(const double* info, int64_t M, double* out, void* stream);
/* :43-52 dirichlet_entropy: alpha (d, M) row-major, simplex dimension is axis 0; out (M,). */
int lrvb_ef_dirichlet_entropy(const double* alpha, int32_t d, int64_t M, double* out,
                              void* stream);
/* :118-120 get_e_log_dirichlet: out (d, M). */
int lrvb_ef_e_log_dirichlet(const double* alpha, int32_t d, int64_t M, double* out,
                            void* stream);
/* :54-69 beta_entropy per row of tau (M,2) row-major (the reference sums them); out (M,). */
int lrvb_ef_beta_entropy(const double* tau, int64_t M, double* out, void* stream);
/* :72-82 wishart_entropy, :88-94 e_log_det_wishart, :97-102 e_log_inv_wishart_diag batched
 * over M factors: df (M,), v (M,k,k) row-major SPD, k <= 8.
 * entropy (M,) / e_log_det (M,) / e_log_inv_diag (M,k); any output may be NULL. */
int lrvb_ef_wishart(const double* df, const double* v, int32_t k, int64_t M, double* entropy,
                    double* e_log_det, double* e_log_inv_diag, void* stream);
/* :20-21 multinoulli_entropy: p (M, d) row-major, out (M,). */
int lrvb_ef_multinoulli_entropy(const double* p, int32_t d, int64_t M, double min_prob,
                                double* out, void* stream);
/* Modeling.py:35-52 get_e_logistic_term_guass_hermite with aggregate_all=False:
 * z_mean, z_sd dev (M,), gh_x / gh_w HOST (Q,), out dev (M,). */
int lrvb_gh_logistic_term(const double* z_mean, const double* z_sd, int64_t M,
                          const double* gh_x_host, const double* gh_w_host, int32_t Q,
                          double* out, void* stream);
/* Deterministic sum of a device vector into out_dev[0] (used to aggregate the terms above
 * the way the reference's np.sum does). */
int lrvb_sum(const double* x_dev, int64_t M, double* out_dev, void* stream);

/* ---- matrix- and simplex-valued parameter types, batched (MatrixParameters.py, SimplexParams.py)
 * All pointers dev, row-major; M = number of parameters; v = k (k + 1) / 2, packed lower triangle
 * in numpy.tril_indices order ((0,0), (1,0), (1,1), (2,0), ...); k <= 8, 2 <= d <= 64.
 * The reference handles one matrix / one simplex row per Python iteration
 * (MatrixParameters.py:236-249, SimplexParams.py:105-150) and differentiates with autograd. */
/* :122-127 unpack_posdef_matrix: free (M, v) -> mat (M, k, k) = L L^T + diag_lb I with
 * L = exp_matrix_diagonal(unvectorize_ld_matrix(free)). */
int lrvb_posdef_unpack(const double* free_dev, int32_t k, int64_t M, double diag_lb, double* mat_dev,
                       void* stream);
/* :114-119 pack_posdef_matrix: mat (M, k, k) (lower triangle read) -> free (M, v).  A matrix with
 * mat - diag_lb I not positive definite gives NaN and is counted in *not_posdef_dev (nullable,
 * int32, caller zeroes it) where numpy.linalg.cholesky raises. */
int lrvb_posdef_pack(const double* mat_dev, int32_t k, int64_t M, double diag_lb, double* free_dev,
                     int32_t* not_posdef_dev, void* stream);
/* :145-147 pos_def_matrix_free_to_vector: free (M, v) -> vectorize_ld_matrix(unpack(free)) (M, v). */
int lrvb_posdef_free_to_vector(const double* free_dev, int32_t k, int64_t M, double diag_lb,
                               double* vec_dev, void* stream);
/* :149-152 its Jacobian (M, v, v), jac[m][r][c] = d vec_r / d free_c, and Hessian (M, v, v, v),
 * hess[m][r][c1][c2]; the blocks PosDefMatrixParamVector.free_to_vector_jac / _hess (:251-297)
 * scatter into block-diagonal sparse matrices. */
int lrvb_posdef_free_to_vector_jac(const double* free_dev, int32_t k, int64_t M, double diag_lb,
                                   double* jac_dev, void* stream);
int lrvb_posdef_free_to_vector_hess(const double* free_dev, int32_t k, int64_t M, double diag_lb,
                                    double* hess_dev, void* stream);
/* SimplexParams.py:11-18 constrain_simplex_matrix: free (M, d-1) -> z (M, d), softmax of [0, free]. */
int lrvb_simplex_constrain(const double* free_dev, int64_t M, int32_t d, double* z_dev, void* stream);
/* :21-23 unconstrain_simplex_matrix: z (M, d) -> free (M, d-1). */
int lrvb_simplex_unconstrain(const double* z_dev, int64_t M, int32_t d, double* free_dev, void* stream);
/* :33-38 constrain_grad_from_moment per row: jac (M, d, d-1); :42-63 constrain_hess_from_moment:
 * hess (M, d, d-1, d-1) -- both taken at z = constrain(free). */
int lrvb_simplex_jac(const double* free_dev, int64_t M, int32_t d, double* jac_dev, void* stream);
int lrvb_simplex_hess(const double* free_dev, int64_t M, int32_t d, double* hess_dev, void* stream);

/* ---- all-reduce of the replicated blocks over NVLink peer memory ---------------------------
 * The reference has no distributed path (SURVEY.md 8e is new): an observation-sharded job sums
 * [KL, grad_g, H_gg] (lrvb_glmm_eval's out_global), the global rows of an HVP, the Schur
 * complement and CG's dot products over the ranks.  These messages are tens of KB, so the cost
 * is latency: one kernel per rank pushes its block into a window of every peer (CUDA IPC, one
 * process per GPU), waits for the peers' blocks and adds them in rank order -- bitwise identical
 * on every rank.  csrc/p2p.cu.
 *  create:   allocates this rank's window for messages of up to max_elems doubles (syncs);
 *  export:   writes lrvb_p2p_handle_bytes() bytes the peers need to map the window
 *            (exchanged by the host, e.g. torch.distributed.all_gather_object);
 *  connect:  handles = world * lrvb_p2p_handle_bytes() bytes, rank-major; maps the peers;
 *  allreduce_sum: in place on buf_dev (n <= max_elems), enqueued on `stream`; EVERY rank must
 *            issue the same sequence of calls;
 *  status:   0, or 1 + r when rank r did not arrive within the deadline (default 120 s; environment
 *            LRVB_P2P_TIMEOUT_S at create, or lrvb_p2p_set_timeout).  The word lives in mapped pinned
 *            HOST memory and is sticky: a timed-out call fills its output with NaN and returns (no
 *            trap, the CUDA context survives), every later lrvb_p2p_allreduce_sum returns LRVB_ESTATE.
 *            lrvb_p2p_status syncs the stream first; _nowait just reads the word.
 *  set_stats / get_stats: when enabled every call measures, inside the kernel (%globaltimer around
 *            the poll loops, maximum over all elements), how long this rank WAITED for its slowest
 *            peer; get_stats (syncs) returns out3 = {calls, sum of the per-call waits (us), largest
 *            per-call wait (us)} since set_stats -- bench.py's collective_wait_us. */
typedef struct lrvb_p2p lrvb_p2p;
int lrvb_p2p_create(lrvb_p2p** out, int32_t rank, int32_t world, int64_t max_elems);
int lrvb_p2p_handle_bytes(void);
int lrvb_p2p_export(lrvb_p2p* h, void* handle_out);
int lrvb_p2p_connect(lrvb_p2p* h, const void* handles);
int lrvb_p2p_allreduce_sum(lrvb_p2p* h, double* buf_dev, int64_t n, void* stream);
int lrvb_p2p_status(lrvb_p2p* h, int32_t* status_out, void* stream);
int lrvb_p2p_status_nowait(lrvb_p2p* h, int32_t* status_out);
int lrvb_p2p_set_timeout(lrvb_p2p* h, double seconds);
int lrvb_p2p_set_stats(lrvb_p2p* h, int32_t enable, void* stream);
int lrvb_p2p_get_stats(lrvb_p2p* h, double* out3_host, void* stream);
int lrvb_p2p_destroy(lrvb_p2p* h);
/* ConjugateGradientSolver.get_hinv_vec (ConjugateGradient.py:81-85) over the shards of one job:
 * lrvb_glmm_cg on vectors in the shard's local layout [globals | u.mean | u.info of the shard's
 * groups] (globals replicated on every rank), with two peer all-reduces per iteration
 * ([r.r, r.z] and [(H p)_g, p_l.q_l]).  root = 1 on the one rank that counts the global entries
 * in dot products and adds the (all-reduced) global block A in the Hessian-vector product.
 * Every rank calls it with the same precond / rtol / maxiter (> 0; scipy's default is 10 x the
 * dimension of the whole job).  info / iters as lrvb_glmm_cg.  Syncs every 8 iterations. */
int lrvb_glmm_cg_sharded(lrvb_glmm* h, lrvb_p2p* comm, const double* b_dev, const double* x0_dev,
                         int32_t precond, double rtol, int32_t maxiter, int32_t root, double* x_dev,
                         int32_t* info_host, int32_t* iters_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LRVB_B200_H */
