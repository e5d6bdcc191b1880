"""Analytic fp64 oracle of approximate leave-one-out cross-validation by the infinitesimal jackknife (IJ) for
small D (numpy / scipy).  TEST INFRASTRUCTURE.

Training row n in group g has the moments z_m = E[u_g] + x.E[beta], z_v = Var[u_g] + x^2.Var[beta] and the
log-likelihood term l_n(z_m, z_v) = y_n z_m - E_q[log(1 + e^z)] (glmm_oracle.obs_terms).  Its gradient with
respect to the free parameters is l_m j_m + l_v j_v with

    j_m = d z_m / d free:  x on beta.mean, 1 on u.mean_g
    j_v = d z_v / d free:  s x^2 on beta.info (s_k = -(i_k - lb) / i_k^2), d_g on u.info_g (d_g likewise)

so with the dense inverse of the oracle Hessian the IJ estimate of the optimum without row n is
theta - w_n H^-1 grad l_n, and the row's moments move by (dz_m, dz_v) = -Q_n (w_n l_m, w_n l_v),
Q_n = [j_m; j_v] H^-1 [j_m; j_v]^T.  lpd = log E_q[p(y_n | z)] by the model's Gauss-Hermite rule, with
y = 0 evaluated as log E[sigma(-z)].
"""
import numpy as np
import scipy.special

from . import predict_oracle as po


def _lb(oracle):
    b = oracle.bounds
    return dict(mu_info=b.mu_info, beta_info=b.beta_info, u_info=b.u_info)


def moment_jacobians(free, X, g, K, G, lower_bounds=None):
    """(J_m, J_v): dense (M, D) d z_m / d free and d z_v / d free of rows X (M, K) in groups g (g = -1: mu)."""
    J_m = po.prediction_jacobian(free, X, g, K, G, np.zeros(1), np.ones(1), lower_bounds, quantity="eta").toarray()
    lb = po._bounds(lower_bounds)
    free, X, g = po._check(free, X, g, K, G)
    M, Dg, D = X.shape[0], 4 + 2 * K, 4 + 2 * K + 2 * G
    p = po._params(free, K, G, lb)
    _, _, info = po._offset(p, g)
    d = -(info - np.where(g < 0, lb["mu_info"], lb["u_info"])) / (info * info)
    s = -(p["beta_i"] - lb["beta_info"]) / (p["beta_i"] ** 2)
    J_v = np.zeros((M, D))
    J_v[:, 4 + K:Dg] = X * X * s[None, :]
    J_v[np.arange(M), np.where(g < 0, 1, Dg + G + g)] = d
    return J_m, J_v


def log_predictive_density(z_m, z_v, y, gh_x, gh_w):
    """log E[p(y | z)] for z ~ N(z_m, z_v): log E[sigma(z)] (y = 1) or log E[sigma(-z)] (y = 0); NaN where z_v <= 0."""
    z_m, z_v, y = (np.asarray(a, dtype=np.float64) for a in (z_m, z_v, y))
    ok = z_v > 0
    m = np.where(y == 0, -z_m, z_m)
    what = np.asarray(gh_w, dtype=np.float64) / np.sqrt(np.pi)
    c = np.sqrt(2.0) * np.asarray(gh_x, dtype=np.float64)
    t = m[:, None] + np.sqrt(np.where(ok, z_v, 1.0))[:, None] * c[None, :]
    return np.where(ok, np.log(np.sum(what * scipy.special.expit(t), axis=1)), np.nan)


def row_terms(oracle, free):
    """z_m, z_v and the weighted W_m = w l_m, W_v = w l_v of every training row of the oracle (its row order)."""
    o = oracle.obs_terms(oracle.unpack(oracle.free_to_vector(free)), order=1)
    return o["z_m"], o["z_v"], o["l_m"], o["l_v"]


def q_dense(oracle, free, Hinv):
    """(Q_mm, Q_mv, Q_vv) (N,) each: [j_m; j_v] H^-1 [j_m; j_v]^T of every training row, from the dense H^-1."""
    J_m, J_v = moment_jacobians(free, oracle.X, oracle.g, oracle.K, oracle.G, _lb(oracle))
    HJ_m, HJ_v = J_m @ Hinv, J_v @ Hinv
    return np.sum(HJ_m * J_m, axis=1), np.sum(HJ_m * J_v, axis=1), np.sum(HJ_v * J_v, axis=1)


def q_from_pieces(oracle, free):
    """Q_n assembled as csrc/predict.cu assembles it, from the arrowhead pieces of H^-1 only: P = S^-1 on beta,
    C_g = -(S^-1 T_g^T) on beta (T_g = L_g^-1 B_g), Sigma_g = L_g^-1 + T_g S^-1 T_g^T, and the forms
    vm = x P_mm x, vs = x P_ms x~, vq = x~ P_ss x~ (x~ = s x^2), cm_r = x.C_g[beta.mean, r], cs_r = x~.C_g[beta.info, r]."""
    K, G, Dg = oracle.K, oracle.G, 4 + 2 * oracle.K
    _, _, blk = oracle.kl_blocks(free)
    Sinv, _ = oracle.schur_global_cov(free)
    B, L = blk["B"], blk["L"]
    det = L[:, 0] * L[:, 2] - L[:, 1] ** 2
    Linv = np.stack([np.stack([L[:, 2], -L[:, 1]], -1), np.stack([-L[:, 1], L[:, 0]], -1)], 1) / det[:, None, None]
    T = Linv @ B                                                  # (G, 2, Dg)
    C = -np.einsum("ij,gri->gjr", Sinv, T)                        # (G, Dg, 2): H^-1[global, (u.mean_g, u.info_g)]
    Sig = Linv + T @ Sinv @ np.transpose(T, (0, 2, 1))            # (G, 2, 2)
    p = po._params(np.asarray(free, dtype=np.float64), K, G, _lb(oracle))
    lb = _lb(oracle)
    s = -(p["beta_i"] - lb["beta_info"]) / p["beta_i"] ** 2
    X, g = oracle.X, oracle.g
    xt = X * X * s[None, :]
    bm, bi = slice(4, 4 + K), slice(4 + K, Dg)
    vm = np.sum((X @ Sinv[bm, bm]) * X, axis=1)
    vs = np.sum((X @ Sinv[bm, bi]) * xt, axis=1)
    vq = np.sum((xt @ Sinv[bi, bi]) * xt, axis=1)
    Cg = C[g]
    cm0, cm1 = np.sum(X * Cg[:, bm, 0], axis=1), np.sum(X * Cg[:, bm, 1], axis=1)
    cs0, cs1 = np.sum(xt * Cg[:, bi, 0], axis=1), np.sum(xt * Cg[:, bi, 1], axis=1)
    s00, s01, s11 = Sig[g, 0, 0], Sig[g, 0, 1], Sig[g, 1, 1]
    info = p["u_i"][g]
    d = -(info - lb["u_info"]) / (info * info)
    return vm + 2 * cm0 + s00, vs + d * cm1 + cs0 + d * s01, vq + 2 * d * cs1 + d * d * s11


def theta_shift(oracle, free, n, Hinv):
    """-w_n H^-1 grad l_n (D,): the IJ change of the optimum when training row n (oracle order) is dropped."""
    J_m, J_v = moment_jacobians(free, oracle.X[n:n + 1], oracle.g[n:n + 1], oracle.K, oracle.G, _lb(oracle))
    _, _, W_m, W_v = row_terms(oracle, free)
    return -Hinv @ (W_m[n] * J_m[0] + W_v[n] * J_v[0])


def approximate_loo(oracle, free, Hinv=None):
    """dict with the pointwise lpd, lpd_loo, eta_mean_loo, eta_var_loo (N,) in the oracle's row order and the
    scalars elpd_loo, elpd_loo_se, p_loo, n_invalid, plus the shifts dz_m, dz_v."""
    if np.any((oracle.y != 0) & (oracle.y != 1)):
        raise ValueError("approximate LOO needs a binary training y")
    if Hinv is None:
        Hinv = np.linalg.inv(oracle.kl_hessian_dense(free))
    q_mm, q_mv, q_vv = q_dense(oracle, free, Hinv)
    z_m, z_v, W_m, W_v = row_terms(oracle, free)
    dz_m = -(q_mm * W_m + q_mv * W_v)
    dz_v = -(q_mv * W_m + q_vv * W_v)
    zm1, zv1 = z_m + dz_m, z_v + dz_v
    lpd = log_predictive_density(z_m, z_v, oracle.y, oracle.gh_x, oracle.gh_w)
    lpd_loo = log_predictive_density(zm1, zv1, oracle.y, oracle.gh_x, oracle.gh_w)
    N = lpd.size
    elpd = float(np.sum(lpd_loo))
    return dict(lpd=lpd, lpd_loo=lpd_loo, eta_mean_loo=zm1, eta_var_loo=np.where(zv1 > 0, zv1, np.nan),
                elpd_loo=elpd, p_loo=float(np.sum(lpd)) - elpd,
                elpd_loo_se=float(np.sqrt(N) * np.std(lpd_loo, ddof=1)) if N > 1 else float("nan"),
                n_invalid=int(np.sum(~(zv1 > 0))), dz_m=dz_m, dz_v=dz_v)
