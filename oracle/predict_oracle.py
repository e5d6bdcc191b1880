"""Analytic fp64 oracle of GLMM prediction on new rows (numpy / scipy).  TEST INFRASTRUCTURE.

For a new row with covariates x (K) and group g, at the free point ``free`` of a model with K
covariates and G groups (flat layout of glmm_oracle.Layout):

    z_m = E[u_g] + x.E[beta],   z_v = Var[u_g] + x^2.Var[beta]     (g = -1: mu in place of u_g)
    t_q = z_m + sqrt(2 z_v) xi_q,   what_q = w_q / sqrt(pi)          (hermgauss nodes, as in training)
    p  = sum what sigma(t_q)                 p2 = sum what sigma(t_q)^2
    a  = sum what sigma'(t_q) = dp/dz_m      b  = sum what sigma'(t_q) sqrt(2) xi_q / (2 sqrt(z_v)) = dp/dz_v

The Jacobian row of p with respect to the free parameters has a x on beta.mean, b x~ on beta.info
(x~_k = -x_k^2 (i_k - lb) / i_k^2), a on u.mean_g and b d_g on u.info_g (d_g = -(i_g - lb) / i_g^2);
that of eta = z_m is the same with a = 1, b = 0.
"""
import numpy as np
import scipy.sparse
import scipy.special


def _check(free, X, g, K, G):
    free = np.asarray(free, dtype=np.float64).reshape(-1)
    X = np.asarray(X, dtype=np.float64).reshape(-1, K)
    g = np.asarray(g, dtype=np.int64).reshape(-1)
    if free.size != 4 + 2 * K + 2 * G:
        raise ValueError("free has %d entries, expected %d" % (free.size, 4 + 2 * K + 2 * G))
    if g.size != X.shape[0] or (g.size and (g.min() < -1 or g.max() >= G)):
        raise ValueError("group ids must be one per row, in [-1, G)")
    return free, X, g


def _params(free, K, G, lb):
    """Constrained means / infos and d info / d free = info - lb."""
    Dg = 4 + 2 * K
    mu_i = np.exp(free[1]) + lb["mu_info"]
    beta_i = np.exp(free[4 + K:Dg]) + lb["beta_info"]
    u_i = np.exp(free[Dg + G:]) + lb["u_info"]
    return dict(mu_m=free[0], mu_i=mu_i, beta_m=free[4:4 + K], beta_i=beta_i,
                u_m=free[Dg:Dg + G], u_i=u_i)


def _bounds(lower_bounds):
    lb = dict(mu_info=0.0, beta_info=0.0, u_info=0.0)
    if lower_bounds is not None:
        lb.update({k: float(v) for k, v in dict(lower_bounds).items() if k in lb})
    return lb


def _offset(p, g):
    """(E, Var, info) of the random effect of every row: u_g, or mu for g = -1."""
    pop = g < 0
    gi = np.where(pop, 0, g)
    e = np.where(pop, p["mu_m"], p["u_m"][gi] if p["u_m"].size else 0.0)
    info = np.where(pop, p["mu_i"], p["u_i"][gi] if p["u_i"].size else 1.0)
    return e, 1.0 / info, info


def predict(free, X, g, K, G, gh_x, gh_w, lower_bounds=None):
    """dict of (M,) arrays: eta_mean, eta_var_mfvb, prob, prob_var_mfvb, and a = dp/dz_m, b = dp/dz_v."""
    lb = _bounds(lower_bounds)
    free, X, g = _check(free, X, g, K, G)
    p = _params(free, K, G, lb)
    e, v, _ = _offset(p, g)
    z_m = e + X @ p["beta_m"]
    z_v = v + (X * X) @ (1.0 / p["beta_i"])
    z_s = np.sqrt(z_v)
    what = np.asarray(gh_w, dtype=np.float64) / np.sqrt(np.pi)
    c = np.sqrt(2.0) * np.asarray(gh_x, dtype=np.float64)
    t = z_m[:, None] + z_s[:, None] * c[None, :]
    sg = scipy.special.expit(t)
    dsg = sg * (1.0 - sg)
    prob = np.sum(what * sg, axis=1)
    p2 = np.sum(what * sg * sg, axis=1)
    a = np.sum(what * dsg, axis=1)
    b = np.sum(what * dsg * c, axis=1) / (2.0 * z_s)
    return dict(eta_mean=z_m, eta_var_mfvb=z_v, prob=prob, prob_var_mfvb=p2 - prob * prob, a=a, b=b)


def prediction_jacobian(free, X, g, K, G, gh_x, gh_w, lower_bounds=None, quantity="prob"):
    """d quantity / d free as scipy CSR (M, D), quantity 'prob' or 'eta'."""
    if quantity not in ("prob", "eta"):
        raise ValueError("quantity must be 'prob' or 'eta'")
    lb = _bounds(lower_bounds)
    free, X, g = _check(free, X, g, K, G)
    M, Dg, D = X.shape[0], 4 + 2 * K, 4 + 2 * K + 2 * G
    p = _params(free, K, G, lb)
    if quantity == "prob":
        r = predict(free, X, g, K, G, gh_x, gh_w, lower_bounds)
        a, b = r["a"], r["b"]
    else:
        a, b = np.ones(M), np.zeros(M)
    _, _, info = _offset(p, g)
    off_lb = np.where(g < 0, lb["mu_info"], lb["u_info"])
    d = -(info - off_lb) / (info * info)
    xt = -(X * X) * ((p["beta_i"] - lb["beta_info"]) / (p["beta_i"] ** 2))[None, :]
    col_m = np.where(g < 0, 0, Dg + g)
    col_i = np.where(g < 0, 1, Dg + G + g)
    rows = np.repeat(np.arange(M), 2 * K + 2)
    cols = np.concatenate([np.tile(np.arange(4, Dg), (M, 1)), col_m[:, None], col_i[:, None]], axis=1)
    vals = np.concatenate([a[:, None] * X, b[:, None] * xt, a[:, None], (b * d)[:, None]], axis=1)
    return scipy.sparse.csr_matrix((vals.reshape(-1), (rows, cols.reshape(-1))), shape=(M, D))


def lr_variances(J, Hinv):
    """diag(J H^-1 J^T) for a (M, D) Jacobian and the dense inverse Hessian."""
    J = scipy.sparse.csr_matrix(J)
    return np.asarray(J.multiply(J @ Hinv).sum(axis=1)).reshape(-1)
