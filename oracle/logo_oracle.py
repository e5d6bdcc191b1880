"""Analytic fp64 oracle of approximate leave-one-group-out (LOGO) cross-validation and group influence by the
infinitesimal jackknife (IJ) for small D (numpy / scipy).  TEST INFRASTRUCTURE.

Dropping group g is w_n -> 0 on its rows.  The group's data gradient in free coordinates is
v_g = sum_{n in g} (W_m j_m + W_v j_v) with W_m = w l_m, W_v = w l_v and the row Jacobians of loo_oracle, so the IJ
estimate of the optimum without the group is theta - H^-1 v_g; delta_g is its global block (Dg).  With the globals at
theta + delta_g (mapped exactly to constrained values) and q(u_g) at its optimum without the group's rows
(mean E[mu]', info max(E[tau]', lb_u), E[tau]' = shape' / rate'), every row n of g gets
z_m = E[mu]' + x.E[beta]', z_v = 1 / info' + x^2.Var[beta]' and lpd_logo = log E_q[p(y_n | z)].
Cook's distance: delta_beta^T P^-1 delta_beta / K with P = (H^-1)[beta.mean, beta.mean].
"""
import numpy as np

from . import loo_oracle as lo


def group_gradients(oracle, free):
    """v (G, D): the data gradient sum_{n in g} (W_m j_m + W_v j_v) of every group, dense."""
    J_m, J_v = lo.moment_jacobians(free, oracle.X, oracle.g, oracle.K, oracle.G, lo._lb(oracle))
    _, _, W_m, W_v = lo.row_terms(oracle, free)
    v = np.zeros((oracle.G, oracle.lay.D))
    np.add.at(v, oracle.g, W_m[:, None] * J_m + W_v[:, None] * J_v)
    return v


def theta_shifts(oracle, free, Hinv):
    """dtheta (G, D) = -H^-1 v_g: the IJ change of the whole optimum when group g is dropped (dense H^-1)."""
    return -group_gradients(oracle, free) @ Hinv


def delta_arrowhead(oracle, free):
    """delta (G, Dg) = -S^-1 (v_glob - B_g^T L_g^-1 v_loc), as csrc/logo.cu assembles it from the arrowhead blocks."""
    lay, G, Dg = oracle.lay, oracle.G, oracle.lay.Dg
    _, _, blk = oracle.kl_blocks(free)
    Sinv, _ = oracle.schur_global_cov(free)
    v = group_gradients(oracle, free)
    gi = np.arange(G)
    vloc = np.stack([v[gi, lay.u_mean + gi], v[gi, lay.u_info + gi]], axis=1)        # (G, 2)
    L = blk["L"]
    det = L[:, 0] * L[:, 2] - L[:, 1] ** 2
    t0 = (L[:, 2] * vloc[:, 0] - L[:, 1] * vloc[:, 1]) / det
    t1 = (-L[:, 1] * vloc[:, 0] + L[:, 0] * vloc[:, 1]) / det
    V = v[:, :Dg] - (blk["B"][:, 0, :] * t0[:, None] + blk["B"][:, 1, :] * t1[:, None])
    return -V @ Sinv


def shifted_globals(oracle, free, delta):
    """Constrained globals at free[:Dg] + delta: dict(mu_m, e_tau, beta_m, beta_i)."""
    Dg, K = oracle.lay.Dg, oracle.K
    lb = oracle.lower_bounds()[:Dg]
    f = np.asarray(free, dtype=np.float64)[:Dg] + delta
    con = np.isfinite(lb)
    vec = f.copy()
    vec[con] = np.exp(f[con]) + lb[con]
    return dict(mu_m=vec[0], e_tau=vec[2] / vec[3], beta_m=vec[4:4 + K], beta_i=vec[4 + K:Dg])


def held_out_moments(oracle, glob, rows):
    """(z_m, z_v) of the training rows `rows` (one group) with q(u_g) at its optimum given the globals `glob`."""
    info = max(glob["e_tau"], oracle.bounds.u_info)
    X = oracle.X[rows]
    return glob["mu_m"] + X @ glob["beta_m"], 1.0 / info + (X * X) @ (1.0 / glob["beta_i"])


def held_out_lpd(oracle, glob, rows):
    z_m, z_v = held_out_moments(oracle, glob, rows)
    return lo.log_predictive_density(z_m, z_v, oracle.y[rows], oracle.gh_x, oracle.gh_w)


def approximate_logo(oracle, free, Hinv=None):
    """dict with lpd_logo, eta_mean_logo, eta_var_logo (N,) in the oracle's row order, elpd_logo_group,
    cooks_distance (G,), delta_global (G, Dg) and the scalars elpd_logo, elpd_logo_se."""
    if np.any((oracle.y != 0) & (oracle.y != 1)):
        raise ValueError("approximate LOGO needs a binary training y")
    K, G, Dg, N = oracle.K, oracle.G, oracle.lay.Dg, oracle.N
    if Hinv is None:
        Hinv = np.linalg.inv(oracle.kl_hessian_dense(free))
    delta = theta_shifts(oracle, free, Hinv)[:, :Dg]
    Pinv = np.linalg.inv(Hinv[4:4 + K, 4:4 + K])
    db = delta[:, 4:4 + K]
    cook = np.einsum("gi,ij,gj->g", db, Pinv, db) / K
    lpd, zm, zv = np.zeros(N), np.zeros(N), np.zeros(N)
    group = np.zeros(G)
    for g in range(G):
        rows = np.nonzero(oracle.g == g)[0]
        if rows.size == 0:
            continue
        glob = shifted_globals(oracle, free, delta[g])
        zm[rows], zv[rows] = held_out_moments(oracle, glob, rows)
        lpd[rows] = lo.log_predictive_density(zm[rows], zv[rows], oracle.y[rows], oracle.gh_x, oracle.gh_w)
        group[g] = np.sum(lpd[rows])
    nonempty = np.bincount(oracle.g, minlength=G) > 0
    Gp = int(np.sum(nonempty))
    se = float(np.sqrt(Gp) * np.std(group[nonempty], ddof=1)) if Gp > 1 else float("nan")
    return dict(lpd_logo=lpd, eta_mean_logo=zm, eta_var_logo=zv, elpd_logo_group=group, cooks_distance=cook,
                delta_global=delta, elpd_logo=float(np.sum(lpd)), elpd_logo_se=se)
