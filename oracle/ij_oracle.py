"""Analytic fp64 oracle of the infinitesimal-jackknife (IJ) bootstrap covariance of the global parameters for small D
(numpy).  TEST INFRASTRUCTURE.

Resampling units u (rows, or whole groups) with multinomial weights changes the optimum, to first order, by
sum_u (w*_u - 1) H^-1 psi_u, psi_u = the unit's weighted score sum_{n in u} (W_m j_m + W_v j_v) (loo_oracle's row
Jacobians, W_m = w l_m, W_v = w l_v).  The multinomial weights have covariance I - 1 1^T / U, so the IJ covariance is

    Sigma_IJ = H^-1 (sum_u psi_u psi_u^T - s s^T / U) H^-1,     s = sum_u psi_u,

U = the units of non-zero weight (Giordano et al., "A Swiss Army Infinitesimal Jackknife").  Two routes:
  * dense: psi_u from the dense row Jacobians and the dense inverse of the oracle Hessian;
  * arrowhead, as csrc/ij.cu assembles it: the global block of H^-1 psi_u is S^-1 V_u with
    V_u = psi_u,glob - B_g^T L_g^-1 psi_u,loc; the groups' meat is V^T V and the rows' meat the per-group expansion
    sum_n h_n h_n^T - sum_g (B_g^T L_g^-1 E_g + E_g^T L_g^-1 B_g) + sum_g B_g^T L_g^-1 F_g L_g^-1 B_g
    with h_n = psi_n,glob, r_n = psi_n,loc, E_g = sum_{n in g} r_n h_n^T, F_g = sum_{n in g} r_n r_n^T.
"""
import numpy as np

from . import loo_oracle as lo


def row_scores(oracle, free):
    """psi (N, D): every training row's weighted score W_m j_m + W_v j_v, dense (the oracle's row order)."""
    J_m, J_v = lo.moment_jacobians(free, oracle.X, oracle.g, oracle.K, oracle.G, lo._lb(oracle))
    _, _, W_m, W_v = lo.row_terms(oracle, free)
    return W_m[:, None] * J_m + W_v[:, None] * J_v


def unit_scores(oracle, free, unit):
    """psi_u (U', D) for unit "row" (all N rows) or "group" (all G groups)."""
    psi = row_scores(oracle, free)
    if unit == "row":
        return psi
    if unit != "group":
        raise ValueError("unit must be 'row' or 'group', got %r" % (unit,))
    out = np.zeros((oracle.G, psi.shape[1]))
    np.add.at(out, oracle.g, psi)
    return out


def n_units(oracle, unit):
    """Units of non-zero weight: rows with w != 0, or groups with such a row."""
    w = np.ones(oracle.N) if oracle.w is None else oracle.w
    if unit == "row":
        return int(np.sum(w != 0))
    return int(np.sum(np.bincount(oracle.g[w != 0], minlength=oracle.G) > 0))


def ij_covariance_dense(oracle, free, unit, centered=True, Hinv=None):
    """Sigma_IJ (D, D) from the dense H^-1; its [:Dg, :Dg] block is the globals' IJ covariance."""
    if Hinv is None:
        Hinv = np.linalg.inv(oracle.kl_hessian_dense(free))
    infl = unit_scores(oracle, free, unit) @ Hinv          # row u = (H^-1 psi_u)^T
    M = infl.T @ infl
    if centered:
        s = infl.sum(axis=0)
        M = M - np.outer(s, s) / n_units(oracle, unit)
    return 0.5 * (M + M.T)


def _pieces(oracle, free):
    lay, G, Dg = oracle.lay, oracle.G, oracle.lay.Dg
    _, _, blk = oracle.kl_blocks(free)
    L = blk["L"]
    det = L[:, 0] * L[:, 2] - L[:, 1] ** 2
    Linv = np.stack([np.stack([L[:, 2], -L[:, 1]], -1), np.stack([-L[:, 1], L[:, 0]], -1)], 1) / det[:, None, None]
    psi = row_scores(oracle, free)
    g = oracle.g
    h = psi[:, :Dg]
    r = np.stack([psi[np.arange(oracle.N), lay.u_mean + g], psi[np.arange(oracle.N), lay.u_info + g]], axis=1)
    return blk["B"], Linv, h, r


def meat_arrowhead(oracle, free, unit):
    """(meat (Dg, Dg), s (Dg)) = (sum_u V_u V_u^T, sum_u V_u) as csrc/ij.cu assembles them."""
    G, Dg, g = oracle.G, oracle.lay.Dg, oracle.g
    B, Linv, h, r = _pieces(oracle, free)
    Vn = h - np.einsum("nri,nr->ni", B[g], np.einsum("nrs,ns->nr", Linv[g], r))    # V_n = h_n - B_g^T L_g^-1 r_n
    Vg = np.zeros((G, Dg))
    np.add.at(Vg, g, Vn)
    s = Vg.sum(axis=0)
    if unit == "group":
        return Vg.T @ Vg, s
    if unit != "row":
        raise ValueError("unit must be 'row' or 'group', got %r" % (unit,))
    E = np.zeros((G, 2, Dg))
    np.add.at(E, g, r[:, :, None] * h[:, None, :])
    F = np.zeros((G, 2, 2))
    np.add.at(F, g, r[:, :, None] * r[:, None, :])
    LB = Linv @ B                                         # (G, 2, Dg): L^-1 B
    LE = Linv @ E
    cross = np.einsum("gri,grj->ij", B, LE)               # sum_g B_g^T L_g^-1 E_g
    quad = np.einsum("gri,grs,gsj->ij", LB, F, LB)        # sum_g B_g^T L_g^-1 F_g L_g^-1 B_g
    return h.T @ h - cross - cross.T + quad, s


def ij_covariance_arrowhead(oracle, free, unit, centered=True):
    """The globals' IJ covariance (Dg, Dg) = S^-1 (meat - s s^T / U) S^-1 from meat_arrowhead."""
    Sinv, _ = oracle.schur_global_cov(free)
    M, s = meat_arrowhead(oracle, free, unit)
    if centered:
        M = M - np.outer(s, s) / n_units(oracle, unit)
    C = Sinv @ M @ Sinv
    return 0.5 * (C + C.T)
