"""Analytic fp64 oracle of the approximate maximum influence perturbation (AMIP) of a linear contrast of E[beta], for
rows and for groups, with the dense H^-1 (numpy / scipy).  TEST INFRASTRUCTURE.

phi = c^T E[beta] = chat^T theta (chat = c padded to D), sigma^2 = chat^T H^-1 chat, a = H^-1 chat.  With
KL(theta; w) = -sum_n w_n l_n(theta) + ... and C = d^2 KL / d theta d w (column n = -grad l_n):

    d phi / d w_n     = -(C^T a)_n
    d sigma^2 / d w_n = q_n + (C^T b)_n,   q_n = a^T (grad^2 l_n) a,  b = H^-1 t,  t = D^3 KL[a, a, .]

Dropping unit u is w_n -> 0 on its rows: mean_shift_u = sum_{n in u} w_n (C^T a)_n and
var_shift_u = -sum_{n in u} w_n (q_n + (C^T b)_n), sd_shift_u = var_shift_u / (2 sd).

t is assembled analytically (DESIGN.md 3e): the data part from the moments of every row along a,
    alpha = j_m . a,  beta1 = j_v . a,  beta2 = a^T (grad^2 z_v) a,
and the derivatives of the Gauss-Hermite term A(z_m, z_v) to third order; the non-data part from the random-effect
term, the entropies and the priors in free coordinates.  r(f) = 1 / (e^f + lb) is the variance of a precision in
free coordinates; its derivatives r', r'', r''' carry every nonlinearity of the exp + lb transform that z_v sees.
"""
import numpy as np
import scipy.special
import scipy.stats

from . import loo_oracle as lo

TARGETS = ("sign", "significance", "significant_opposite")


def r_derivs(info, lb):
    """(r', r'', r''') of r = 1 / info as a function of f = log(info - lb)."""
    e = info - lb
    return -e / info ** 2, e * (e - lb) / info ** 3, e * (-e * e + 4 * e * lb - lb * lb) / info ** 4


def chain3(h1, h2, h3, e):
    """Third derivative in f of h(e^f + lb) from h', h'', h''' at e^f + lb (e = e^f)."""
    return h3 * e ** 3 + 3 * h2 * e ** 2 + h1 * e


def gh_derivs(z_m, z_v, gh_x, gh_w):
    """The derivatives of A(z_m, z_v) = E[log(1 + e^z)], z ~ N(z_m, z_v), by the Gauss-Hermite rule, differentiated
    exactly node by node: dict A_v, A_mm, A_mv, A_vv, A_mmm, A_mmv, A_mvv, A_vvv (N,) each."""
    what = np.asarray(gh_w, dtype=np.float64) / np.sqrt(np.pi)
    c = np.sqrt(2.0) * np.asarray(gh_x, dtype=np.float64)
    s = np.sqrt(z_v)
    t = z_m[:, None] + s[:, None] * c[None, :]
    sg = scipy.special.expit(t)
    sb = scipy.special.expit(-t)
    d1 = sg * sb
    d2 = d1 * (sb - sg)

    def S(f, p):
        return np.sum(what * f * c ** p, axis=1)

    S0, S1 = S(sg, 0), S(sg, 1)
    P0, P1, P2 = S(d1, 0), S(d1, 1), S(d1, 2)
    R0, R1, R2, R3 = S(d2, 0), S(d2, 1), S(d2, 2), S(d2, 3)
    return dict(A_v=S1 / (2 * s), A_mm=P0, A_mv=P1 / (2 * s), A_vv=P2 / (4 * z_v) - S1 / (4 * s ** 3),
                A_mmm=R0, A_mmv=R1 / (2 * s), A_mvv=R2 / (4 * z_v) - P1 / (4 * s ** 3),
                A_vvv=R3 / (8 * s ** 3) - 3 * P2 / (8 * z_v ** 2) + 3 * S1 / (8 * s ** 5))


def row_moments(oracle, free, a):
    """alpha, beta1, beta2 (N,) of every row along a (D,), the oracle's row order."""
    K, G, Dg = oracle.K, oracle.G, oracle.lay.Dg
    b = oracle.bounds
    p = oracle.unpack(oracle.free_to_vector(free))
    X, g = oracle.X, oracle.g
    s1, s2, _ = r_derivs(p["beta_i"], b.beta_info)
    d1, d2, _ = r_derivs(p["u_i"], b.u_info)
    a_bm, a_bi, a_um, a_ui = a[4:4 + K], a[4 + K:Dg], a[Dg:Dg + G], a[Dg + G:]
    alpha = X @ a_bm + a_um[g]
    beta1 = (X * X) @ (s1 * a_bi) + d1[g] * a_ui[g]
    beta2 = (X * X) @ (s2 * a_bi ** 2) + d2[g] * a_ui[g] ** 2
    return alpha, beta1, beta2


def third_contraction(oracle, free, a):
    """(t (D,), q (N,)): t = D^3 KL[a, a, .] in free coordinates and q_n = a^T (grad^2 l_n) a (unweighted), rows in
    the oracle's order."""
    free = np.asarray(free, dtype=np.float64)
    a = np.asarray(a, dtype=np.float64)
    lay, pr, bd = oracle.lay, oracle.prior, oracle.bounds
    K, G, Dg, D = lay.K, lay.G, lay.Dg, lay.D
    vec = oracle.free_to_vector(free)
    p = oracle.unpack(vec)
    X, g = oracle.X, oracle.g
    w = np.ones(oracle.N) if oracle.w is None else oracle.w
    z_m = p["u_m"][g] + X @ p["beta_m"]
    z_v = (1.0 / p["u_i"])[g] + (X * X) @ (1.0 / p["beta_i"])
    A = gh_derivs(z_m, z_v, oracle.gh_x, oracle.gh_w)
    l_v, l_mm, l_mv, l_vv = -A["A_v"], -A["A_mm"], -A["A_mv"], -A["A_vv"]
    l_mmm, l_mmv, l_mvv, l_vvv = -A["A_mmm"], -A["A_mmv"], -A["A_mvv"], -A["A_vvv"]
    al, b1, b2 = row_moments(oracle, free, a)
    q = l_mm * al * al + 2 * l_mv * al * b1 + l_vv * b1 * b1 + l_v * b2
    c_m = l_mmm * al * al + 2 * l_mmv * al * b1 + l_mvv * b1 * b1 + l_mv * b2
    c_v = l_mmv * al * al + 2 * l_mvv * al * b1 + l_vvv * b1 * b1 + l_vv * b2
    c_h = 2 * (l_mv * al + l_vv * b1)
    s1, s2, s3 = r_derivs(p["beta_i"], bd.beta_info)
    d1, d2, d3 = r_derivs(p["u_i"], bd.u_info)
    a_bi, a_um, a_ui = a[4 + K:Dg], a[Dg:Dg + G], a[Dg + G:]
    t = np.zeros(D)
    # data: -sum_n w_n D^3 l_n[a, a, .]
    t[4:4 + K] = -X.T @ (w * c_m)
    S2 = X * X
    t[4 + K:Dg] = -(s1 * (S2.T @ (w * c_v)) + s2 * a_bi * (S2.T @ (w * c_h)) + s3 * a_bi ** 2 * (S2.T @ (w * l_v)))
    t[Dg:Dg + G] = -np.bincount(g, weights=w * c_m, minlength=G)
    t[Dg + G:] = -np.bincount(g, weights=w * (c_v * d1[g] + c_h * d2[g] * a_ui[g] + l_v * d3[g] * a_ui[g] ** 2),
                              minlength=G)
    # non-data: KL_nd = E S~ + sum of one-variable terms, S~ = S / 2 + rate0,
    # S = sum_g (mu_m - u_m,g)^2 + G r(mu_i) + sum_g r(u_i,g), E = shape / rate
    mu_m, mu_i, sh, ra = p["mu_m"], p["mu_i"], p["a"], p["b"]
    am, ai, aa, ab = a[0], a[1], a[2], a[3]
    dm, da = mu_m - p["u_m"], am - a_um
    m1, m2, m3 = r_derivs(mu_i, bd.mu_info)
    S = np.sum(dm ** 2) + G / mu_i + np.sum(1 / p["u_i"])
    S_a = np.sum(2 * dm * da) + G * m1 * ai + np.sum(d1 * a_ui)
    S_aa = np.sum(2 * da ** 2) + G * m2 * ai ** 2 + np.sum(d2 * a_ui ** 2)
    ea, eb = sh - bd.tau_shape, ra - bd.tau_rate
    E = sh / ra
    Ea, Eaa, Eaaa = ea / ra, ea / ra, ea / ra
    Eb = -sh * eb / ra ** 2
    Eab = Eaab = -ea * eb / ra ** 2
    Ebb = -sh * eb * (ra - 2 * eb) / ra ** 3
    Eabb = -ea * eb * (ra - 2 * eb) / ra ** 3
    Ebbb = -sh * eb * (ra * ra - 6 * eb * ra + 6 * eb * eb) / ra ** 4
    E1 = Ea * aa + Eb * ab                                     # E'[a]
    E2 = Eaa * aa * aa + 2 * Eab * aa * ab + Ebb * ab * ab     # E''[a, a]
    St, St_a, St_aa = 0.5 * S + pr.tau_rate, 0.5 * S_a, 0.5 * S_aa
    t[2] += (Eaaa * aa * aa + 2 * Eaab * aa * ab + Eabb * ab * ab) * St + 2 * (Eaa * aa + Eab * ab) * St_a + Ea * St_aa
    t[3] += (Eaab * aa * aa + 2 * Eabb * aa * ab + Ebbb * ab * ab) * St + 2 * (Eab * aa + Ebb * ab) * St_a + Eb * St_aa
    # S-variables: E''[a,a] S~'_j + 2 E'[a] (S~'' a)_j + E S~'''[a,a]_j
    t[0] += E2 * np.sum(dm) + 2 * E1 * np.sum(da)
    t[1] += 0.5 * G * (E2 * m1 + 2 * E1 * m2 * ai + E * m3 * ai * ai)
    t[Dg:Dg + G] += -E2 * dm - 2 * E1 * da
    t[Dg + G:] += 0.5 * (E2 * d1 + 2 * E1 * d2 * a_ui + E * d3 * a_ui ** 2)
    # one-variable terms: u entropy (always), then the entropies and priors of mu, beta and tau
    eu = p["u_i"] - bd.u_info
    t[Dg + G:] += chain3(0.5 / p["u_i"], -0.5 / p["u_i"] ** 2, 1.0 / p["u_i"] ** 3, eu) * a_ui ** 2
    cg = 0.5 * G + pr.tau_shape - 1.0                # - cg E[log tau] from the random effect and the tau prior
    psi1, psi2, psi3 = (scipy.special.polygamma(n, sh) for n in (1, 2, 3))
    gA = (-1 + (sh - 1 - cg) * psi1, psi1 + (sh - 1 - cg) * psi2, 2 * psi2 + (sh - 1 - cg) * psi3)
    kb = 0.5 * G + pr.tau_shape                      # coefficient of log rate
    t[2] += chain3(*gA, ea) * aa * aa
    t[3] += chain3(kb / ra, -kb / ra ** 2, 2 * kb / ra ** 3, eb) * ab * ab
    emi = mu_i - bd.mu_info
    t[1] += chain3(0.5 / mu_i - 0.5 * pr.mu_info / mu_i ** 2, -0.5 / mu_i ** 2 + pr.mu_info / mu_i ** 3,
                   1.0 / mu_i ** 3 - 3 * pr.mu_info / mu_i ** 4, emi) * ai * ai
    bi = p["beta_i"]
    t[4 + K:Dg] += chain3(0.5 / bi - 0.5 * pr.beta_info / bi ** 2, -0.5 / bi ** 2 + pr.beta_info / bi ** 3,
                          1.0 / bi ** 3 - 3 * pr.beta_info / bi ** 4, bi - bd.beta_info) * a_bi ** 2
    return t, q


def contrast(c, K, D):
    """chat (D,): c (length K, or an integer k for e_k) placed on the beta.mean block."""
    chat = np.zeros(D)
    if np.ndim(c) == 0:
        chat[4 + int(c)] = 1.0
    else:
        chat[4:4 + K] = np.asarray(c, dtype=np.float64)
    return chat


def influences(oracle, free, c, Hinv=None):
    """dict: estimate, var, sd, a, t, b, q and the per-row shifts mean_shift, var_shift, sd_shift (oracle order)."""
    free = np.asarray(free, dtype=np.float64)
    D, K = oracle.lay.D, oracle.K
    if Hinv is None:
        Hinv = np.linalg.inv(oracle.kl_hessian_dense(free))
    chat = contrast(c, K, D)
    a = Hinv @ chat
    var = float(chat @ a)
    sd = np.sqrt(var)
    t, q = third_contraction(oracle, free, a)
    b = Hinv @ t
    J_m, J_v = lo.moment_jacobians(free, oracle.X, oracle.g, K, oracle.G, lo._lb(oracle))
    _, _, W_m, W_v = lo.row_terms(oracle, free)
    w = np.ones(oracle.N) if oracle.w is None else oracle.w
    mean_shift = -(W_m * (J_m @ a) + W_v * (J_v @ a))
    var_shift = -w * q + (W_m * (J_m @ b) + W_v * (J_v @ b))
    return dict(estimate=float(chat @ free), var=var, sd=sd, a=a, t=t, b=b, q=q, mean_shift=mean_shift,
                var_shift=var_shift, sd_shift=var_shift / (2 * sd))


def greedy_drop(stat, push, eligible, max_fraction):
    """The shortest prefix of the eligible units, most harmful first, whose summed push takes `stat` across zero:
    (n_drop, dropped indices) or (None, empty).  Harm is the push toward zero (-push for stat >= 0, push for stat < 0);
    ties keep the lower index first; at most floor(max_fraction * #eligible) units."""
    side = 1.0 if stat >= 0 else -1.0
    idx = np.nonzero(eligible)[0]
    order = idx[np.argsort(side * push[idx], kind="stable")]
    nmax = int(np.floor(max_fraction * idx.size + 1e-9))
    cum = np.cumsum(side * push[order][:nmax])
    hit = np.nonzero(side * stat + cum < 0)[0]
    if hit.size == 0:
        return None, order[:0]
    n = int(hit[0]) + 1
    return n, order[:n]


def approximate_max_influence(oracle, free, c, unit="row", level=0.95, max_fraction=0.1, Hinv=None):
    """dict: estimate, sd_lr, z, mean_shift, sd_shift (per row in the oracle's order, or per group) and targets
    {name: dict(n_drop, fraction, dropped, predicted_estimate, predicted_sd)}."""
    r = influences(oracle, free, c, Hinv)
    w = np.ones(oracle.N) if oracle.w is None else oracle.w
    if unit == "row":
        ms, ss, elig = r["mean_shift"], r["sd_shift"], w != 0
    else:
        G = oracle.G
        ms = np.bincount(oracle.g, weights=r["mean_shift"], minlength=G)
        ss = np.bincount(oracle.g, weights=r["sd_shift"], minlength=G)
        elig = np.bincount(oracle.g, weights=(w != 0).astype(np.float64), minlength=G) > 0
    phi, sd = r["estimate"], r["sd"]
    z = float(scipy.stats.norm.ppf(0.5 + 0.5 * level))
    s = 1.0 if phi >= 0 else -1.0
    lin = dict(sign=(s * phi, s * ms), significance=(s * phi - z * sd, s * ms - z * ss),
               significant_opposite=(s * phi + z * sd, s * ms + z * ss))
    n_elig = int(np.sum(elig))
    targets = {}
    for name in TARGETS:
        stat, push = lin[name]
        n, dropped = greedy_drop(stat, push, elig, max_fraction)
        targets[name] = dict(n_drop=n, fraction=None if n is None else n / n_elig, dropped=dropped,
                             predicted_estimate=None if n is None else phi + float(np.sum(ms[dropped])),
                             predicted_sd=None if n is None else sd + float(np.sum(ss[dropped])))
    return dict(estimate=phi, sd_lr=sd, z=z, mean_shift=ms, sd_shift=ss, targets=targets)
