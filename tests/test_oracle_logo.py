"""The approximate leave-one-group-out oracle (oracle/logo_oracle.py) against independent computations: central
differences of exact refits in one group's weights, the arrowhead assembly the device kernel uses against the dense
H^-1, the closed form of q(u_g) without the group's rows, and exact refits without the group."""
import numpy as np
import pytest

from oracle import glmm_oracle as go
from oracle import logo_oracle as lg

N, K, G, Q = 360, 3, 12, 6


def _oracle(w, bounds=0.0, seed=41):
    X, y, g = go.make_glmm_data(N, K, G, seed)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(Q)
    return go.GLMMOracle(X, y, g, gh_x, gh_w, weights=w, G=G, bounds=go.GLMMBounds(bounds, bounds, bounds, bounds,
                                                                                   bounds))


def _newton(oracle, x0, gtol=1e-12, maxiter=100):
    """Damped Newton on the oracle KL to |grad| <= gtol (dense: the model is small)."""
    x = np.array(x0, dtype=np.float64)
    for _ in range(maxiter):
        gr = oracle.kl_grad(x)
        if np.max(np.abs(gr)) <= gtol:
            return x
        H = oracle.kl_hessian_dense(x)
        lam = 0.0
        while True:
            try:
                np.linalg.cholesky(H + lam * np.eye(H.shape[0]))
                break
            except np.linalg.LinAlgError:
                lam = max(1e-6, 10 * lam)
        step = np.linalg.solve(H + lam * np.eye(H.shape[0]), gr)
        f0, t = oracle.kl(x), 1.0
        while oracle.kl(x - t * step) > f0 and t > 1e-10:
            t *= 0.5
        x = x - t * step
    raise AssertionError("Newton did not converge: |grad| = %g" % np.max(np.abs(oracle.kl_grad(x))))


@pytest.fixture(scope="module")
def fitted():
    w = np.random.default_rng(6).uniform(0.5, 1.5, size=N)
    oracle = _oracle(w)
    xo = _newton(oracle, go.make_free(oracle.lay.D, 41))
    return oracle, w, xo


def test_ij_shift_matches_central_differences_of_refits(fitted):
    oracle, w, xo = fitted
    dtheta = lg.theta_shifts(oracle, xo, np.linalg.inv(oracle.kl_hessian_dense(xo)))
    h = 1e-4
    for g in (0, 5, 11):
        rows = oracle.g == g
        fits = []
        for sgn in (1.0, -1.0):
            wg = w.copy()
            wg[rows] *= 1.0 + sgn * h
            fits.append(_newton(_oracle(wg), xo))
        # d theta / d eps for w_n -> (1 + eps) w_n on the group is H^-1 v_g; dropping the group is eps = -1
        fd = (fits[0] - fits[1]) / (2 * h)
        err = np.max(np.abs(dtheta[g] + fd))
        assert err <= 1e-6 * np.max(np.abs(dtheta[g])), (g, err, np.max(np.abs(dtheta[g])))


@pytest.mark.parametrize("bounds", [0.0, 0.1])
def test_arrowhead_delta_matches_dense(bounds):
    oracle = _oracle(np.random.default_rng(7).uniform(0.5, 1.5, size=N), bounds=bounds, seed=42)
    x = go.make_free(oracle.lay.D, 42)
    dense = lg.theta_shifts(oracle, x, np.linalg.inv(oracle.kl_hessian_dense(x)))[:, :oracle.lay.Dg]
    arrow = lg.delta_arrowhead(oracle, x)
    assert np.max(np.abs(arrow - dense)) <= 1e-10 * np.max(np.abs(dense))


@pytest.mark.parametrize("bounds", [0.0, 0.05])
def test_refit_without_group_has_closed_form_local_factor(bounds):
    w = np.ones(N)
    g0 = 4
    w[np.arange(N)[_oracle(w).g == g0]] = 0.0
    oracle = _oracle(w, bounds=bounds)
    xo = _newton(oracle, go.make_free(oracle.lay.D, 43))
    vec = oracle.free_to_vector(xo)
    p = oracle.unpack(vec)
    lay = oracle.lay
    assert abs(p["u_m"][g0] - p["mu_m"]) <= 1e-8 * max(1.0, abs(p["mu_m"]))
    info = max(p["a"] / p["b"], bounds)
    assert abs(p["u_i"][g0] - info) <= 1e-8 * info
    # the dropped group's gradient is zero: its IJ shift is exactly zero
    v = lg.group_gradients(oracle, xo)
    assert np.all(v[g0] == 0.0)
    assert lay.D == v.shape[1]


def test_close_to_exact_refits(fitted):
    """IJ error well under the effect of dropping the group: on the 4 groups of largest Cook's distance,
    |elpd_logo_g - exact_g| <= 0.35 |elpd_new_g - exact_g| + 1e-8, where elpd_new_g is the same held-out predictive
    at the unshifted optimum and exact_g that of an exact refit without the group.  Measured ratios here: 0.09, 0.31,
    0.16, 0.18 (0.28 at worst with N = 900, G = 30): dropping a whole group of 30 rows is not a small change, and the
    first-order step leaves about a third of the effect on the most influential group."""
    oracle, w, xo = fitted
    r = lg.approximate_logo(oracle, xo)
    zero = np.zeros(oracle.lay.Dg)
    for g in np.argsort(-r["cooks_distance"], kind="stable")[:4]:
        rows = np.nonzero(oracle.g == g)[0]
        w0 = w.copy()
        w0[rows] = 0.0
        o0 = _oracle(w0)
        x0 = _newton(o0, xo)
        exact = np.sum(lg.held_out_lpd(o0, lg.shifted_globals(o0, x0, zero), rows))
        new = np.sum(lg.held_out_lpd(oracle, lg.shifted_globals(oracle, xo, zero), rows))
        err, effect = abs(r["elpd_logo_group"][g] - exact), abs(new - exact)
        assert err <= 0.35 * effect + 1e-8, (int(g), r["elpd_logo_group"][g], new, exact)


def test_aggregates_and_empty_groups():
    X, y, g = go.make_glmm_data(N, K, G - 2, 44)
    g = np.where(g >= 3, g + 2, g)                      # ids 3 and 4 have no rows
    gh_x, gh_w = np.polynomial.hermite.hermgauss(Q)
    oracle = go.GLMMOracle(X, y, g, gh_x, gh_w, G=G)
    x = go.make_free(oracle.lay.D, 44)
    r = lg.approximate_logo(oracle, x)
    for e in (3, 4):
        assert np.all(r["delta_global"][e] == 0.0) and r["cooks_distance"][e] == 0.0 and r["elpd_logo_group"][e] == 0
    assert np.all(np.isfinite(r["lpd_logo"])) and np.all(r["lpd_logo"] < 0) and np.all(r["eta_var_logo"] > 0)
    ne = np.array([i not in (3, 4) for i in range(G)])
    np.testing.assert_allclose(r["elpd_logo_se"], np.sqrt(G - 2) * np.std(r["elpd_logo_group"][ne], ddof=1),
                               rtol=1e-14)
    np.testing.assert_allclose(r["elpd_logo"], np.sum(r["elpd_logo_group"]), rtol=1e-12)
    assert np.all(r["cooks_distance"] >= 0)


def test_non_binary_y_is_refused(fitted):
    oracle, w, xo = fitted
    bad = go.GLMMOracle(oracle.X, np.where(np.arange(N) == 7, 0.5, oracle.y), oracle.g, oracle.gh_x, oracle.gh_w,
                        weights=w, G=G)
    with pytest.raises(ValueError):
        lg.approximate_logo(bad, xo)
