"""The approximate-LOO oracle (oracle/loo_oracle.py) against independent computations: central differences
of exact refits in one observation weight, Q_n from the arrowhead pieces the device kernel uses, and the
properties the definitions imply."""
import numpy as np
import pytest

from oracle import glmm_oracle as go
from oracle import loo_oracle as lo
from oracle import predict_oracle as po

N, K, G, Q = 240, 3, 6, 6


def _oracle(w, bounds=0.0, seed=31):
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
    w = np.random.default_rng(4).uniform(0.5, 1.5, size=N)
    rows = [3, 77, 150, 239]
    w[rows] = 1.0                      # the rows whose weight is varied around 1
    oracle = _oracle(w)
    xo = _newton(oracle, go.make_free(oracle.lay.D, 31))
    return oracle, w, rows, xo


def test_ij_shift_matches_central_differences_of_refits(fitted):
    oracle, w, rows, xo = fitted
    Hinv = np.linalg.inv(oracle.kl_hessian_dense(xo))
    eps = 1e-4
    for n in rows:
        fits = []
        for sgn in (1.0, -1.0):
            wn = w.copy()
            wn[n] = 1.0 + sgn * eps
            fits.append(_newton(_oracle(wn), xo))
        dtheta_dw = (fits[0] - fits[1]) / (2 * eps)
        shift = lo.theta_shift(oracle, xo, n, Hinv)          # -w_n H^-1 grad l_n, w_n = 1
        err = np.max(np.abs(shift + dtheta_dw))
        assert err <= 1e-6 * np.max(np.abs(shift)), (n, err, np.max(np.abs(shift)))


@pytest.mark.parametrize("bounds", [0.0, 0.1])
def test_q_from_arrowhead_pieces_matches_dense(bounds):
    oracle = _oracle(np.random.default_rng(5).uniform(0.5, 1.5, size=N), bounds=bounds, seed=32)
    x = go.make_free(oracle.lay.D, 32)
    Hinv = np.linalg.inv(oracle.kl_hessian_dense(x))
    for a, b, nm in zip(lo.q_from_pieces(oracle, x), lo.q_dense(oracle, x, Hinv), ("mm", "mv", "vv")):
        np.testing.assert_allclose(a, b, rtol=1e-9, atol=1e-12 * np.max(np.abs(b)), err_msg="Q_" + nm)
    # Q_mm is the LR variance of eta that prediction computes for the same rows
    J = po.prediction_jacobian(x, oracle.X, oracle.g, K, G, oracle.gh_x, oracle.gh_w,
                               dict(mu_info=bounds, beta_info=bounds, u_info=bounds), quantity="eta")
    np.testing.assert_allclose(lo.q_dense(oracle, x, Hinv)[0], po.lr_variances(J, Hinv), rtol=1e-12)


def test_weight_zero_row_has_zero_shift(fitted):
    oracle, w, rows, xo = fitted
    w0 = w.copy()
    w0[[5, 100]] = 0.0
    o0 = _oracle(w0)
    x0 = _newton(o0, xo)
    r = lo.approximate_loo(o0, x0)
    for n in (5, 100):
        assert r["dz_m"][n] == 0.0 and r["dz_v"][n] == 0.0
        assert r["lpd_loo"][n] == r["lpd"][n] and r["eta_mean_loo"][n] == o0.obs_terms(
            o0.unpack(o0.free_to_vector(x0)), order=0)["z_m"][n]
        assert np.all(lo.theta_shift(o0, x0, n, np.linalg.inv(o0.kl_hessian_dense(x0))) == 0.0)
    assert r["n_invalid"] == 0 and np.isfinite(r["elpd_loo"])
    np.testing.assert_allclose(r["p_loo"], np.sum(r["lpd"]) - np.sum(r["lpd_loo"]), rtol=1e-12)


def test_lpd_of_y0_is_log_one_minus_p():
    gh_x, gh_w = np.polynomial.hermite.hermgauss(20)
    z_m, z_v = np.array([-2.0, 0.3, 1.5, 40.0]), np.array([0.5, 1.0, 0.2, 0.01])
    p = np.exp(lo.log_predictive_density(z_m, z_v, np.ones(4), gh_x, gh_w))
    lpd0 = lo.log_predictive_density(z_m, z_v, np.zeros(4), gh_x, gh_w)
    np.testing.assert_allclose(lpd0[:3], np.log1p(-p[:3]), rtol=1e-12)
    # p -> 1: 1 - p cancels to 0; the quadrature of sigma(-z) ~ e^-z keeps log E[e^-z] = -z_m + z_v / 2
    assert abs(lpd0[3] - (-40.0 + 0.005)) < 1e-9
    assert np.isnan(lo.log_predictive_density([0.0], [-1e-3], [1.0], gh_x, gh_w)[0])


def test_non_binary_y_is_refused(fitted):
    oracle, w, rows, xo = fitted
    bad = go.GLMMOracle(oracle.X, np.where(np.arange(N) == 7, 0.5, oracle.y), oracle.g, oracle.gh_x, oracle.gh_w,
                        weights=w, G=G)
    with pytest.raises(ValueError):
        lo.approximate_loo(bad, xo)
