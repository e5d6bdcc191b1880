"""The infinitesimal-jackknife covariance oracle (oracle/ij_oracle.py) against independent computations: the arrowhead
assembly the device kernels use against the dense H^-1, the IJ shifts of the LOO and LOGO oracles (which their tests
pin against refits), and the spread of exact refits under multinomial bootstrap weights."""
import numpy as np
import pytest

from oracle import glmm_oracle as go
from oracle import ij_oracle as ij
from oracle import logo_oracle as lg
from oracle import loo_oracle as lo

N, K, G, Q = 400, 2, 12, 6


def _oracle(w, bounds=0.0, seed=51):
    X, y, g = go.make_glmm_data(N, K, G, seed)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(Q)
    return go.GLMMOracle(X, y, g, gh_x, gh_w, weights=w, G=G,
                         bounds=go.GLMMBounds(bounds, bounds, bounds, bounds, bounds))


def _newton(oracle, x0, gtol=1e-7, maxiter=100):
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
    oracle = _oracle(np.ones(N))
    return oracle, _newton(oracle, go.make_free(oracle.lay.D, 51))


@pytest.mark.parametrize("bounds", [0.0, 0.05])
@pytest.mark.parametrize("unit", ["row", "group"])
@pytest.mark.parametrize("centered", [True, False])
def test_arrowhead_matches_dense(bounds, unit, centered):
    w = np.random.default_rng(7).uniform(0.5, 1.5, size=N)
    w[[3, 40, 41]] = 0.0
    oracle = _oracle(w, bounds=bounds, seed=52)
    x = go.make_free(oracle.lay.D, 52)
    Dg = oracle.lay.Dg
    dense = ij.ij_covariance_dense(oracle, x, unit, centered)[:Dg, :Dg]
    arrow = ij.ij_covariance_arrowhead(oracle, x, unit, centered)
    assert np.max(np.abs(arrow - dense)) <= 1e-10 * np.max(np.abs(dense))
    assert np.array_equal(arrow, arrow.T)


def test_meat_is_the_outer_products_of_the_loo_and_logo_shifts(fitted):
    oracle, xo = fitted
    Hinv = np.linalg.inv(oracle.kl_hessian_dense(xo))
    rows = np.array([lo.theta_shift(oracle, xo, n, Hinv) for n in range(N)])
    groups = lg.theta_shifts(oracle, xo, Hinv)
    for unit, shifts in (("row", rows), ("group", groups)):
        ref = shifts.T @ shifts
        got = ij.ij_covariance_dense(oracle, xo, unit, centered=False, Hinv=Hinv)
        assert np.max(np.abs(got - ref)) <= 1e-12 * np.max(np.abs(ref)), unit


def test_zero_weight_units_do_not_count():
    w = np.ones(N)
    oracle = _oracle(w)
    w[oracle.g == 4] = 0.0
    w[[0, 1]] = 0.0
    oracle = _oracle(w)
    assert ij.n_units(oracle, "row") == N - int(np.sum(oracle.g == 4)) - int(np.sum(oracle.g[[0, 1]] != 4))
    assert ij.n_units(oracle, "group") == G - 1
    psi = ij.unit_scores(oracle, go.make_free(oracle.lay.D, 3), "group")
    assert np.all(psi[4] == 0.0)


@pytest.mark.timeout(600)
@pytest.mark.parametrize("unit", ["row", "group"])
def test_matches_the_bootstrap_of_exact_refits(fitted, unit):
    """The IJ variances of E[beta] against the sample variances of 200 Newton refits under multinomial bootstrap
    weights on the rows or on whole groups (seeded).  Measured ratios bootstrap / IJ: rows 1.12, 1.09; groups 0.98,
    0.89 (the sampling error of a variance from 200 draws is about 10 %)."""
    oracle, xo = fitted
    rng = np.random.default_rng(5 if unit == "row" else 6)
    fits = []
    for _ in range(200):
        if unit == "row":
            w = rng.multinomial(N, np.full(N, 1.0 / N)).astype(np.float64)
        else:
            w = rng.multinomial(G, np.full(G, 1.0 / G)).astype(np.float64)[oracle.g]
        fits.append(_newton(_oracle(w), xo)[4:4 + K])
    boot = np.var(np.array(fits), axis=0, ddof=1)
    ijv = np.diag(ij.ij_covariance_dense(oracle, xo, unit))[4:4 + K]
    ratio = boot / ijv
    assert np.all((ratio > 0.75) & (ratio < 1.35)), ratio
