"""The approximate-maximum-influence oracle (oracle/amip_oracle.py) against independent computations: the third
derivative of the KL by torch.func on oracle/glmm_torch.py, central differences of exact refits in one row's weight,
and the greedy search on hand-made influences."""
import numpy as np
import pytest
import torch

from oracle import amip_oracle as am
from oracle import glmm_oracle as go
from oracle.glmm_torch import GLMMTorch

N, K, G, Q = 240, 3, 9, 6


def _oracle(w, bounds=0.0, seed=51, gh=Q):
    X, y, g = go.make_glmm_data(N, K, G, seed)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(gh)
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


def _autodiff_t(oracle, x, a):
    """D^3 KL[a, a, .] = grad_theta (a . H(theta) a) by torch.func on the autodiff restatement of the KL."""
    m = GLMMTorch(oracle)
    at = torch.as_tensor(a, dtype=torch.float64)

    def quad(f):
        return torch.dot(at, torch.func.jvp(torch.func.grad(m.kl), (f,), (at,))[1])

    return torch.func.grad(quad)(torch.as_tensor(x, dtype=torch.float64)).numpy()


@pytest.mark.parametrize("bounds", [0.0, 0.1])
def test_third_derivative_matches_autodiff(bounds):
    rng = np.random.default_rng(52)
    w = rng.uniform(0.5, 1.5, size=N)
    w[[3, 40]] = 0.0
    oracle = _oracle(w, bounds=bounds)
    x = go.make_free(oracle.lay.D, 52, scale=0.3)
    a = rng.standard_normal(oracle.lay.D)
    t, q = am.third_contraction(oracle, x, a)
    ref = _autodiff_t(oracle, x, a)
    np.testing.assert_allclose(t, ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    # q_n = a^T grad^2 l_n a: the weighted sum over the rows is the data part of a^T H a
    base = _oracle(np.zeros(N), bounds=bounds)
    H, H0 = oracle.kl_hessian_dense(x), base.kl_hessian_dense(x)
    np.testing.assert_allclose(-np.sum(w * q), a @ (H - H0) @ a, rtol=1e-10)


@pytest.fixture(scope="module")
def fitted():
    w = np.random.default_rng(53).uniform(0.5, 1.5, size=N)
    oracle = _oracle(w)
    xo = _newton(oracle, go.make_free(oracle.lay.D, 53))
    return oracle, w, xo


def test_variance_derivative_matches_central_differences_of_refits(fitted):
    oracle, w, xo = fitted
    c = np.array([0.5, -1.0, 2.0])
    r = am.influences(oracle, xo, c)
    chat = am.contrast(c, K, oracle.lay.D)
    h = 1e-4
    for n in (0, 77, 200):
        vals, phis = [], []
        for sgn in (1.0, -1.0):
            wn = w.copy()
            wn[n] += sgn * h
            o = _oracle(wn)
            x = _newton(o, xo)
            vals.append(chat @ np.linalg.solve(o.kl_hessian_dense(x), chat))
            phis.append(chat @ x)
        dvar = (vals[0] - vals[1]) / (2 * h)
        dphi = (phis[0] - phis[1]) / (2 * h)
        # var_shift = -w_n dsigma^2/dw_n, mean_shift = -w_n dphi/dw_n
        assert abs(-w[n] * dvar - r["var_shift"][n]) <= 1e-6 * abs(r["var_shift"][n]), (n, -w[n] * dvar,
                                                                                          r["var_shift"][n])
        assert abs(-w[n] * dphi - r["mean_shift"][n]) <= 1e-6 * abs(r["mean_shift"][n]), n


def test_contrast_forms(fitted):
    oracle, w, xo = fitted
    a = am.influences(oracle, xo, 1)
    b = am.influences(oracle, xo, np.array([0.0, 1.0, 0.0]))
    for f in ("estimate", "var", "mean_shift", "var_shift"):
        np.testing.assert_array_equal(a[f], b[f])
    assert a["estimate"] == xo[5]


def test_group_shifts_are_sums_of_row_shifts(fitted):
    oracle, w, xo = fitted
    rows = am.approximate_max_influence(oracle, xo, 0, unit="row")
    grp = am.approximate_max_influence(oracle, xo, 0, unit="group")
    np.testing.assert_allclose(grp["mean_shift"], np.bincount(oracle.g, rows["mean_shift"], minlength=G), rtol=1e-12)
    np.testing.assert_allclose(grp["sd_shift"], np.bincount(oracle.g, rows["sd_shift"], minlength=G), rtol=1e-12)
    for name in am.TARGETS:
        d = rows["targets"][name]
        if d["n_drop"] is not None:
            np.testing.assert_allclose(d["predicted_estimate"],
                                       rows["estimate"] + rows["mean_shift"][d["dropped"]].sum(), rtol=1e-12)


def test_greedy_search_on_hand_made_influences():
    push = np.array([-1.0, 0.5, -2.0, -1.0, -1.0, 3.0])
    elig = np.ones(6, dtype=bool)
    # ties keep the lower index first: -2 (2), then -1 at 0, 3, 4
    n, d = am.greedy_drop(2.5, push, elig, 1.0)
    assert n == 2 and list(d) == [2, 0]
    # exactly reaching zero does not cross it
    n, d = am.greedy_drop(4.0, push, elig, 1.0)
    assert n == 4 and list(d) == [2, 0, 3, 4]
    # the cap on the fraction: 3 of 6 units at most
    assert am.greedy_drop(4.0, push, elig, 0.5)[0] is None
    # unreachable: the harmful pushes sum to -5
    n, d = am.greedy_drop(5.0, push, elig, 1.0)
    assert n is None and d.size == 0
    # a negative statistic is pushed up: most positive first
    n, d = am.greedy_drop(-0.4, push, elig, 1.0)
    assert n == 1 and list(d) == [5]
    # an ineligible unit (zero weight) is never dropped and does not count in the cap
    elig[2] = False
    n, d = am.greedy_drop(2.5, push, elig, 1.0)
    assert list(d) == [0, 3, 4]
    assert am.greedy_drop(2.5, push, elig, 0.4)[0] is None      # floor(0.4 * 5) = 2 units


def test_targets_on_hand_made_influences(monkeypatch):
    oracle = _oracle(np.ones(N))
    fake = dict(estimate=1.0, var=0.25, sd=0.5, mean_shift=np.zeros(N), sd_shift=np.zeros(N))
    fake["mean_shift"][[5, 6, 7]] = [-0.3, -0.4, -0.5]
    fake["sd_shift"][[5, 6, 7]] = [0.2, 0.0, 0.0]
    monkeypatch.setattr(am, "influences", lambda *args, **kw: fake)
    r = am.approximate_max_influence(oracle, None, 0, level=0.95, max_fraction=1.0)
    z = r["z"]
    assert abs(z - 1.959963984540054) < 1e-12
    # sign: 1 - 0.5 - 0.4 - 0.3 = -0.2 < 0 with all three
    s = r["targets"]["sign"]
    assert s["n_drop"] == 3 and list(s["dropped"]) == [7, 6, 5]
    assert abs(s["predicted_estimate"] + 0.2) < 1e-12 and abs(s["predicted_sd"] - 0.7) < 1e-12
    assert s["fraction"] == 3 / N
    # significance: the lower bound 1 - z 0.5 = 0.02; unit 5 pushes it by -0.3 - z 0.2, the most of the three
    s = r["targets"]["significance"]
    assert s["n_drop"] == 1 and list(s["dropped"]) == [5]
    # opposite significance: the upper bound 1 + z 0.5 = 1.98 takes pushes -0.5, -0.4 and -0.3 + z 0.2: never below 0
    s = r["targets"]["significant_opposite"]
    assert s["n_drop"] is None and s["dropped"].size == 0 and s["predicted_estimate"] is None
    # a statistic below zero is pushed up: with the bound at -0.02 the same units cannot make it significant
    fake["estimate"] = 0.96
    r = am.approximate_max_influence(oracle, None, 0, level=0.95, max_fraction=1.0)
    assert r["targets"]["significance"]["n_drop"] is None
