"""The prediction oracle (oracle/predict_oracle.py) against independent computations: numerical
integration of the predictive moments and torch autodiff of the prediction."""
import numpy as np
import pytest
import scipy.integrate
import scipy.special
import scipy.stats
import torch

from oracle import predict_oracle as po

K, G = 4, 3


def _case(seed, lb):
    rng = np.random.default_rng(seed)
    D = 4 + 2 * K + 2 * G
    free = 0.3 * rng.standard_normal(D)
    X = rng.standard_normal((7, K))
    g = np.array([0, 2, -1, 1, -1, 2, 0])
    bounds = dict(mu_info=lb, beta_info=lb, u_info=lb)
    return free, X, g, bounds


@pytest.mark.parametrize("lb", [0.0, 0.1])
def test_predictive_moments_match_numerical_integration(lb):
    free, X, g, bounds = _case(1, lb)
    X = 0.5 * X     # predictive sd <= 2: there 200 Gauss-Hermite nodes are exact to ~1e-16 (at sd ~4, 1e-11)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(200)
    r = po.predict(free, X, g, K, G, gh_x, gh_w, bounds)
    for i in range(X.shape[0]):
        m, sd = r["eta_mean"][i], np.sqrt(r["eta_var_mfvb"][i])
        dens = scipy.stats.norm(m, sd).pdf
        lo, hi = m - 40 * sd, m + 40 * sd
        p = scipy.integrate.quad(lambda e: scipy.special.expit(e) * dens(e), lo, hi, epsabs=1e-14, epsrel=1e-13,
                                 limit=200)[0]
        p2 = scipy.integrate.quad(lambda e: scipy.special.expit(e) ** 2 * dens(e), lo, hi, epsabs=1e-14,
                                  epsrel=1e-13, limit=200)[0]
        assert abs(r["prob"][i] - p) < 1e-12, (i, r["prob"][i], p)
        assert abs(r["prob_var_mfvb"][i] + r["prob"][i] ** 2 - p2) < 1e-12, i
        assert abs(r["prob_var_mfvb"][i] - (p2 - p * p)) < 1e-12, i


def _torch_prediction(free, X, g, gh_x, gh_w, bounds, quantity):
    """Forward of the prediction in torch, written from the definitions (not from the oracle)."""
    Dg = 4 + 2 * K
    Xt, gt = torch.from_numpy(X), torch.from_numpy(g)
    c = torch.from_numpy(np.sqrt(2.0) * gh_x)
    what = torch.from_numpy(gh_w / np.sqrt(np.pi))

    def f(fr):
        beta_m, beta_i = fr[4:4 + K], torch.exp(fr[4 + K:Dg]) + bounds["beta_info"]
        u_m, u_i = fr[Dg:Dg + G], torch.exp(fr[Dg + G:]) + bounds["u_info"]
        mu_m, mu_i = fr[0], torch.exp(fr[1]) + bounds["mu_info"]
        pop = gt < 0
        gs = torch.where(pop, torch.zeros_like(gt), gt)
        e = torch.where(pop, mu_m, u_m[gs])
        v = torch.where(pop, 1.0 / mu_i, 1.0 / u_i[gs])
        z_m = e + Xt @ beta_m
        if quantity == "eta":
            return z_m
        z_v = v + (Xt * Xt) @ (1.0 / beta_i)
        t = z_m[:, None] + torch.sqrt(z_v)[:, None] * c[None, :]
        return torch.sum(what * torch.sigmoid(t), dim=1)

    return torch.autograd.functional.jacobian(f, torch.from_numpy(free)).numpy()


@pytest.mark.parametrize("quantity", ["prob", "eta"])
@pytest.mark.parametrize("lb", [0.0, 0.1])
def test_analytic_jacobian_matches_autodiff(quantity, lb):
    free, X, g, bounds = _case(2, lb)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(8)
    J = po.prediction_jacobian(free, X, g, K, G, gh_x, gh_w, bounds, quantity=quantity)
    Jt = _torch_prediction(free, X, g, gh_x, gh_w, bounds, quantity)
    assert J.shape == Jt.shape
    assert np.max(np.abs(J.toarray() - Jt)) < 1e-12


def test_lr_variances_are_the_diagonal_of_j_hinv_jt():
    rng = np.random.default_rng(3)
    D = 4 + 2 * K + 2 * G
    A = rng.standard_normal((D, D))
    Hinv = A @ A.T + D * np.eye(D)
    free, X, g, bounds = _case(4, 0.0)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(8)
    J = po.prediction_jacobian(free, X, g, K, G, gh_x, gh_w, bounds)
    Jd = J.toarray()
    np.testing.assert_allclose(po.lr_variances(J, Hinv), np.diag(Jd @ Hinv @ Jd.T), rtol=1e-13)


def test_group_ids_are_checked():
    free, X, _, bounds = _case(5, 0.0)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(8)
    for bad in ([0, 1, 2, 3, 0, 0, 0], [0, -2, 0, 0, 0, 0, 0]):
        with pytest.raises(ValueError):
            po.predict(free, X, np.array(bad), K, G, gh_x, gh_w, bounds)
