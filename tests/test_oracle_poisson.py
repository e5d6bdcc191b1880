"""The Poisson GLMM oracle (oracle/poisson_oracle.py) on the CPU: its analytic KL, gradient, Hessian and HVP against
torch autodiff of the restated KL, the closed-form E_q[exp(eta)] against Gauss-Hermite quadrature, and Newton on the
oracle reaching its optimum."""
import numpy as np
import pytest

from helpers import assert_close
from oracle import glmm_oracle as go
from oracle import poisson_oracle as pois


def _oracle(N, K, G, seed, offset, weights, empty, bounds=0.0):
    X, y, g, off = pois.make_poisson_data(N, K, G - empty, seed, offset=offset)
    rng = np.random.default_rng(seed + 5)
    if empty:
        g = np.sort(rng.choice(G, size=G - empty, replace=False))[g]
    w = None
    if weights:
        w = rng.uniform(0.5, 1.5, N)
        w[rng.choice(N, size=max(1, N // 10), replace=False)] = 0.0
    b = go.GLMMBounds(bounds, bounds, bounds, bounds, bounds)
    return pois.PoissonOracle(X, y, g, offset=off, weights=w, G=G, bounds=b)


CASES = [(200, 3, 8, False, False, 0), (150, 5, 10, True, True, 2), (120, 4, 9, True, False, 3),
         (90, 2, 6, False, True, 1)]


@pytest.mark.parametrize("N,K,G,offset,weights,empty", CASES)
def test_derivatives_match_autodiff(N, K, G, offset, weights, empty):
    o = _oracle(N, K, G, 300 + N, offset, weights, empty, bounds=0.05 if offset else 0.0)
    t = pois.PoissonTorch(o)
    x = go.make_free(o.lay.D, N)
    kl = o.kl(x)
    assert abs(kl - t.value(x)) <= 1e-10 * abs(kl)
    g = o.kl_grad(x)
    assert_close(g, t.grad(x), rtol=1e-10, atol=0.0, scale=np.abs(g).max(), what="gradient")
    H = o.kl_hessian_dense(x)
    assert_close(H, t.hessian(x), rtol=1e-10, atol=0.0, scale=np.abs(H).max(), what="Hessian")
    assert_close(o.kl_hessian_csr(x).toarray(), H, rtol=0.0, atol=0.0, what="CSR")
    v = np.random.default_rng(N).standard_normal(o.lay.D)
    hv = o.kl_hvp(x, v)
    assert_close(hv, t.hvp(x, v), rtol=1e-10, atol=0.0, scale=np.abs(hv).max(), what="HVP")


def test_lgamma_constant_and_zero_weights():
    """The KL depends on rows of weight 0 through nothing, and y enters the constant as w lgamma(y + 1)."""
    o = _oracle(100, 3, 7, 11, True, True, 1)
    x = go.make_free(o.lay.D, 3)
    keep = o.w != 0
    sub = pois.PoissonOracle(o.X[keep], o.y[keep], o.g[keep], offset=o.offset[keep], weights=o.w[keep], G=o.G)
    assert abs(o.kl(x) - sub.kl(x)) <= 1e-12 * abs(o.kl(x))
    y2 = o.y.copy()
    y2[~keep] += 7.0
    o2 = pois.PoissonOracle(o.X, y2, o.g, offset=o.offset, weights=o.w, G=o.G)
    assert o2.kl(x) == o.kl(x)


def test_closed_form_matches_quadrature():
    """E_q[exp(eta)] = exp(m + v / 2) against a 64-node Gauss-Hermite rule, and the oracle's row moments."""
    o = _oracle(60, 4, 5, 21, True, False, 0)
    x = go.make_free(o.lay.D, 5, scale=0.3)
    p = o.unpack(o.free_to_vector(x))
    t = o.obs_terms(p, order=2)
    gx, gw = np.polynomial.hermite.hermgauss(64)
    quad = np.sum(gw / np.sqrt(np.pi) * np.exp(t["z_m"][:, None] + np.sqrt(2 * t["z_v"])[:, None] * gx), axis=1)
    e = np.exp(t["z_m"] + 0.5 * t["z_v"])
    assert_close(quad, e, rtol=1e-13, atol=0.0, what="E exp(eta)")
    assert_close(t["l_m"], o.y - e, rtol=1e-14, atol=1e-14, what="l_m")
    m_ref = p["u_m"][o.g] + o.X @ p["beta_m"] + o.offset
    assert_close(t["z_m"], m_ref, rtol=1e-15, atol=0.0, what="m")


def test_newton_reaches_the_optimum():
    o = _oracle(400, 3, 12, 31, True, True, 2)
    x0 = go.make_free(o.lay.D, 7)
    xo = pois.newton_optimum(o, x0)
    g = o.kl_grad(xo)
    assert np.max(np.abs(g)) < 1e-9
    assert o.kl(xo) < o.kl(x0)
    assert np.all(np.linalg.eigvalsh(o.kl_hessian_dense(xo)) > 0)
