"""Analytic fp64 oracle of the Poisson log-link GLMM for small D (numpy), and a torch-CPU-fp64 autodiff restatement of
its KL.  TEST INFRASTRUCTURE ONLY.

The model is the logistic GLMM of glmm_oracle.py with the observation term replaced: under q the linear predictor
eta_n = x_n . beta + u_g + o_n (o = an offset, e.g. log exposure) is N(m_n, v_n), so E_q[exp(eta_n)] = e_n =
exp(m_n + v_n / 2) exactly and

    E_q log p(y_n | eta_n) = w_n (y_n m_n - e_n - lgamma(y_n + 1)),
    l_m = w (y - e),  l_v = -w e / 2,  l_mm = -w e,  l_mv = -w e / 2,  l_vv = -w e / 4.

Everything else (priors, entropies, random-effect term, the chain rule to free coordinates, the arrowhead blocks,
solves) is GLMMOracle's, which reads the likelihood only through ``obs_terms``; so do the LOO / LOGO / IJ oracles.
"""
import math

import numpy as np
import scipy.special
import torch

from .glmm_oracle import GLMMOracle
from .glmm_torch import digamma_acc, lgamma_acc


class PoissonOracle(GLMMOracle):
    """GLMMOracle with the Poisson log-link observation term; ``offset`` (N,) or None."""

    def __init__(self, X, y, g, offset=None, weights=None, prior=None, bounds=None, G=None):
        super().__init__(X, y, g, np.zeros(0), np.zeros(0), weights=weights, prior=prior, bounds=bounds, G=G)
        self.offset = None if offset is None else np.asarray(offset, dtype=np.float64)

    def obs_terms(self, p, order=2):
        S = self.X * self.X
        z_m = p["u_m"][self.g] + self.X @ p["beta_m"]
        if self.offset is not None:
            z_m = z_m + self.offset
        z_v = (1.0 / p["u_i"])[self.g] + S @ (1.0 / p["beta_i"])
        e = np.exp(z_m + 0.5 * z_v)
        w = np.ones(self.N) if self.w is None else self.w
        out = dict(z_m=z_m, z_v=z_v, S=S, ell=w * (self.y * z_m - e - scipy.special.gammaln(self.y + 1.0)))
        if order >= 1:
            out["l_m"] = w * (self.y - e)
            out["l_v"] = -0.5 * w * e
        if order >= 2:
            out["l_mm"] = -w * e
            out["l_mv"] = -0.5 * w * e
            out["l_vv"] = -0.25 * w * e
        return out


class PoissonTorch:
    """Line-for-line torch spelling of PoissonOracle.kl, differentiated by torch.func (independent of the
    hand-derived derivatives above)."""

    def __init__(self, oracle):
        o = oracle
        self.o = o
        self.X = torch.from_numpy(o.X)
        self.S = self.X * self.X
        self.y = torch.from_numpy(o.y)
        self.g = torch.from_numpy(o.g)
        self.w = None if o.w is None else torch.from_numpy(o.w)
        self.off = None if o.offset is None else torch.from_numpy(o.offset)
        lb = o.lower_bounds()
        self.con = torch.from_numpy(np.isfinite(lb))
        self.lb = torch.from_numpy(np.where(np.isfinite(lb), lb, 0.0))

    def kl(self, free):
        o, lay, pr = self.o, self.o.lay, self.o.prior
        K, G = lay.K, lay.G
        vec = torch.where(self.con, torch.exp(free) + self.lb, free)
        mu_m, mu_i, a, b = vec[0], vec[1], vec[2], vec[3]
        beta_m, beta_i = vec[4:4 + K], vec[4 + K:4 + 2 * K]
        u_m, u_i = vec[lay.u_mean:lay.u_mean + G], vec[lay.u_info:lay.u_info + G]
        z_m = u_m[self.g] + self.X @ beta_m
        if self.off is not None:
            z_m = z_m + self.off
        z_v = (1.0 / u_i)[self.g] + self.S @ (1.0 / beta_i)
        ell = self.y * z_m - torch.exp(z_m + 0.5 * z_v) - torch.lgamma(self.y + 1.0)
        if self.w is not None:
            ell = self.w * ell
        e_tau = a / b
        e_log_tau = digamma_acc(a) - torch.log(b)
        re = torch.sum(-0.5 * e_tau * ((mu_m - u_m) ** 2 + 1 / mu_i + 1 / u_i)) + 0.5 * G * e_log_tau
        loglik = torch.sum(ell) + re
        l2pi = math.log(2 * math.pi)
        ent = (0.5 * (-torch.log(mu_i) + 1 + l2pi)
               + 0.5 * torch.sum(-torch.log(beta_i) + 1 + l2pi)
               + 0.5 * torch.sum(-torch.log(u_i) + 1 + l2pi)
               + a - torch.log(b) + lgamma_acc(a) + (1 - a) * digamma_acc(a))
        prior = (-0.5 * pr.mu_info * ((mu_m - pr.mu_mean) ** 2 + 1 / mu_i)
                 + torch.sum(-0.5 * pr.beta_info * ((beta_m - pr.beta_mean) ** 2 + 1 / beta_i))
                 + (pr.tau_shape - 1) * e_log_tau - pr.tau_rate * e_tau)
        return -(loglik + ent + prior)

    def value(self, free):
        return float(self.kl(torch.as_tensor(free, dtype=torch.float64)))

    def grad(self, free):
        f = torch.as_tensor(free, dtype=torch.float64)
        return torch.func.grad(self.kl)(f).numpy()

    def hessian(self, free):
        f = torch.as_tensor(free, dtype=torch.float64)
        return torch.func.hessian(self.kl)(f).numpy()

    def hvp(self, free, v):
        f = torch.as_tensor(free, dtype=torch.float64)
        v = torch.as_tensor(v, dtype=torch.float64)
        return torch.func.jvp(torch.func.grad(self.kl), (f,), (v,))[1].numpy()


def make_poisson_data(N, K, G, seed, offset=False, rate=1.0):
    """Seeded synthetic Poisson-GLMM data, group-sorted: (X, y, g, offset or None).  rate scales the mean count."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, K)) / np.sqrt(K)
    base, rem = divmod(N, G)
    counts = np.full(G, base, dtype=np.int64)
    counts[:rem] += 1
    g = np.repeat(np.arange(G, dtype=np.int64), counts)
    beta = rng.normal(0.0, 0.5, K)
    u = rng.normal(0.0, 0.4, G)
    off = np.log(rng.uniform(0.5, 2.0, N)) if offset else None
    eta = np.log(rate) + X @ beta + u[g] + (0.0 if off is None else off)
    y = rng.poisson(np.exp(eta)).astype(np.float64)
    return X, y, g, off


def newton_optimum(oracle, x0, tol=1e-10, maxiter=100):
    """Damped Newton on the oracle KL from x0 (dense Hessian, backtracking on the KL): the optimum's free vector."""
    x = np.array(x0, dtype=np.float64)
    f = oracle.kl(x)
    for _ in range(maxiter):
        g = oracle.kl_grad(x)
        if np.max(np.abs(g)) < tol:
            break
        step = np.linalg.solve(oracle.kl_hessian_dense(x), g)
        t = 1.0
        while t > 1e-8:
            xn = x - t * step
            fn = oracle.kl(xn)
            if np.isfinite(fn) and fn <= f:
                break
            t *= 0.5
        x, f = xn, fn
    return x
