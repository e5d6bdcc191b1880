"""Linear-response (LRVB) covariances of the GLMM posterior on the device.

``north_star`` names ``ModelSensitivity.LinearResponseCovariances``; the reference's nearest
code is ``ParametricSensitivityLinearApproximation`` (ModelSensitivity.py:555-612: Cholesky of
the Hessian at the optimum, then ``-cho_solve(chol, cross_hessian)``) and ``Example.ipynb`` cell
15 (``-solve(objective_hess, summary_jac.T)``); the class with this name lives in the successor
library (README.md:14).  This module provides it over the CUDA path:

    Cov(m) = J_m H^{-1} J_m^T,      J_m = d m / d free at the optimum,

where ``H^{-1}`` is applied either by the direct arrowhead solve (Schur complement of the 2x2
local blocks, csrc/solve.cu k_schur on the FP64 tensor cores + small SPD inverse) or by the
device conjugate gradient -- the dense ``cho_factor`` of the reference is O(D^3) and is not used.
"""
import numpy as np
import scipy.sparse

from .GLMM import ApproximateMaxInfluence, DropResult
from ._tensors import is_torch, to_device


class LinearResponseCovariances(object):
    def __init__(self, objective, opt_par_value, validate_optimum=False, grad_tol=1e-8,
                 method="schur", cg_tol=1e-8, cg_preconditioner="block_jacobi"):
        """objective: a device ``SparseObjectives.Objective``; opt_par_value: the free parameter
        at the optimum (numpy or CUDA tensor).  method: 'schur' (direct) or 'cg'."""
        if not getattr(getattr(objective, "model", None), "_lrvb_device_model", False):
            raise TypeError("LinearResponseCovariances needs a device Objective")
        if method not in ("schur", "cg"):
            raise ValueError("method must be 'schur' or 'cg'")
        self.objective = objective
        self.model = objective.model
        self.method = method
        self.cg_tol = cg_tol
        self.cg_preconditioner = cg_preconditioner
        self.cg_infos = []
        self.cg_iterations = []
        self.set_base_values(opt_par_value, validate_optimum, grad_tol)

    def set_base_values(self, opt_par_value, validate_optimum=False, grad_tol=1e-8):
        self._opt0 = opt_par_value
        if validate_optimum:
            g = self.objective.fun_free_grad(opt_par_value)
            gmax = float(abs(g).max())
            if gmax > grad_tol:
                raise ValueError("Gradient at the claimed optimum has max-abs {} > {}".format(
                    gmax, grad_tol))
        self.model.evaluate(opt_par_value, 2, "free")
        self._sinv = None
        self._pred_blocks = None      # (cross, local covariances) of get_prediction_variances

    def _ensure_point(self):
        self.model.evaluate(self._opt0, 2, "free")

    # ---- pieces ----
    def get_hessian_at_opt(self):
        """Sparse Hessian at the optimum (scipy CSR for numpy input, DeviceCSR for torch)."""
        return self.objective.fun_free_hessian(self._opt0)

    def get_global_covariance(self):
        """(H^{-1})[:Dg,:Dg]: LRVB covariance of the global free parameters (Dg,Dg).  method
        'schur': one Schur complement + SPD inverse; method 'cg': Dg conjugate-gradient solves with
        device Hessian-vector products (ConjugateGradient.py:81-105; BASELINE configs[3]), their
        ``info`` / iteration counts appended to ``cg_infos`` / ``cg_iterations``."""
        import torch
        self._ensure_point()
        if self.method == "cg":
            Dg, D = self.model.Dg, self.model.D
            cov = torch.empty(Dg, Dg, dtype=torch.float64, device=self.model.device)
            e = torch.zeros(D, dtype=torch.float64, device=self.model.device)
            for i in range(Dg):
                e.zero_()
                e[i] = 1.0
                x, info, iters = self.model.cg(e, None, precond=self._cg_precond(), rtol=self.cg_tol)
                self.cg_infos.append(info)
                self.cg_iterations.append(iters)
                cov[i] = x[:Dg]
            cov = 0.5 * (cov + cov.t())
            return cov if is_torch(self._opt0) else cov.cpu().numpy()
        if self._sinv is None:
            self._sinv = self.model.global_covariance()
        return self._sinv if is_torch(self._opt0) else self._sinv.cpu().numpy()

    def _cg_precond(self):
        p = self.cg_preconditioner
        return 0 if p is None else p

    def get_local_covariances(self):
        """Per-group LRVB covariance of (u.mean_g, u.info_g) free parameters, (G,3)=(mm,mi,ii)."""
        self._ensure_point()
        if self._sinv is None:
            self._sinv = self.model.global_covariance()
        cov = self.model.local_cov(self._sinv)
        return cov if is_torch(self._opt0) else cov.cpu().numpy()

    def hinv(self, rhs):
        """H^{-1} rhs for rhs (D,) or (nrhs, D) -> same shape (device tensor)."""
        import torch
        self._ensure_point()
        if self.method == "schur":
            return self.model.solve(rhs)
        if scipy.sparse.issparse(rhs):
            rhs = rhs.toarray()
        shape = tuple(rhs.shape)
        rows = rhs.reshape(-1, self.model.D)
        out = []
        for row in rows:
            x, info, iters = self.model.cg(row, None, precond=self._cg_precond(), rtol=self.cg_tol)
            self.cg_infos.append(info)
            self.cg_iterations.append(iters)
            out.append(x)
        return torch.stack(out).reshape(shape)

    def get_moment_jacobian(self, calculate_moments=None):
        """Jacobian of the moments w.r.t. the free parameters.  The model's analytic
        [E mu, E tau, E beta, E u] Jacobian is used; an arbitrary ``calculate_moments`` callable
        would need autodiff, which this library does not provide."""
        if calculate_moments is not None:
            raise TypeError("pass explicit Jacobians to get_lr_covariance_from_jacobians; "
                            "arbitrary moment callables need autodiff")
        x = self._opt0.detach().cpu().numpy() if is_torch(self._opt0) else self._opt0
        return self.model.moment_jacobian(x)

    def get_lr_covariance_factors(self, moment_jacobian1, moment_jacobian2=None):
        """J1 H^{-1} J2^T WITHOUT forming H^{-1} J2^T (a dense (m2, D) block -- 160 GB at the target size)
        or the (m1, m2) result: for the arrowhead H = [[A, B^T], [B, L]] with S = A - B^T L^{-1} B and
        T = L^{-1} B,

            J1 H^{-1} J2^T = W1 S^{-1} W2^T + J1l L^{-1} J2l^T,      W = Jg - Jl T   (m, Dg),

        where Jg / Jl are the global / local columns of a Jacobian.  The Jacobians stay sparse (scipy
        sparse, dense arrays or torch tensors are accepted); the only dense objects are (m, Dg).
        Returns an ``ArrowheadCovariance`` (``diagonal()``, ``block(rows1, rows2)``, ``matvec``,
        ``toarray()`` for small m)."""
        import torch
        if moment_jacobian2 is None:
            moment_jacobian2 = moment_jacobian1
        model = self.model
        local = getattr(model, "local", None)
        if local is not None:
            raise NotImplementedError("factored covariances of a sharded model: use get_global_covariance / "
                                      "get_local_covariances, or hinv() on explicit right-hand sides")
        self._ensure_point()
        if self._sinv is None:
            self._sinv = model.global_covariance()
        Dg, G, D = model.Dg, model.G, model.D
        _, B, L = model.blocks()
        det = L[:, 0] * L[:, 2] - L[:, 1] * L[:, 1]
        linv = torch.stack([L[:, 2] / det, -L[:, 1] / det, L[:, 0] / det], dim=1)          # (G, 3): 00, 01, 11
        # T in the column order of the local parameters [u.mean (G) | u.info (G)]: (2G, Dg)
        T = torch.cat([linv[:, 0:1] * B[:, 0, :] + linv[:, 1:2] * B[:, 1, :],
                       linv[:, 1:2] * B[:, 0, :] + linv[:, 2:3] * B[:, 1, :]], dim=0)
        linv_h = linv.cpu().numpy()

        def split(j):
            if is_torch(j):
                j = j.detach().cpu().numpy()
            js = scipy.sparse.csr_matrix(j) if not scipy.sparse.issparse(j) else j.tocsr()
            if js.shape[1] != D:
                raise ValueError("Wrong number of columns for a moment Jacobian.  Expected {}, got {}".format(
                    D, js.shape[1]))
            jg = torch.from_numpy(np.ascontiguousarray(js[:, :Dg].toarray())).to(model.device)
            jl = js[:, Dg:].tocsr()
            jl_t = torch.sparse_csr_tensor(torch.from_numpy(jl.indptr.astype(np.int64)),
                                           torch.from_numpy(jl.indices.astype(np.int64)),
                                           torch.from_numpy(jl.data.astype(np.float64)),
                                           size=jl.shape).to(model.device)
            w = jg - (torch.sparse.mm(jl_t, T) if jl.nnz else torch.zeros_like(jg))
            return w, jl

        w1, jl1 = split(moment_jacobian1)
        same = moment_jacobian2 is moment_jacobian1
        w2, jl2 = (w1, jl1) if same else split(moment_jacobian2)
        # sparse local term J1l L^-1 J2l^T on the host (L^-1 is 2x2 block diagonal)
        gi = np.arange(G)
        Ls = scipy.sparse.csr_matrix(
            (np.concatenate([linv_h[:, 0], linv_h[:, 1], linv_h[:, 1], linv_h[:, 2]]),
             (np.concatenate([gi, gi, gi + G, gi + G]), np.concatenate([gi, gi + G, gi, gi + G]))), (2 * G, 2 * G))
        local_term = (jl1 @ Ls @ jl2.T).tocsr()
        return ArrowheadCovariance(w1, self._sinv, w2, local_term, symmetric=same)

    def get_prediction_variances(self, X_new, groups_new):
        """Predictions for new rows with their LRVB variances at the optimum: a ``GLMM.Prediction`` with
        eta_mean, eta_var_mfvb, prob, prob_var_mfvb, prob_var_lr, eta_var_lr, where the LR variance of a
        row is j H^{-1} j^T for j = its gradient with respect to the free parameters
        (``model.prediction_jacobian``).  Always from the direct arrowhead pieces (S^{-1}, the beta x local
        block of H^{-1} and the local covariances), whatever ``method`` is; one device pass over the rows
        (csrc/predict.cu), nothing of size (M, D) or (M, Dg) is formed.  Covariances BETWEEN rows:
        ``get_lr_covariance_factors(model.prediction_jacobian(...))``."""
        model = self.model
        if getattr(model, "local", None) is not None:
            raise NotImplementedError("prediction of a sharded model: build a single-GPU LogisticGLMM of the "
                                      "job and use its LinearResponseCovariances")
        self._ensure_point()
        if self._sinv is None:
            self._sinv = model.global_covariance()
        if self._pred_blocks is None:
            self._pred_blocks = (model.prediction_cross(self._sinv), model.local_cov(self._sinv))
        cross, lcov = self._pred_blocks
        return model.predict_lr(self._sinv, cross, lcov, X_new, groups_new)

    def get_approximate_loo(self):
        """Approximate leave-one-out cross-validation of the training rows at the optimum by the infinitesimal
        jackknife (Giordano et al., "A Swiss Army Infinitesimal Jackknife"): a ``GLMM.ApproximateLOO`` with the
        pointwise lpd, lpd_loo, eta_mean_loo, eta_var_loo (caller's row order; numpy for a numpy optimum, CUDA
        tensors for a CUDA one) and elpd_loo, elpd_loo_se, p_loo, n_invalid.  The same as dropping each row's
        weight in ``WeightSensitivityLinearApproximation`` and pushing the shift of the optimum through the row's
        moments, for all N rows in one device pass instead of N solves.  Always from the direct arrowhead
        pieces, whatever ``method`` is (cached with ``get_prediction_variances``)."""
        model = self.model
        if getattr(model, "local", None) is not None:
            raise NotImplementedError("approximate LOO of a sharded model: build a single-GPU LogisticGLMM of the "
                                      "job and use its LinearResponseCovariances")
        model._check_binary_y()
        self._ensure_point()
        if self._sinv is None:
            self._sinv = model.global_covariance()
        if self._pred_blocks is None:
            self._pred_blocks = (model.prediction_cross(self._sinv), model.local_cov(self._sinv))
        cross, lcov = self._pred_blocks
        r = model.approximate_loo(self._sinv, cross, lcov)
        if is_torch(self._opt0):
            return r
        return r._replace(**{f: getattr(r, f).cpu().numpy() for f in ("lpd", "lpd_loo", "eta_mean_loo",
                                                                      "eta_var_loo")})

    def get_approximate_logo(self):
        """Approximate leave-one-group-out cross-validation and group influence at the optimum by the infinitesimal
        jackknife: a ``GLMM.ApproximateLOGO`` with the pointwise lpd_logo, eta_mean_logo, eta_var_logo (caller's row
        order), the per-group elpd_logo_group, cooks_distance and delta_global (G, Dg), and elpd_logo, elpd_logo_se;
        numpy for a numpy optimum, CUDA tensors for a CUDA one.  delta_global[g] is the global block of
        ``WeightSensitivityLinearApproximation.get_dinput_dhyper_times`` with the weights of group g's rows dropped,
        for all groups at once.  Always from S^-1, whatever ``method`` is (cached with ``get_prediction_variances``)."""
        model = self.model
        if getattr(model, "local", None) is not None:
            raise NotImplementedError("approximate LOGO of a sharded model: build a single-GPU LogisticGLMM of the "
                                      "job and use its LinearResponseCovariances")
        model._check_binary_y()
        self._ensure_point()
        if self._sinv is None:
            self._sinv = model.global_covariance()
        r = model.approximate_logo(self._sinv)
        if is_torch(self._opt0):
            return r
        return r._replace(**{f: getattr(r, f).cpu().numpy() for f in ("lpd_logo", "eta_mean_logo", "eta_var_logo",
                                                                      "elpd_logo_group", "cooks_distance",
                                                                      "delta_global")})

    def get_approximate_max_influence(self, c, unit="row", level=0.95, max_fraction=0.1):
        """The approximate maximum influence perturbation (AMIP, Broderick, Giordano and Meager) of the contrast
        phi = c^T E[beta] at the optimum: how few rows (unit="row") or whole groups (unit="group") must be dropped to
        change its sign, its significance at ``level``, or to make it significant with the opposite sign.  ``c`` is a
        length-K vector or an integer k (e_k).  Returns a ``GLMM.ApproximateMaxInfluence``; per-unit fields are numpy
        for a numpy optimum and CUDA tensors for a CUDA one.

        With a = H^-1 chat (chat = c on the beta.mean block), b = H^-1 t and t = D^3 KL[a, a, .]
        (``model.third_derivative_contraction``), dropping unit u (w_n -> 0 on its rows) moves phi and
        sd_lr^2 = chat^T H^-1 chat to first order by sum_{n in u} w_n (C^T a)_n and -sum_{n in u} w_n (q_n + (C^T b)_n)
        (C = d^2 KL / d theta d w, ``weight_cross_rmatvec``).  Each target is a linear statistic -- s phi,
        s phi - z sd_lr, s phi + z sd_lr with s = sign(phi) -- and its search sorts the units of non-zero weight by
        their push toward zero (ties by index) and takes the shortest prefix that carries the statistic across zero,
        of at most floor(max_fraction * units) units.  Always from the direct arrowhead pieces, whatever ``method``
        is."""
        import scipy.special
        import torch
        model = self.model
        if getattr(model, "local", None) is not None:
            raise NotImplementedError("approximate maximum influence of a sharded model: build a single-GPU "
                                      "LogisticGLMM of the job and use its LinearResponseCovariances")
        if unit not in ("row", "group"):
            raise ValueError("unit must be 'row' or 'group', got %r" % (unit,))
        level, max_fraction = float(level), float(max_fraction)
        if not 0.0 < level < 1.0:
            raise ValueError("level must lie in (0, 1), got %r" % (level,))
        if not 0.0 < max_fraction <= 1.0:
            raise ValueError("max_fraction must lie in (0, 1], got %r" % (max_fraction,))
        chat = self._contrast(c)
        self._ensure_point()
        if self._sinv is None:
            self._sinv = model.global_covariance()
        dev = model.device
        ch = torch.from_numpy(chat).to(dev)

        def solve(rhs):
            return model.solve_finish(self._sinv, model.solve_reduce_rhs(rhs), rhs)

        a = solve(ch)
        x = self._opt0.detach().to(dev, torch.float64) if is_torch(self._opt0) else \
            torch.from_numpy(np.asarray(self._opt0, dtype=np.float64)).to(dev)
        t, q = model.third_derivative_contraction(a)
        b = solve(t)
        ca, cb = model.weight_cross_rmatvec(a), model.weight_cross_rmatvec(b)
        w = torch.ones(model.N, dtype=torch.float64, device=dev) if model.w is None else model.w
        perm = None if model.perm is None else to_device(model.perm, torch.int64)
        if perm is not None:                     # caller's row order
            w = torch.empty_like(w).index_copy_(0, perm, w)
        est, var = float(torch.dot(ch, x.reshape(-1))), float(torch.dot(ch, a))
        if not var > 0.0:
            raise np.linalg.LinAlgError("the LRVB variance of the contrast is {} (not positive)".format(var))
        sd = float(np.sqrt(var))
        mean_shift = w * ca
        sd_shift = -w * (q + cb) / (2.0 * sd)
        keep = w != 0
        if unit == "group":
            # the model's rows are group-sorted: fixed-order segment sums, no atomics
            counts = torch.bincount(model.g.to(torch.int64), minlength=model.G)
            srt = (lambda v: v) if perm is None else (lambda v: v.index_select(0, perm))
            gsum = lambda v: torch.segment_reduce(srt(v), "sum", lengths=counts, initial=0.0)   # noqa: E731
            mean_shift, sd_shift = gsum(mean_shift), gsum(sd_shift)
            keep = gsum(keep.to(torch.float64)) > 0
        z = float(scipy.special.ndtri(0.5 + 0.5 * level))
        s = 1.0 if est >= 0 else -1.0
        linear = dict(sign=(s * est, s * mean_shift),
                      significance=(s * est - z * sd, s * mean_shift - z * sd_shift),
                      significant_opposite=(s * est + z * sd, s * mean_shift + z * sd_shift))
        elig = torch.nonzero(keep).reshape(-1)
        nmax = int(np.floor(max_fraction * elig.numel() + 1e-9))
        host = not is_torch(self._opt0)
        targets = {}
        for name, (stat, push) in linear.items():
            side = 1.0 if stat >= 0 else -1.0
            key, order = torch.sort(side * push.index_select(0, elig), stable=True)
            hit = torch.nonzero(side * stat + torch.cumsum(key[:nmax], 0) < 0).reshape(-1)
            if hit.numel() == 0:
                drop = elig[:0]
                targets[name] = DropResult(None, None, drop.cpu().numpy() if host else drop, None, None)
                continue
            n = int(hit[0]) + 1
            drop = elig.index_select(0, order[:n])
            targets[name] = DropResult(n, n / elig.numel(), drop.cpu().numpy() if host else drop,
                                       est + float(mean_shift.index_select(0, drop).sum()),
                                       sd + float(sd_shift.index_select(0, drop).sum()))
        if host:
            mean_shift, sd_shift = mean_shift.cpu().numpy(), sd_shift.cpu().numpy()
        return ApproximateMaxInfluence(est, sd, z, mean_shift, sd_shift, targets)

    def _contrast(self, c):
        """c (length K, numpy / list / torch) or an integer k -> chat (D,) numpy with c on the beta.mean block."""
        K, D = self.model.K, self.model.D
        chat = np.zeros(D)
        if isinstance(c, (int, np.integer)) and not isinstance(c, (bool, np.bool_)):
            if not 0 <= int(c) < K:
                raise ValueError("coefficient index must lie in [0, {}), got {}".format(K, int(c)))
            chat[4 + int(c)] = 1.0
            return chat
        v = c.detach().cpu().numpy() if is_torch(c) else np.asarray(c)
        if v.ndim != 1 or v.shape[0] != K or not np.issubdtype(v.dtype, np.number) or \
                np.issubdtype(v.dtype, np.complexfloating):
            raise ValueError("c must be an integer in [0, {0}) or a real vector of length {0}".format(K))
        v = v.astype(np.float64)
        if not np.all(np.isfinite(v)) or not np.any(v != 0):
            raise ValueError("c must be finite and not all zero")
        chat[4:4 + K] = v
        return chat

    MAX_DENSE = 1 << 26

    def get_lr_covariance_from_jacobians(self, moment_jacobian1, moment_jacobian2=None):
        """J1 H^{-1} J2^T for (m1, D) / (m2, D) Jacobians (dense, scipy-sparse or torch) as a dense
        matrix; beyond 2^26 entries use ``get_lr_covariance_factors``."""
        import torch
        if moment_jacobian2 is None:
            moment_jacobian2 = moment_jacobian1
        m1, m2 = moment_jacobian1.shape[0], moment_jacobian2.shape[0]
        if m1 * m2 > self.MAX_DENSE:
            raise ValueError("the covariance would have {} x {} entries; use get_lr_covariance_factors "
                             "(diagonal / blocks / products without the dense matrix)".format(m1, m2))
        if self.method == "schur" and getattr(self.model, "local", None) is None:
            cov = self.get_lr_covariance_factors(moment_jacobian1, moment_jacobian2).toarray()
            cov = torch.from_numpy(cov) if not is_torch(cov) else cov
            return cov.to(self.model.device) if (is_torch(moment_jacobian1) or is_torch(self._opt0)) \
                else cov.cpu().numpy()

        def dense(j):
            if scipy.sparse.issparse(j):
                j = j.toarray()
            return j.reshape(-1, self.model.D)

        hinv_j2t = self.hinv(dense(moment_jacobian2))   # (m2, D): rows are H^{-1} J2[i]
        j1 = dense(moment_jacobian1)
        if not is_torch(j1):
            j1 = torch.from_numpy(np.ascontiguousarray(j1, dtype=np.float64))
        cov = torch.matmul(j1.to(hinv_j2t.device), hinv_j2t.t())
        return cov if (is_torch(moment_jacobian1) or is_torch(self._opt0)) else cov.cpu().numpy()

    def get_lr_covariance(self, calculate_moments=None):
        """LRVB covariance of the model's default moments [E mu, E tau, E beta, E u]."""
        j = self.get_moment_jacobian(calculate_moments)
        return self.get_lr_covariance_from_jacobians(j, j)


class ArrowheadCovariance(object):
    """C = W1 Sinv W2^T + R with W (m, Dg) dense on the device, Sinv (Dg, Dg), R (m1, m2) scipy sparse:
    the linear-response covariance J1 H^{-1} J2^T of an arrowhead Hessian in factored form."""

    def __init__(self, w1, sinv, w2, local_term, symmetric=False):
        self.w1, self.sinv, self.w2, self.local_term, self.symmetric = w1, sinv, w2, local_term, symmetric
        self.shape = (w1.shape[0], w2.shape[0])

    def diagonal(self):
        """diag(C) (m1 == m2) as a numpy array."""
        import torch
        assert self.shape[0] == self.shape[1]
        d = torch.sum(torch.matmul(self.w1, self.sinv) * self.w2, dim=1)
        return d.cpu().numpy() + self.local_term.diagonal()

    def block(self, rows1, rows2):
        """Dense C[rows1][:, rows2] (index arrays or slices) as numpy."""
        import torch
        r1 = np.arange(self.shape[0])[rows1]
        r2 = np.arange(self.shape[1])[rows2]
        t1 = torch.from_numpy(r1).to(self.w1.device)
        t2 = torch.from_numpy(r2).to(self.w1.device)
        low = torch.matmul(torch.matmul(self.w1.index_select(0, t1), self.sinv), self.w2.index_select(0, t2).t())
        return low.cpu().numpy() + self.local_term[r1][:, r2].toarray()

    def matvec(self, v):
        """C v for v (m2,) numpy -> numpy."""
        import torch
        vt = torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).to(self.w1.device)
        low = torch.matmul(self.w1, torch.matmul(self.sinv, torch.matmul(self.w2.t(), vt)))
        return low.cpu().numpy() + self.local_term @ np.asarray(v, dtype=np.float64)

    def toarray(self):
        if self.shape[0] * self.shape[1] > LinearResponseCovariances.MAX_DENSE:
            raise ValueError("covariance of {} x {} entries: use diagonal() / block() / matvec()".format(*self.shape))
        import torch
        low = torch.matmul(torch.matmul(self.w1, self.sinv), self.w2.t())
        return low.cpu().numpy() + self.local_term.toarray()


class WeightSensitivityLinearApproximation(object):
    """Linear approximation of the optimum as a function of the observation weights: the
    reference's ``ParametricSensitivityLinearApproximation`` (ModelSensitivity.py:555-612) with
    ``hyper_par`` = the weight vector of the GLMM.  There the sensitivity is the dense matrix
    ``-cho_solve(chol(H), cross_hessian)`` of shape (D, N); here it is an operator

        d input / d hyper = -H^{-1} C,    C = d^2 KL / d free d w   (column n = -grad l_n)

    applied with the device cross-Hessian products (csrc/sensitivity.cu) and the arrowhead solve,
    so N = 10^6..10^7 observations are fine.  ``get_dinput_dhyper()`` still returns the dense
    matrix when it is small enough to be a matrix.
    """
    MAX_DENSE = 1 << 24

    def __init__(self, objective, input_val0, hyper_val0=None, method="schur"):
        self.lr = LinearResponseCovariances(objective, input_val0, method=method)
        self.model = objective.model
        if not hasattr(self.model, "weight_cross_matvec"):
            raise TypeError("the model does not provide the weight cross-Hessian")
        self.input_val0 = input_val0
        n = self.model.N
        if hyper_val0 is None:
            w = getattr(self.model, "w", None)
            hyper_val0 = np.ones(n) if w is None else self._to_caller_order(w)
        self.hyper_val0 = np.asarray(hyper_val0, dtype=np.float64).reshape(-1)
        if self.hyper_val0.size != n:
            raise ValueError("Wrong size for weights.  Expected {}, got {}".format(
                n, self.hyper_val0.size))

    def _to_caller_order(self, w_sorted):
        w = w_sorted.detach().cpu().numpy()
        if self.model.perm is None:
            return w
        perm = np.asarray(self.model.perm.cpu() if is_torch(self.model.perm) else self.model.perm)
        out = np.empty_like(w)
        out[perm] = w
        return out

    def _ret(self, t):
        return t if is_torch(self.input_val0) else t.cpu().numpy()

    def get_dinput_dhyper_times(self, hyper_diff):
        """(d input / d hyper) @ hyper_diff -> (D,): the first-order change of the optimum."""
        self.lr._ensure_point()
        return self._ret(-self.lr.hinv(self.model.weight_cross_matvec(hyper_diff)))

    def get_dhyper_influence(self, v):
        """(d input / d hyper)^T v -> (N,): the influence of every observation's weight on the
        functional ``v . input`` (e.g. a row of a moment Jacobian)."""
        self.lr._ensure_point()
        return self._ret(-self.model.weight_cross_rmatvec(self.lr.hinv(v)))

    def get_dinput_dhyper(self):
        """The dense (D, N) Jacobian, as in the reference (only when D * N <= 2^24 entries)."""
        import torch
        D, n = self.model.D, self.model.N
        if D * n > self.MAX_DENSE:
            raise ValueError("d input / d hyper would have {} x {} entries; use "
                             "get_dinput_dhyper_times / get_dhyper_influence".format(D, n))
        eye = torch.eye(D, dtype=torch.float64, device=self.model.device)
        rows = [self.get_dhyper_influence(eye[i]) for i in range(D)]
        rows = [r if is_torch(r) else torch.from_numpy(r) for r in rows]
        return self._ret(torch.stack([r.to(self.model.device) for r in rows]))

    def predict_input_par_from_hyperparameters(self, new_hyper_par_value):
        diff = np.asarray(new_hyper_par_value, dtype=np.float64).reshape(-1) - self.hyper_val0
        step = self.get_dinput_dhyper_times(diff)
        if is_torch(self.input_val0):
            return self.input_val0 + step
        return np.asarray(self.input_val0, dtype=np.float64) + step
