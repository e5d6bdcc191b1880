"""Logistic and Poisson GLMM variational objectives bound to the CUDA library (single GPU).

The reference has no GLMM class: its users compose this KL from ``UVNParam`` / ``GammaParam`` /
``UVNParamVector`` bundles, ``Modeling.get_e_logistic_term_guass_hermite`` (Modeling.py:35-52)
and ``ExponentialFamilies`` terms (SURVEY.md A.1) inside a zero-argument ``fun`` handed to
``Objective(par, fun)`` (SparseObjectives.py:95-100), and autograd differentiates it.  Here the
same composition is a model object: it owns the ``ModelParamsDict`` (so the flat layout is the
reference's, ParameterDictionary.py:39-46) and evaluates value / gradient / arrowhead Hessian /
HVP / solves by calling ``liblrvb_b200.so`` through ctypes.  ``SparseObjectives.Objective``
accepts it in place of ``fun``.

    KL(free) = -( sum_n w_n [y_n z_n - GH(z_mean_n, z_sd_n)]
                  + sum_g [-1/2 E[tau]((E mu - E u_g)^2 + Var mu + Var u_g) + 1/2 E log tau]
                  + entropies(mu, beta, u, tau) + priors(mu, beta, tau) )

``PoissonGLMM`` is the same objective with the Poisson log-link observation term
w_n [y_n m_n - exp(m_n + v_n / 2) - lgamma(y_n + 1)] (m_n, v_n: mean and variance of the linear predictor, offset
included), exact under q.
"""
import ctypes
import weakref
from collections import namedtuple
from dataclasses import dataclass

import numpy as np

from . import _native as nat
from ._tensors import PointKey, is_torch, like_input, to_device
from .GammaParams import GammaParam
from .NormalParams import UVNParam, UVNParamVector
from .ParameterDictionary import ModelParamsDict


@dataclass
class GLMMPrior:
    """mu ~ N(mu_mean, 1/mu_info), beta_k ~ N(beta_mean, 1/beta_info), tau ~ Gamma(shape, rate)
    (ExponentialFamilies.py:191-195)."""
    mu_mean: float = 0.0
    mu_info: float = 0.01
    beta_mean: float = 0.0
    beta_info: float = 0.01
    tau_shape: float = 3.0
    tau_rate: float = 3.0


Prediction = namedtuple("Prediction", ["eta_mean", "eta_var_mfvb", "prob", "prob_var_mfvb", "prob_var_lr",
                                       "eta_var_lr"])
Prediction.__doc__ = """Per-row predictions for new observations (``LogisticGLMM.predict``,
``LinearResponseCovariances.get_prediction_variances``): the linear predictor eta = u_g + x.beta and
prob = E_q[sigma(eta)] with their mean-field variances and, from the linear-response pass, their LRVB
variances (None where not computed)."""

ApproximateLOO = namedtuple("ApproximateLOO", ["lpd", "lpd_loo", "eta_mean_loo", "eta_var_loo", "elpd_loo",
                                               "elpd_loo_se", "p_loo", "n_invalid"])
ApproximateLOO.__doc__ = """Approximate leave-one-out cross-validation of the training rows by the infinitesimal
jackknife (``LogisticGLMM.approximate_loo``, ``LinearResponseCovariances.get_approximate_loo``).  Per row (N,), in
the caller's row order: lpd = log E_q[p(y_n | eta)], lpd_loo = the same with q moved to the IJ estimate of the fit
without row n, and the moments eta_mean_loo, eta_var_loo of eta = u_g + x.beta there (NaN in lpd_loo and
eta_var_loo where the shifted variance is <= 0).  Scalars: elpd_loo = sum lpd_loo, p_loo = sum lpd - elpd_loo,
elpd_loo_se = sqrt(N) std(lpd_loo, ddof=1) (NaN when n_invalid > 0), n_invalid = rows with NaN."""

ApproximateLOGO = namedtuple("ApproximateLOGO", ["lpd_logo", "eta_mean_logo", "eta_var_logo", "elpd_logo_group",
                                                 "cooks_distance", "delta_global", "elpd_logo", "elpd_logo_se"])
ApproximateLOGO.__doc__ = """Approximate leave-one-group-out cross-validation and group influence by the infinitesimal
jackknife (``LogisticGLMM.approximate_logo``, ``LinearResponseCovariances.get_approximate_logo``).  Per row (N,), in
the caller's row order: lpd_logo = log E_q[p(y_n | eta)] with the globals at the IJ estimate of the fit without the
row's group and q(u_g) at its optimum without the group's rows (mean E[mu], info max(E[tau], lb)), and the moments
eta_mean_logo, eta_var_logo of eta = u_g + x.beta there.  Per group (G,): elpd_logo_group = the sum of lpd_logo over
the group's rows, cooks_distance = delta_beta^T P^-1 delta_beta / K (P = the LRVB covariance of E[beta]) and
delta_global (G, Dg) = the IJ shift of the global free parameters.  Scalars: elpd_logo = sum lpd_logo, elpd_logo_se =
sqrt(G') std(elpd_logo_group over the G' non-empty groups, ddof=1) (NaN when G' < 2).  An empty group has zero
delta_global, cooks_distance and elpd_logo_group."""

IJCovariance = namedtuple("IJCovariance", ["unit", "n_units", "global_cov", "moment_cov", "beta_cov", "beta_se_ij",
                                           "beta_se_lr"])
IJCovariance.__doc__ = """The infinitesimal-jackknife (IJ) approximation of the bootstrap covariance of the global
parameters (``LinearResponseCovariances.get_ij_covariance``), with rows or whole groups resampled (unit = "row" or
"group"; "group" is the cluster-robust sandwich covariance).  n_units = the units of non-zero weight; global_cov (Dg, Dg)
in free coordinates; moment_cov (2+K, 2+K) of [E mu, E tau, E beta]; beta_cov (K, K) of E[beta]; beta_se_ij = the
square root of its diagonal; beta_se_lr = the LRVB (posterior) standard deviations of E[beta], for comparison."""

DropResult = namedtuple("DropResult", ["n_drop", "fraction", "dropped", "predicted_estimate", "predicted_sd"])
DropResult.__doc__ = """One target of ``LinearResponseCovariances.get_approximate_max_influence``: the fewest units (rows or
groups) whose removal the first-order prediction says is enough to reach the target, n_drop (None if no such set
within max_fraction), fraction = n_drop over the units of non-zero weight, dropped = their indices (caller's row order
or group ids, most influential first), and the predicted estimate and sd_lr without them (None with n_drop)."""

ApproximateMaxInfluence = namedtuple("ApproximateMaxInfluence", ["estimate", "sd_lr", "z", "mean_shift", "sd_shift",
                                                                 "targets"])
ApproximateMaxInfluence.__doc__ = """The approximate maximum influence perturbation (AMIP) of phi = c^T E[beta]
(``LinearResponseCovariances.get_approximate_max_influence``).  Scalars: estimate = phi, sd_lr = its LRVB standard
deviation sqrt(c^T H^-1 c), z = the normal quantile of the interval phi +/- z sd_lr.  Per unit (rows in the caller's
order, or groups by id): mean_shift and sd_shift, the first-order changes of phi and sd_lr when the unit is dropped
(its weights set to 0).  targets: dict of ``DropResult`` for "sign" (phi crosses 0), "significance" (the interval
bound nearest 0 crosses it) and "significant_opposite" (the far bound crosses 0)."""


class _DevView(object):
    """Zero-copy torch view of library-owned device memory (__cuda_array_interface__)."""

    def __init__(self, ptr, shape, typestr="<f8"):
        self.__cuda_array_interface__ = {
            "shape": tuple(int(s) for s in shape), "typestr": typestr,
            "data": (int(ptr), False), "version": 2, "strides": None}


def _view(ptr, shape, owner):
    torch = nat.require_cuda()
    n = int(np.prod(shape))
    if n == 0:
        return torch.empty(tuple(shape), dtype=torch.float64, device="cuda")
    t = torch.as_tensor(_DevView(ptr, shape), device="cuda")
    t._lrvb_owner = owner  # keep the handle alive as long as the view
    return t


class _Pattern(object):
    """One exported sparsity pattern: device ``crow`` (D+1) / ``col`` (capacity) int32, the nnz (device
    scalar, read once when first needed) and, once some caller has asked for a host matrix, the host
    copies of the index arrays (read-only, shared by the scipy matrices handed out)."""
    __slots__ = ("crow", "col", "nnz_dev", "_nnz", "shape", "host_template", "host_blocks")

    def __init__(self, crow, col, nnz_dev, shape):
        self.crow, self.col, self.nnz_dev, self._nnz, self.shape = crow, col, nnz_dev, None, tuple(shape)
        self.host_template = None
        self.host_blocks = []      # [pinned tensor, weakref to the ndarray handed out on it (or None)]

    def host_block(self, torch, nnz, dtype):
        """A pinned host block for ``data``: one whose previous ndarray is gone is used again, otherwise a new
        one is pinned (milliseconds).  The pattern owns its blocks, so in steady state a caller that drops --
        or still holds -- the previous matrix when it asks for the next one rotates between the same two
        blocks and no step ever waits for ``cudaHostAlloc`` (torch's caching host allocator hands a freed
        block out again only once the event of its last copy has been seen complete: sporadic re-pinning,
        2 ms steps among 0.6 ms ones)."""
        for ent in self.host_blocks:
            if (ent[1] is None or ent[1]() is None) and ent[0].numel() >= nnz and ent[0].dtype == dtype:
                return ent
        ent = [torch.empty(nnz, dtype=dtype, pin_memory=True), None]
        self.host_blocks.append(ent)
        return ent

    @property
    def nnz(self):
        if self._nnz is None:
            self._nnz = int(self.nnz_dev.item())
        return self._nnz


class _PendingRefill(object):
    """A refill whose pattern check has not been read yet: the kernel's flag lands in mapped pinned
    host memory, ``event`` marks the kernel's completion, ``fallback`` is the conditional full export
    that ran on the device if (and only if) the flag was raised."""
    __slots__ = ("event", "flag_pin", "slot", "fallback", "resolved", "mismatch")

    def __init__(self, event, flag_pin, slot, fallback):
        self.event, self.flag_pin, self.slot, self.fallback = event, flag_pin, slot, fallback
        self.resolved, self.mismatch = False, False

    def resolve(self):
        if not self.resolved:
            self.event.synchronize()
            self.mismatch = bool(int(self.flag_pin[self.slot]) != 0)
            self.resolved = True
            if not self.mismatch:
                self.fallback = None
        return self.mismatch


class DeviceCSR(object):
    """CSR Hessian resident on the device: ``crow_indices`` (D+1) int32, ``col_indices`` (nnz)
    int32 sorted within each row, ``values`` (nnz) float64 -- the canonical form scipy produces
    from get_sparse_sub_hessian triplets (SparseObjectives.py:591-619).

    The index arrays belong to a ``_Pattern`` that is shared between the matrices of successive
    evaluations as long as the set of exact zeros does not change (csrc/csr.cu: refill + zero-mask
    check); they must be treated as read-only.  Accessors resolve a pending pattern check first (one
    event wait, no copy on the compute stream)."""

    def __init__(self, pattern, val, pending=None):
        self._pattern, self._val, self._pending = pattern, val, pending
        self.shape = pattern.shape

    def _resolve(self):
        pend = self._pending
        if pend is not None:
            self._pending = None
            if pend.resolve():
                # the zero pattern changed at this evaluation: the conditional full export holds the result
                self._pattern, self._val = pend.fallback
        return self._pattern

    @property
    def nnz(self):
        return self._resolve().nnz

    @property
    def crow_indices(self):
        return self._resolve().crow

    @property
    def col_indices(self):
        pat = self._resolve()
        return pat.col[:pat.nnz]

    @property
    def values(self):
        pat = self._resolve()
        return self._val[:pat.nnz]

    def to_scipy(self, cache=None):
        """Host copy as ``scipy.sparse.csr_matrix``.  ``data`` lands in a pinned host block from
        torch's caching host allocator by an asynchronous copy on the current stream (the scipy matrix
        keeps the block alive, no second host copy).  The index arrays are downloaded once per PATTERN:
        later matrices of the same pattern share the host copies (made read-only) and are assembled
        without scipy's O(nnz) validation pass, so only ``data`` -- 2/3 of the bytes -- crosses PCIe.
        (``cache`` is accepted for compatibility; the cache lives in the pattern.)"""
        import scipy.sparse
        torch = nat.require_cuda()
        pat = self._resolve()
        nnz = pat.nnz
        ent = pat.host_block(torch, nnz, self._val.dtype)
        hv = ent[0][:nnz]
        hv.copy_(self._val[:nnz], non_blocking=True)
        if pat.host_template is None:
            hc = torch.empty(nnz, dtype=torch.int32, pin_memory=True)
            hr = torch.empty(pat.crow.numel(), dtype=torch.int32, pin_memory=True)
            hc.copy_(pat.col[:nnz], non_blocking=True)
            hr.copy_(pat.crow, non_blocking=True)
            if 8 * nnz <= (1 << 30):
                # a caller that still holds the previous matrix when it asks for the next one needs TWO value
                # blocks in rotation; pinning a block costs milliseconds (8 ms for 16 MB), so the second one
                # is created now, next to the pattern download, and parked in the host allocator's cache
                ent[1] = lambda: True                # (marks this block as taken while the spare is made)
                pat.host_block(torch, nnz, self._val.dtype)
            torch.cuda.current_stream().synchronize()
            data = hv.numpy()
            ent[1] = weakref.ref(data)
            m = scipy.sparse.csr_matrix((data, hc.numpy(), hr.numpy()), shape=self.shape, copy=False)
            m.has_sorted_indices = True
            m.indices.flags.writeable = False     # shared with later matrices of the same pattern
            m.indptr.flags.writeable = False
            tmpl = dict(m.__dict__)
            tmpl.pop("data", None)
            pat.host_template = tmpl
            return m
        torch.cuda.current_stream().synchronize()
        m = scipy.sparse.csr_matrix.__new__(scipy.sparse.csr_matrix)
        m.__dict__.update(pat.host_template)
        data = hv.numpy()
        ent[1] = weakref.ref(data)
        m.data = data
        return m

    def toarray(self):
        return self.to_scipy().toarray()

    def to_torch_sparse_csr(self):
        torch = nat.require_cuda()
        return torch.sparse_csr_tensor(self.crow_indices, self.col_indices, self.values,
                                       size=self.shape)


def group_sort(groups):
    """Stable sort of group ids -> (sorted ids, permutation).  Bit-exact with
    ``numpy.argsort(kind='stable')`` for host input; device input uses torch's stable sort."""
    if is_torch(groups) and groups.is_cuda:
        import torch
        s, perm = torch.sort(groups.to(torch.int64), stable=True)
        return s, perm
    g = np.asarray(groups).astype(np.int64)
    perm = np.argsort(g, kind="stable")
    return g[perm], perm


class _DeviceGLMM(object):
    """What ``LogisticGLMM`` and ``PoissonGLMM`` share: the staging of the data, the variational parameters, the
    device handle and every call that reads only the per-row weights of an evaluation (value, gradient, Hessian,
    solves, LRVB covariances, weight sensitivity, IJ).  Prediction, LOO, LOGO and the third-derivative contraction
    evaluate the logistic likelihood; ``PoissonGLMM`` refuses them."""

    _lrvb_device_model = True
    family = "logistic"

    def _stage(self, X, y, groups, weights, offset, prior, num_groups, min_info, min_shape, min_rate, name):
        """Checks the shapes, sorts the rows by group (``self.perm``; y, weights and offset follow X), puts the data
        on the device 16-byte aligned and builds the parameter dictionary, the prior and the bounds."""
        torch = nat.require_cuda()
        self.prior = prior or GLMMPrior()

        Xs = X.shape
        if len(Xs) != 2:
            raise ValueError("X must be (N, K)")
        N, K = int(Xs[0]), int(Xs[1])
        for nm, v in ((("y", y), ("groups", groups)) + ((("weights", weights),) if weights is not None else ())
                      + ((("offset", offset),) if offset is not None else ())):
            if int(np.prod(v.shape)) != N:
                raise ValueError("Wrong size for {}.  Expected {}, got {}".format(
                    nm, N, int(np.prod(v.shape))))

        g_sorted, perm = self._sorted_groups(groups)
        self.perm = perm
        self.X = to_device(X)
        self.y = to_device(y).reshape(-1)
        self.w = None if weights is None else to_device(weights).reshape(-1)
        self.offset = None if offset is None else to_device(offset).reshape(-1)
        if perm is not None:
            pd = to_device(perm, torch.int64)
            self.X = self.X.index_select(0, pd).contiguous()
            self.y = self.y.index_select(0, pd).contiguous()
            if self.w is not None:
                self.w = self.w.index_select(0, pd).contiguous()
            if self.offset is not None:
                self.offset = self.offset.index_select(0, pd).contiguous()
        self.g = to_device(g_sorted, torch.int32).reshape(-1)
        for nm in ("X", "y", "w", "offset", "g"):   # views into larger buffers: the library needs 16-B alignment
            t = getattr(self, nm)
            if t is not None and t.numel() and t.data_ptr() % 16:
                setattr(self, nm, t.clone())
        if num_groups is None:
            num_groups = int(self.g.max().item()) + 1 if N > 0 else 0
        self.N, self.K, self.G = N, K, int(num_groups)
        self.Dg = 4 + 2 * K
        self.D = self.Dg + 2 * self.G

        # variational parameters; push order = flat layout (ParameterDictionary.py:39-46)
        self.glmm_par = ModelParamsDict(name)
        self.glmm_par.push_param(UVNParam("mu", min_info=min_info))
        self.glmm_par.push_param(GammaParam("tau", min_shape=min_shape, min_rate=min_rate))
        self.glmm_par.push_param(UVNParamVector("beta", K, min_info=min_info))
        self.glmm_par.push_param(UVNParamVector("u", self.G, min_info=min_info))
        assert self.glmm_par.free_size() == self.D

        self._prior_c = nat.Prior(self.prior.mu_mean, self.prior.mu_info, self.prior.beta_mean,
                                  self.prior.beta_info, self.prior.tau_shape, self.prior.tau_rate)
        self._bounds_c = nat.Bounds(min_info, min_shape, min_rate, min_info, min_info)
        self.lower_bounds = dict(mu_info=min_info, tau_shape=min_shape, tau_rate=min_rate,
                                 beta_info=min_info, u_info=min_info)

    def _bind(self, h, lib):
        """Takes ownership of the created handle ``h`` and sets up the views and staging buffers of its results."""
        torch = nat.require_cuda()
        self._h = h
        self._lib = lib
        dev = self.X.device
        # views of the handle's own result buffers: an evaluation writes there directly
        og, gl = ctypes.c_void_p(), ctypes.c_void_p()
        nat.check(lib.lrvb_glmm_result_buffers(h, ctypes.byref(og), ctypes.byref(gl)))
        self._out_global = _view(og.value, (1 + self.Dg + self.Dg * self.Dg,), self)
        self._grad_local = _view(gl.value, (2 * self.G,), self)
        self._x_dev = torch.zeros(self.D, dtype=torch.float64, device=dev)
        self._x_pin = torch.zeros(self.D, dtype=torch.float64).pin_memory()
        self._x_event = None
        self._g_pin = None
        self._cache = dict(x=None, order=-1, coords=None)
        self._eval_id = 0                 # bumped by every evaluation: keys the host copies below
        self._host = dict(id=-1)          # KL / gradient of evaluation `id` already on the host
        self._kl_pin = None
        self._csr_pattern = None          # _Pattern of the last full export (shared by refilled matrices)
        self._csr_pending = None          # refill whose pattern check has not been read yet
        self._csr_flag_pin, self._csr_slot = None, 0
        self._csr_flag_dev, self._csr_fallback = None, None
        self._csr_refill_min = 400000     # structural nnz below which a full export is cheaper than a refill
        self._D_in = self.D
        self._coords = "free"
        self.device = dev

    # ---------------------------------------------------------------------------------------
    @staticmethod
    def _sorted_groups(groups):
        if is_torch(groups):
            import torch
            gl = groups.reshape(-1).to(torch.int64)
            if gl.numel() < 2 or bool((gl[1:] >= gl[:-1]).all()):
                return gl, None
            return group_sort(gl)
        g = np.asarray(groups).reshape(-1)
        if not np.issubdtype(g.dtype, np.integer):
            gi = g.astype(np.int64)
            if not np.array_equal(gi, g):
                raise ValueError("group ids must be integers")
            g = gi
        if g.size < 2 or np.all(g[1:] >= g[:-1]):
            return g.astype(np.int64), None
        return group_sort(g)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.lrvb_glmm_destroy(h)
            except Exception:
                pass
            self._h = None

    # ---- evaluation -------------------------------------------------------------------------
    def set_shard(self, g0, G_total):
        """This model is the shard [g0, g0 + G) of a job with ``G_total`` groups: ``evaluate``
        then takes the job's FULL flat vector and the device gathers its own entries
        (lrvb_glmm_set_shard); results stay in the local layout.  ``G_total = 0`` undoes it."""
        nat.check(self._lib.lrvb_glmm_set_shard(self._h, int(g0), int(G_total)))
        self._D_in = self.D if not G_total else self.Dg + 2 * int(G_total)
        if self._D_in != self._x_dev.numel():
            torch = nat.require_cuda()
            self._x_dev = torch.zeros(self._D_in, dtype=torch.float64, device=self.device)
            self._x_pin = torch.zeros(self._D_in, dtype=torch.float64).pin_memory()
        self.invalidate()

    def _stage_x(self, x):
        """Evaluation point -> device tensor the kernels read: a contiguous fp64 CUDA tensor is
        used where it is (kept alive until the next evaluation), anything else goes through the
        staging buffer (pinned for host input)."""
        torch = nat.require_cuda()
        if is_torch(x):
            if x.numel() != self._D_in:
                raise ValueError("Wrong size for parameter {}.  Expected {}, got {}".format(
                    self.glmm_par.name, self._D_in, x.numel()))
            xd = x.detach()
            if xd.is_cuda and xd.dtype == torch.float64 and xd.is_contiguous() and xd.device == self.device:
                return xd
            self._x_dev.copy_(xd.reshape(-1))
            return self._x_dev
        xa = np.asarray(x, dtype=np.float64).reshape(-1)
        if xa.size != self._D_in:
            raise ValueError("Wrong size for parameter {}.  Expected {}, got {}".format(
                self.glmm_par.name, self._D_in, xa.size))
        if self._x_event is not None:
            self._x_event.synchronize()  # the previous async copy has left the pinned buffer
        self._x_pin.numpy()[:] = xa
        self._x_dev.copy_(self._x_pin, non_blocking=True)
        self._x_event = torch.cuda.Event()
        self._x_event.record()
        return self._x_dev

    def _same_point(self, x, coords):
        c = self._cache
        return c["x"] is not None and c["coords"] == coords and c["x"].matches(x)

    def evaluate(self, x, order, coords="free", force=False):
        """Runs the fused evaluation of ``order`` (0 value, 1 +gradient, 2 +Hessian blocks) at
        ``x`` unless the cached evaluation already covers it."""
        if coords not in ("free", "vector"):
            raise ValueError("coords must be 'free' or 'vector'")
        if not force and self._cache["order"] >= order and self._same_point(x, coords):
            return
        if coords != self._coords:
            nat.check(self._lib.lrvb_glmm_set_coords(self._h, 1 if coords == "vector" else 0))
            self._coords = coords
        xd = self._stage_x(x)
        nat.check(self._lib.lrvb_glmm_eval(self._h, nat.ptr(xd), int(order), None, None,
                                           nat.stream_ptr()))
        self._cache = dict(x=PointKey(x), order=int(order), coords=coords)
        self._eval_id += 1

    def invalidate(self):
        self._cache = dict(x=None, order=-1, coords=None)
        self._eval_id += 1

    # raw device results of the last evaluation
    def kl_tensor(self):
        return self._out_global[0]

    def _enqueue_host_copies(self):
        """Asynchronous copies of KL and the gradient of the current evaluation into pinned host memory
        on the current stream (no synchronisation): whoever synchronises next -- typically the download of
        the Hessian values -- makes them readable, so ``fun_free_hessian`` + ``fun_free_grad`` + ``fun_free``
        at one point cost ONE stream synchronisation instead of three."""
        torch = nat.require_cuda()
        if self._g_pin is None:
            self._g_pin = torch.empty(self.D, dtype=torch.float64).pin_memory()
            self._kl_pin = torch.empty(1, dtype=torch.float64).pin_memory()
        self._kl_pin.copy_(self._out_global[0:1], non_blocking=True)
        if self._cache["order"] >= 1:
            self._g_pin[:self.Dg].copy_(self._out_global[1:1 + self.Dg], non_blocking=True)
            self._g_pin[self.Dg:].copy_(self._grad_local, non_blocking=True)
        self._host = dict(id=self._eval_id, order=self._cache["order"], pending=True)

    def kl_host(self):
        """KL of the last evaluation as a Python float."""
        torch = nat.require_cuda()
        if self._host.get("id") != self._eval_id:
            self._enqueue_host_copies()
        if self._host.get("pending"):
            torch.cuda.current_stream().synchronize()
            self._host["pending"] = False
        return float(self._kl_pin[0])

    def grad_tensor(self):
        import torch
        return torch.cat([self._out_global[1:1 + self.Dg], self._grad_local])

    def grad_host(self):
        """Gradient of the last evaluation as a fresh numpy array (pinned staging buffer, at most one
        synchronisation; none if an earlier host read of this evaluation already synchronised)."""
        torch = nat.require_cuda()
        if self._host.get("id") != self._eval_id or self._host.get("order", -1) < 1:
            self._enqueue_host_copies()
        if self._host.get("pending"):
            torch.cuda.current_stream().synchronize()
            self._host["pending"] = False
        return self._g_pin.numpy().copy()

    def blocks(self):
        """(A (Dg,Dg), B (G,2,Dg), L (G,3)) views of the cached Hessian (free or vector
        coordinates, whichever was evaluated)."""
        a, b, l = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        nat.check(self._lib.lrvb_glmm_blocks(self._h, ctypes.byref(a), ctypes.byref(b),
                                             ctypes.byref(l)))
        return (_view(a.value, (self.Dg, self.Dg), self), _view(b.value, (self.G, 2, self.Dg), self),
                _view(l.value, (self.G, 3), self))

    def obs_weights(self):
        """(5, N) per-observation derivative weights of the last evaluation (sorted order)."""
        w, ld = ctypes.c_void_p(), ctypes.c_int64()
        nat.check(self._lib.lrvb_glmm_obs_weights(self._h, ctypes.byref(w), ctypes.byref(ld)))
        return _view(w.value, (5, ld.value), self)[:, :self.N]

    def max_abs_diagonal(self):
        """Largest |H_ii| of the cached Hessian (one small device reduction)."""
        A, _, L = self.blocks()
        m = A.diagonal().abs().max()
        if self.G > 0:
            m = max(m, L[:, 0].abs().max(), L[:, 2].abs().max())
        return float(m)

    def add_diagonal_(self, lam):
        """H <- H + lam I on the CACHED blocks (Levenberg damping of the device Newton iteration);
        the next evaluation overwrites them."""
        A, _, L = self.blocks()
        A.diagonal().add_(float(lam))
        if self.G > 0:
            L[:, 0].add_(float(lam))
            L[:, 2].add_(float(lam))

    def set_global_block(self, A):
        nat.check(self._lib.lrvb_glmm_set_global_block(self._h, nat.ptr(A), nat.stream_ptr()))

    def _export_full(self, run_if=None, bufs=None):
        """Full CSR export -> (_Pattern, values); with ``run_if`` (device int32) the export runs on the
        device only if the flag is set (lrvb_glmm_hessian_csr_if).  ``bufs``: (crow, col, val, nnz) to
        write into instead of fresh tensors."""
        torch = nat.require_cuda()
        cap = ctypes.c_int64()
        nat.check(self._lib.lrvb_glmm_hessian_csr_capacity(self._h, ctypes.byref(cap)))
        if bufs is None:
            bufs = (torch.empty(self.D + 1, dtype=torch.int32, device=self.device),
                    torch.empty(cap.value, dtype=torch.int32, device=self.device),
                    torch.empty(cap.value, dtype=torch.float64, device=self.device),
                    torch.empty((), dtype=torch.int64, device=self.device))
        crow, col, val, nnz = bufs
        if run_if is None:
            nat.check(self._lib.lrvb_glmm_hessian_csr(self._h, nat.ptr(crow), nat.ptr(col), nat.ptr(val),
                                                      cap.value, nat.ptr(nnz), nat.stream_ptr()))
        else:
            nat.check(self._lib.lrvb_glmm_hessian_csr_if(self._h, nat.ptr(run_if), nat.ptr(crow), nat.ptr(col),
                                                         nat.ptr(val), cap.value, nat.ptr(nnz), nat.stream_ptr()))
        return _Pattern(crow, col, nnz, (self.D, self.D)), val

    def hessian_csr(self):
        """Device CSR of the cached Hessian.  The first call exports the pattern; later calls rewrite the
        values alone for that pattern in one pass (csrc/csr.cu refill) while the device checks that the
        set of exact zeros is unchanged -- if it is not, a conditional full export that was enqueued
        behind the refill has produced the new pattern, which the returned object (and the next call)
        adopt.  Nothing here synchronises the compute stream."""
        torch = nat.require_cuda()
        pend = self._csr_pending
        if pend is not None:
            # the previous refill's verdict (its kernel finished long ago: an event wait, no stream copy)
            self._csr_pending = None
            if pend.resolve():
                self._csr_pattern = pend.fallback[0]
                self._csr_fallback = None            # consumed: they now ARE the pattern / a result
                self._csr_flag_dev.zero_()           # stream-ordered before the next refill
        pat = self._csr_pattern
        # small problems are launch-bound: the four launches of a full export are cheaper than the refill
        # plus its conditional fallback (and the host-side bookkeeping of the pending check)
        small = self.Dg * self.Dg + 4 * self.Dg * self.G < self._csr_refill_min
        if pat is None or small:
            pat, val = self._export_full()
            self._csr_pattern = pat
            return DeviceCSR(pat, val)
        if self._csr_flag_pin is None:
            self._csr_flag_pin = torch.zeros(8, dtype=torch.int32).pin_memory()
            self._csr_flag_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
            self._csr_slot = 0
        slot = self._csr_slot = (self._csr_slot + 1) % 8
        self._csr_flag_pin[slot] = 0
        flag = self._csr_flag_dev         # stays 0 until a mismatch; reset when that mismatch is resolved
        val = torch.empty(pat.nnz, dtype=torch.float64, device=self.device)
        host_ptr = ctypes.c_void_p(self._csr_flag_pin.data_ptr() + 4 * slot)
        nat.check(self._lib.lrvb_glmm_hessian_csr_refill(self._h, nat.ptr(pat.crow), nat.ptr(val), nat.ptr(flag),
                                                         host_ptr, nat.stream_ptr()))
        ev = torch.cuda.Event()
        ev.record()
        # the conditional full export writes into buffers that are kept from call to call (they are touched
        # only if the pattern changed, in which case they leave with the result and new ones are made)
        if self._csr_fallback is None:
            cap = ctypes.c_int64()
            nat.check(self._lib.lrvb_glmm_hessian_csr_capacity(self._h, ctypes.byref(cap)))
            self._csr_fallback = (torch.empty(self.D + 1, dtype=torch.int32, device=self.device),
                                  torch.empty(cap.value, dtype=torch.int32, device=self.device),
                                  torch.empty(cap.value, dtype=torch.float64, device=self.device),
                                  torch.empty((), dtype=torch.int64, device=self.device))
        fallback = self._export_full(run_if=flag, bufs=self._csr_fallback)
        pend = _PendingRefill(ev, self._csr_flag_pin, slot, fallback)
        self._csr_pending = pend
        return DeviceCSR(pat, val, pend)

    def hessian_scipy(self):
        """Host ``scipy.sparse.csr_matrix`` of the cached Hessian (what ``Objective.fun_free_hessian``
        returns for numpy input, SparseObjectives.py:156-158); re-uses the cached pattern."""
        csr = self.hessian_csr()
        self._enqueue_host_copies()           # KL and gradient ride on the same synchronisation
        m = csr.to_scipy()
        self._host["pending"] = False
        return m

    def hvp_cached(self, v_dev, out=None, include_A=True):
        """H v with the cached Hessian; v_dev a CUDA fp64 tensor (D,)."""
        torch = nat.require_cuda()
        if v_dev.numel() != self.D:
            raise ValueError("Wrong size for HVP vector.  Expected {}, got {}".format(
                self.D, v_dev.numel()))
        if out is None:
            out = torch.empty(self.D, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_hvp(self._h, nat.ptr(v_dev), nat.ptr(out),
                                          1 if include_A else 0, nat.stream_ptr()))
        return out

    # ---- cross-Hessian with the observation weights (csrc/sensitivity.cu) ------------------
    def weight_cross_matvec(self, dw):
        """C dw (D,), C = d^2 KL / d free d w (column n = -grad_free l_n), at the point and in the
        coordinates of the last evaluation; ``dw`` (N,) in the caller's observation order."""
        torch = nat.require_cuda()
        d = to_device(dw).reshape(-1)
        if d.numel() != self.N:
            raise ValueError("Wrong size for weights.  Expected {}, got {}".format(self.N, d.numel()))
        if self.perm is not None:
            d = d.index_select(0, to_device(self.perm, torch.int64))
        d = d.contiguous()
        if d.numel() and d.data_ptr() % 16:
            d = d.clone()
        out = torch.empty(self.D, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_weight_cross_matvec(self._h, nat.ptr(d), nat.ptr(out),
                                                          nat.stream_ptr()))
        return out

    def weight_cross_rmatvec(self, v):
        """C^T v (N,) in the caller's observation order: minus the directional derivative of every
        observation's log-likelihood term along ``v`` (D,)."""
        torch = nat.require_cuda()
        vd = to_device(v).reshape(-1).contiguous()
        if vd.numel() != self.D:
            raise ValueError("Wrong size for parameter {}.  Expected {}, got {}".format(
                self.glmm_par.name, self.D, vd.numel()))
        out = torch.empty(self.N, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_weight_cross_rmatvec(self._h, nat.ptr(vd), nat.ptr(out),
                                                           nat.stream_ptr()))
        if self.perm is not None:
            res = torch.empty_like(out)
            res.index_copy_(0, to_device(self.perm, torch.int64), out)
            return res
        return out

    def third_derivative_contraction(self, a):
        """(t (D,), q (N,)) at the point and in the free coordinates of the last evaluation: t = D^3 KL[a, a, .], the
        derivative of a^T H a, and q_n = a^T (grad^2 l_n) a, the unweighted quadratic form of every row's
        log-likelihood term (caller's row order); CUDA tensors.  One pass over the rows plus one over the groups
        (csrc/amip.cu).  With a = H^-1 c, d (c^T H^-1 c) / d w_n = q_n + (C^T H^-1 t)_n (``weight_cross_rmatvec``)."""
        torch = nat.require_cuda()
        ad = to_device(a).reshape(-1).contiguous()
        if ad.numel() != self.D:
            raise ValueError("Wrong size for parameter {}.  Expected {}, got {}".format(
                self.glmm_par.name, self.D, ad.numel()))
        t = torch.empty(self.D, dtype=torch.float64, device=self.device)
        q = torch.empty(self.N, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_third_contract(self._h, nat.ptr(ad), nat.ptr(t), nat.ptr(q), nat.stream_ptr()))
        if self.perm is not None:
            res = torch.empty_like(q)
            res.index_copy_(0, to_device(self.perm, torch.int64), q)
            q = res
        return t, q

    # names shared with distributed.ShardedLogisticGLMM (where they add the all-reduce)
    def hvp(self, v):
        return self.hvp_cached(to_device(v).reshape(-1))

    def cg(self, b, x0=None, precond=0, rtol=1e-8, maxiter=0):
        return self.cg_cached(to_device(b).reshape(-1),
                              None if x0 is None else to_device(x0).reshape(-1),
                              precond, rtol, maxiter)

    def global_covariance(self):
        """(H^-1)_gg = S^-1: the linear-response covariance of the global free parameters."""
        return self.spd_inverse_(self.schur_cached(include_A=True))

    def solve(self, b_dev):
        """x = H^-1 b (b (D,) or (nrhs, D)) by block elimination with the cached Hessian."""
        b_dev = to_device(b_dev)
        Sinv = self.global_covariance()
        rhs = self.solve_reduce_rhs(b_dev, include_bg=True)
        return self.solve_finish(Sinv, rhs, b_dev)

    def make_preconditioner(self, M):
        """The `M=` of scipy.sparse.linalg.cg (ConjugateGradient.py:84) as a device descriptor.
        M: None / 0; 'block_jacobi' / 1; 'schur' (M = H^-1 applied exactly through the Schur
        complement of the local blocks); a scipy sparse matrix, a (D, D) numpy array or a torch
        tensor (M r by device SpMV / GEMV).  Returns (nat.CGPrecond, keep-alive tuple)."""
        import scipy.sparse
        torch = nat.require_cuda()
        d = nat.CGPrecond()
        keep = ()
        if M is None or (isinstance(M, int) and M == 0):
            d.kind = nat.PRECOND_NONE
        elif (isinstance(M, str) and M == "block_jacobi") or (isinstance(M, int) and M == 1):
            d.kind = nat.PRECOND_BLOCK_JACOBI
        elif isinstance(M, str) and M == "schur":
            sinv = self.global_covariance()
            d.kind, d.Sinv_dev, keep = nat.PRECOND_SCHUR, sinv.data_ptr(), (sinv,)
        elif scipy.sparse.issparse(M):
            m = scipy.sparse.csr_matrix(M)
            if m.shape != (self.D, self.D):
                raise ValueError("Wrong shape for the preconditioner.  Expected {}, got {}".format(
                    (self.D, self.D), m.shape))
            m.sort_indices()
            ip = to_device(m.indptr.astype(np.int32), torch.int32)
            ix = to_device(m.indices.astype(np.int32), torch.int32)
            dv = to_device(m.data.astype(np.float64))
            d.kind, d.indptr_dev, d.indices_dev, d.data_dev = (nat.PRECOND_CSR, ip.data_ptr(),
                                                               ix.data_ptr(), dv.data_ptr())
            keep = (ip, ix, dv)
        elif is_torch(M) or isinstance(M, np.ndarray):
            m = to_device(M)
            if tuple(m.shape) != (self.D, self.D):
                raise ValueError("Wrong shape for the preconditioner.  Expected {}, got {}".format(
                    (self.D, self.D), tuple(m.shape)))
            d.kind, d.dense_dev, keep = nat.PRECOND_DENSE, m.data_ptr(), (m,)
        else:
            raise ValueError("device CG takes preconditioner None, 'block_jacobi', 'schur', a scipy sparse "
                             "matrix, a numpy array or a torch tensor; got %r (a Python operator cannot run "
                             "inside the device iteration)" % (M,))
        return d, keep

    def cg_cached(self, b_dev, x0_dev=None, precond=0, rtol=1e-8, maxiter=0):
        """scipy-cg-compatible solve with the cached Hessian -> (x_dev, info, iters)."""
        torch = nat.require_cuda()
        x = torch.empty(self.D, dtype=torch.float64, device=self.device)
        info, iters = ctypes.c_int32(), ctypes.c_int32()
        desc, keep = self.make_preconditioner(precond)
        nat.check(self._lib.lrvb_glmm_cg_m(self._h, nat.ptr(b_dev), nat.ptr(x0_dev), ctypes.byref(desc),
                                           float(rtol), int(maxiter), nat.ptr(x), ctypes.byref(info),
                                           ctypes.byref(iters), nat.stream_ptr()))
        del keep
        return x, info.value, iters.value

    def schur_cached(self, include_A=True):
        """S = [A] - sum_g B_g^T L_g^-1 B_g  (Dg,Dg)."""
        torch = nat.require_cuda()
        S = torch.empty(self.Dg, self.Dg, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_schur(self._h, nat.ptr(S), 1 if include_A else 0,
                                            nat.stream_ptr()))
        return S

    @staticmethod
    def spd_inverse_(S):
        """In-place inverse of an SPD device matrix; raises if not positive definite."""
        info = ctypes.c_int32()
        nat.check(nat.load().lrvb_spd_inverse(nat.ptr(S), S.shape[0], ctypes.byref(info),
                                              nat.stream_ptr()))
        if info.value != 0:
            raise np.linalg.LinAlgError(
                "matrix not positive definite (pivot {})".format(info.value))
        return S

    def solve_reduce_rhs(self, b_dev, include_bg=True):
        torch = nat.require_cuda()
        b2 = b_dev.reshape(-1, self.D)
        rhs = torch.empty(b2.shape[0], self.Dg, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_solve_reduce_rhs(self._h, nat.ptr(b2), b2.shape[0],
                                                       nat.ptr(rhs), 1 if include_bg else 0,
                                                       nat.stream_ptr()))
        return rhs

    def solve_finish(self, Sinv, rhs_g, b_dev):
        torch = nat.require_cuda()
        b2 = b_dev.reshape(-1, self.D)
        x = torch.empty_like(b2)
        nat.check(self._lib.lrvb_glmm_solve_finish(self._h, nat.ptr(Sinv), nat.ptr(rhs_g),
                                                   nat.ptr(b2), b2.shape[0], nat.ptr(x),
                                                   nat.stream_ptr()))
        return x.reshape(b_dev.shape)

    def local_cov(self, Sinv):
        torch = nat.require_cuda()
        cov = torch.empty(self.G, 3, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_local_cov(self._h, nat.ptr(Sinv), nat.ptr(cov),
                                                nat.stream_ptr()))
        return cov

    # ---- prediction on new rows (csrc/predict.cu) --------------------------------------------
    def _check_prediction_rows(self, X_new, groups_new):
        """Checks new rows on the host -> (g (M,) int64, numpy or torch as given, M)."""
        if len(X_new.shape) != 2 or int(X_new.shape[1]) != self.K:
            raise ValueError("X_new must be (M, K) with K = {}, got shape {}".format(self.K, tuple(X_new.shape)))
        M = int(X_new.shape[0])
        if is_torch(groups_new):
            import torch
            g = groups_new.reshape(-1)
            if g.dtype.is_floating_point or g.dtype.is_complex or g.dtype == torch.bool:
                raise ValueError("group ids must be integers, got dtype {}".format(g.dtype))
            g = g.to(torch.int64)
            lo, hi = (int(g.min()), int(g.max())) if g.numel() else (0, 0)
        else:
            g = np.asarray(groups_new).reshape(-1)
            if not np.issubdtype(g.dtype, np.integer):
                if not np.issubdtype(g.dtype, np.floating) or not np.all(np.floor(g) == g):
                    raise ValueError("group ids must be integers")
            g = g.astype(np.int64)
            lo, hi = (int(g.min()), int(g.max())) if g.size else (0, 0)
        if int(np.prod(g.shape)) != M:
            raise ValueError("Wrong size for groups_new.  Expected {}, got {}".format(M, int(np.prod(g.shape))))
        if lo < -1 or hi >= self.G:
            raise ValueError("group ids must lie in [-1, {}) (-1: population level), got [{}, {}]".format(
                self.G, lo, hi))
        return g, M

    def _prediction_rows(self, X_new, groups_new):
        """Checks new rows before any kernel runs -> (X (M,K) fp64 CUDA, g (M,) int32 CUDA, M)."""
        torch = nat.require_cuda()
        g, M = self._check_prediction_rows(X_new, groups_new)
        X = to_device(X_new)
        if X.numel() and X.data_ptr() % 16:
            X = X.clone()
        return X, to_device(g, torch.int32), M

    def _prediction_result(self, out, nfields, like):
        f = [like_input(out[i], *like) for i in range(nfields)]
        return Prediction(*(f + [None] * (6 - nfields)))

    def predict(self, free, X_new, groups_new):
        """Predictions for new rows ``X_new`` (M, K) in groups ``groups_new`` (M,), integer ids in [-1, G)
        (-1: population level, the random effect at its mean mu -- lme4's ``re.form = NA``), at the free
        point ``free`` (read directly: no pass over the training rows): a ``Prediction`` with eta_mean, eta_var_mfvb, prob, prob_var_mfvb in the caller's row
        order (numpy for numpy input, CUDA tensors for CUDA tensor input); the LR fields are None."""
        torch = nat.require_cuda()
        X, g, M = self._prediction_rows(X_new, groups_new)
        f = to_device(free).reshape(-1)
        if f.numel() != self.D:
            raise ValueError("Wrong size for parameter {}.  Expected {}, got {}".format(
                self.glmm_par.name, self.D, f.numel()))
        out = torch.empty(4, M, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_predict(self._h, nat.ptr(f), nat.ptr(X), self.K, nat.ptr(g), None, M, nat.ptr(out),
                                              nat.stream_ptr()))
        return self._prediction_result(out, 4, (X_new, groups_new))

    def prediction_cross(self, Sinv):
        """(G, 2, 2K) block of H^-1 between beta and every group's (u.mean_g, u.info_g), at the cached Hessian."""
        torch = nat.require_cuda()
        cross = torch.empty(self.G, 2, 2 * self.K, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_predict_cross(self._h, nat.ptr(Sinv), nat.ptr(cross), nat.stream_ptr()))
        return cross

    def predict_lr(self, Sinv, cross, local_cov, X_new, groups_new):
        """``predict`` plus the LRVB variances at the cached Hessian from its arrowhead pieces: S^-1
        (``global_covariance``), ``prediction_cross`` and ``local_cov``.  The rows are visited group by
        group (a stable sort of the ids, no copy of X) so that each group's blocks are read from cache."""
        torch = nat.require_cuda()
        X, g, M = self._prediction_rows(X_new, groups_new)
        order = None
        if M > 1:
            _, perm = group_sort(g)
            order = perm.to(torch.int64).contiguous()
        out = torch.empty(6, M, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_predict_lr(self._h, nat.ptr(Sinv), nat.ptr(cross), nat.ptr(local_cov),
                                                 nat.ptr(X), self.K, nat.ptr(g), nat.ptr(order), M, nat.ptr(out),
                                                 nat.stream_ptr()))
        return self._prediction_result(out, 6, (X_new, groups_new))

    def _check_binary_y(self):
        """Raises ValueError unless every training y is 0 or 1 (checked once: y is fixed with the model)."""
        if not getattr(self, "_y_binary", False):
            if self.N and bool(((self.y != 0) & (self.y != 1)).any()):
                raise ValueError("approximate LOO needs a binary training y (0 or 1): a logistic GLMM has no "
                                 "predictive density for other values")
            self._y_binary = True

    def approximate_loo(self, Sinv, cross, local_cov):
        """Approximate leave-one-out cross-validation of the training rows by the infinitesimal jackknife at the
        cached Hessian (normally the optimum), from the arrowhead pieces of ``predict_lr``: S^-1
        (``global_covariance``), ``prediction_cross`` and ``local_cov``.  Dropping row n is the weight change
        w_n -> 0; its first-order effect on the row's moments is (dz_m, dz_v) = -Q_n (w_n l_m, w_n l_v) with
        Q_n = [j_m; j_v] H^-1 [j_m; j_v]^T, one device pass over the rows (csrc/predict.cu).  Returns an
        ``ApproximateLOO`` with CUDA tensors in the caller's row order and Python scalars."""
        torch = nat.require_cuda()
        self._check_binary_y()
        out = torch.empty(4, self.N, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_loo(self._h, nat.ptr(Sinv), nat.ptr(cross), nat.ptr(local_cov), nat.ptr(out),
                                          nat.stream_ptr()))
        if self.perm is not None:
            res = torch.empty_like(out)
            res.index_copy_(1, to_device(self.perm, torch.int64), out)
            out = res
        lpd, lpd_loo = out[0], out[1]
        n_invalid = int(torch.isnan(out[3]).sum())
        elpd = float(lpd_loo.sum())
        se = float(lpd_loo.std(correction=1)) * np.sqrt(self.N) if self.N > 1 else float("nan")
        return ApproximateLOO(lpd, lpd_loo, out[2], out[3], elpd, se, float(lpd.sum()) - elpd, n_invalid)

    def approximate_logo(self, Sinv):
        """Approximate leave-one-group-out cross-validation and group influence by the infinitesimal jackknife at the
        cached Hessian (normally the optimum), given S^-1 (``global_covariance``).  Dropping group g is w_n -> 0 on
        its rows; the globals move by delta_g = -S^-1 (v_glob - B_g^T L_g^-1 v_loc) (v = the group's data gradient),
        all groups in three device passes (csrc/logo.cu).  Returns an ``ApproximateLOGO`` with CUDA tensors (rows in
        the caller's order) and Python scalars."""
        torch = nat.require_cuda()
        self._check_binary_y()
        Pinv = self.spd_inverse_(Sinv[4:4 + self.K, 4:4 + self.K].clone())
        delta = torch.empty(self.G, self.Dg, dtype=torch.float64, device=self.device)
        grp = torch.empty(2, self.G, dtype=torch.float64, device=self.device)
        out = torch.empty(3, self.N, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_logo(self._h, nat.ptr(Sinv), nat.ptr(Pinv), nat.ptr(delta), nat.ptr(grp),
                                           nat.ptr(out), nat.stream_ptr()))
        if self.perm is not None:
            res = torch.empty_like(out)
            res.index_copy_(1, to_device(self.perm, torch.int64), out)
            out = res
        if getattr(self, "_group_nonempty", None) is None:
            self._group_nonempty = torch.bincount(self.g.to(torch.int64), minlength=self.G) > 0
        fold = grp[1][self._group_nonempty]
        se = float(fold.std(correction=1)) * np.sqrt(fold.numel()) if fold.numel() > 1 else float("nan")
        return ApproximateLOGO(out[0], out[1], out[2], grp[1], grp[0], delta, float(out[0].sum()), se)

    def ij_meat(self, unit):
        """The meat of the infinitesimal-jackknife bootstrap covariance of the globals at the cached Hessian (normally
        the optimum): (meat (Dg, Dg), s (Dg)) = (sum_u V_u V_u^T, sum_u V_u) over the rows (unit="row") or the groups
        (unit="group"), where S^-1 V_u = the global block of H^-1 psi_u and psi_u = the unit's weighted score, as in
        ``approximate_logo``.  The IJ covariance is S^-1 (meat - s s^T / U) S^-1 with U = the units of non-zero weight
        (``LinearResponseCovariances.get_ij_covariance``).  CUDA tensors; device passes of csrc/ij.cu."""
        torch = nat.require_cuda()
        if unit not in ("row", "group"):
            raise ValueError("unit must be 'row' or 'group', got %r" % (unit,))
        meat = torch.empty(self.Dg, self.Dg, dtype=torch.float64, device=self.device)
        s = torch.empty(self.Dg, dtype=torch.float64, device=self.device)
        nat.check(self._lib.lrvb_glmm_ij_meat(self._h, 0 if unit == "row" else 1, nat.ptr(meat), nat.ptr(s),
                                              nat.stream_ptr()))
        return meat, s

    def prediction_jacobian(self, free, X_new, groups_new, quantity="prob"):
        """d prob / d free (or d eta / d free) of new rows as scipy CSR (M, D): a x on beta.mean, b x~ on
        beta.info (x~_k = -x_k^2 (i_k - lb) / i_k^2), a on u.mean_g and b d_g on u.info_g (d_g = -(i_g - lb) /
        i_g^2; mu's columns for g = -1), with a = dp/dz_m, b = dp/dz_v (a = 1, b = 0 for eta).  Assembled on
        the host (host inputs never visit the device) with 2K + 2 entries per row: meant for small M, e.g. covariances BETWEEN rows through
        ``LinearResponseCovariances.get_lr_covariance_factors``."""
        import scipy.sparse
        if quantity not in ("prob", "eta"):
            raise ValueError("quantity must be 'prob' or 'eta'")
        g, M = self._check_prediction_rows(X_new, groups_new)
        Xh = X_new.detach().cpu().numpy() if is_torch(X_new) else X_new
        Xh = np.ascontiguousarray(Xh, dtype=np.float64)
        gh = g.cpu().numpy() if is_torch(g) else g
        f = free.detach().cpu().numpy() if is_torch(free) else np.asarray(free, dtype=np.float64)
        f = f.reshape(-1)
        if f.size != self.D:
            raise ValueError("Wrong size for parameter {}.  Expected {}, got {}".format(
                self.glmm_par.name, self.D, f.size))
        K, G, Dg, lb = self.K, self.G, self.Dg, self.lower_bounds
        pop = gh < 0
        gs = np.where(pop, 0, gh)
        beta_i = np.exp(f[4 + K:Dg]) + lb["beta_info"]
        u_m, u_i = f[Dg:Dg + G], np.exp(f[Dg + G:]) + lb["u_info"]
        mu_i = np.exp(f[1]) + lb["mu_info"]
        info = np.where(pop, mu_i, u_i[gs] if G else 1.0)
        d = -(info - np.where(pop, lb["mu_info"], lb["u_info"])) / (info * info)
        if quantity == "prob":
            z_m = np.where(pop, f[0], u_m[gs] if G else 0.0) + Xh @ f[4:4 + K]
            z_s = np.sqrt(1.0 / info + (Xh * Xh) @ (1.0 / beta_i))
            c = np.sqrt(2.0) * self.gh_x
            sg = 1.0 / (1.0 + np.exp(-(z_m[:, None] + z_s[:, None] * c[None, :])))
            dsg = (self.gh_w / np.sqrt(np.pi)) * sg * (1.0 - sg)
            a, b = dsg.sum(axis=1), (dsg * c).sum(axis=1) / (2.0 * z_s)
        else:
            a, b = np.ones(M), np.zeros(M)
        xt = -(Xh * Xh) * ((beta_i - lb["beta_info"]) / (beta_i * beta_i))[None, :]
        cols = np.concatenate([np.tile(np.arange(4, Dg), (M, 1)), np.where(pop, 0, Dg + gh)[:, None],
                               np.where(pop, 1, Dg + G + gh)[:, None]], axis=1)
        vals = np.concatenate([a[:, None] * Xh, b[:, None] * xt, a[:, None], (b * d)[:, None]], axis=1)
        rows = np.repeat(np.arange(M), 2 * K + 2)
        return scipy.sparse.csr_matrix((vals.reshape(-1), (rows, cols.reshape(-1))), shape=(M, self.D))

    # ---- moments (for LinearResponseCovariances) ------------------------------------------------
    def moment_names(self):
        return (["e_mu", "e_tau"] + ["e_beta_%d" % k for k in range(self.K)]
                + ["e_u_%d" % g for g in range(self.G)])

    def moment_jacobian(self, free):
        """d [E mu, E tau, E beta (K), E u (G)] / d free as scipy CSR ((2+K+G), D).
        E tau = shape/rate (GammaParams.py:9-10) with shape = exp(f)+lb (Parameters.py:55)."""
        import scipy.sparse
        free = np.asarray(free, dtype=np.float64).reshape(-1)
        K, G, Dg = self.K, self.G, self.Dg
        a = np.exp(free[2]) + self.lower_bounds["tau_shape"]
        b = np.exp(free[3]) + self.lower_bounds["tau_rate"]
        rows = [0, 1, 1] + list(range(2, 2 + K)) + list(range(2 + K, 2 + K + G))
        cols = [0, 2, 3] + list(range(4, 4 + K)) + list(range(Dg, Dg + G))
        vals = [1.0, np.exp(free[2]) / b, -a / (b * b) * np.exp(free[3])] + [1.0] * (K + G)
        return scipy.sparse.csr_matrix((vals, (rows, cols)), (2 + K + G, self.D))


class LogisticGLMM(_DeviceGLMM):
    """Data + variational parameters + device handle of one logistic GLMM (or one shard of it).

    X (N,K) float64, y (N,) in {0,1}, groups (N,) integer ids in [0, num_groups); observations
    are stably sorted by group if they are not already (``self.perm`` records the permutation).
    ``gh_x, gh_w``: Gauss-Hermite nodes/weights (default ``hermgauss(num_gh_points)``).
    """

    def __init__(self, X, y, groups, num_gh_points=8, gh_x=None, gh_w=None, weights=None,
                 prior=None, num_groups=None, min_info=0.0, min_shape=0.0, min_rate=0.0,
                 include_global_terms=True, name="glmm_par"):
        nat.require_cuda()
        lib = nat.load()
        if gh_x is None or gh_w is None:
            gh_x, gh_w = np.polynomial.hermite.hermgauss(int(num_gh_points))
        self.gh_x = np.ascontiguousarray(np.asarray(gh_x, dtype=np.float64))
        self.gh_w = np.ascontiguousarray(np.asarray(gh_w, dtype=np.float64))
        if self.gh_x.shape != self.gh_w.shape or self.gh_x.ndim != 1:
            raise ValueError("gh_x and gh_w must be 1-d arrays of the same length")
        self._stage(X, y, groups, weights, None, prior, num_groups, min_info, min_shape, min_rate, name)
        h = ctypes.c_void_p()
        nat.check(lib.lrvb_glmm_create(
            ctypes.byref(h), self.N, self.K, self.G, self.gh_x.size, nat.ptr(self.X), nat.ptr(self.y),
            nat.ptr(self.g), nat.ptr(self.w), nat.darray(self.gh_x), nat.darray(self.gh_w),
            ctypes.byref(self._prior_c), ctypes.byref(self._bounds_c),
            1 if include_global_terms else 0, nat.stream_ptr()))
        self._bind(h, lib)


class PoissonGLMM(_DeviceGLMM):
    """Data + variational parameters + device handle of one Poisson log-link GLMM for counts (lme4's
    ``glmer(y ~ x + (1 | g) + offset(log(exposure)), family = poisson)``).

    X (N,K) float64, y (N,) counts (finite, >= 0; non-integer values are accepted), groups (N,) integer ids in
    [0, num_groups), offset (N,) or None: added to the linear predictor (log exposure).  Rows are stably sorted by
    group as in ``LogisticGLMM``.  Under q the observation term w [y m - exp(m + v/2) - lgamma(y + 1)] is exact, so
    there is no quadrature.  Evaluation, Hessian, solves, ``LinearResponseCovariances`` (except prediction, LOO, LOGO
    and AMIP), ``WeightSensitivityLinearApproximation`` and ``get_ij_covariance`` (cluster-robust standard errors for
    overdispersed counts) work as for the logistic model.
    """

    family = "poisson"

    def __init__(self, X, y, groups, offset=None, weights=None, prior=None, num_groups=None, min_info=0.0,
                 min_shape=0.0, min_rate=0.0, include_global_terms=True, name="glmm_par"):
        nat.require_cuda()
        lib = nat.load()
        self._stage(X, y, groups, weights, offset, prior, num_groups, min_info, min_shape, min_rate, name)
        h = ctypes.c_void_p()
        nat.check(lib.lrvb_glmm_create_poisson(
            ctypes.byref(h), self.N, self.K, self.G, nat.ptr(self.X), nat.ptr(self.y), nat.ptr(self.g),
            nat.ptr(self.w), nat.ptr(self.offset), ctypes.byref(self._prior_c), ctypes.byref(self._bounds_c),
            1 if include_global_terms else 0, nat.stream_ptr()))
        self._bind(h, lib)

    def _logistic_only(self, *args, **kwargs):
        raise NotImplementedError("not implemented for the Poisson family: prediction, approximate LOO / LOGO and the "
                                  "third-derivative contraction of AMIP evaluate the logistic likelihood")

    predict = predict_lr = prediction_jacobian = approximate_loo = approximate_logo = _logistic_only
    third_derivative_contraction = _check_binary_y = _logistic_only
