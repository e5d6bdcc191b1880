"""Observation-sharded GLMM across the GPUs of one box (one process per GPU, torch.distributed).

The data term is a sum over observations and every observation touches the Dg global
parameters and exactly ONE group's two local parameters, so (SURVEY.md 8e):

  * observations are stably sorted by group and cut into contiguous GROUP-ALIGNED shards balanced
    by observation count (``partition_groups``); rank r owns groups [g0_r, g1_r) and all their
    observations;
  * local gradient entries, border rows B_g, local 2x2 blocks L_g and the local slices of CG
    vectors are rank-private and are never communicated;
  * one all-reduce (sum) of the packed buffer [KL, grad_g (Dg), H_gg (Dg*Dg)] per evaluation --
    exactly ``lrvb_glmm_eval``'s ``out_global``; rank 0 alone adds the terms that depend on no
    group (priors / entropies of mu, beta, tau: ``include_global_terms``);
  * per HVP one all-reduce of (B^T v_l) (Dg doubles); per CG iteration that plus one all-reduce
    of two scalars; per Schur complement one all-reduce of S (Dg*Dg).

The reference has no distributed path at all (SURVEY.md section 2); this module is the new
repo's one parallelism strategy.  The class is written against a small "local model" interface
(the CUDA ``GLMM.LogisticGLMM``; tests drive the same algebra with an oracle-backed double over
gloo on CPU), and keeps the ``Objective`` contract: full-length free vectors in, full-length
results out, identical on every rank.
"""
import numpy as np

from ._tensors import PointKey, is_torch


def partition_groups(counts, world):
    """Group-aligned cut points balanced by observation count.

    counts: (G,) observations per group.  Returns bounds (world+1,) int64 with bounds[0] = 0,
    bounds[-1] = G; rank r owns groups [bounds[r], bounds[r+1]).  Deterministic: boundary r is
    the first group index at which the cumulative observation count reaches r*N/world (ties keep
    ranks non-empty where possible)."""
    counts = np.asarray(counts, dtype=np.int64)
    G = counts.size
    csum = np.concatenate([[0], np.cumsum(counts)])
    N = int(csum[-1])
    bounds = np.zeros(world + 1, dtype=np.int64)
    bounds[-1] = G
    for r in range(1, world):
        target = (N * r) // world
        b = int(np.searchsorted(csum, target, side="left"))
        b = min(max(b, int(bounds[r - 1])), G)
        bounds[r] = b
    # give empty trailing ranks at least one group when there are enough groups
    if G >= world:
        for r in range(1, world):
            bounds[r] = max(bounds[r], bounds[r - 1] + 1)
        for r in range(world - 1, 0, -1):
            bounds[r] = min(bounds[r], bounds[r + 1] - 1)
    return bounds


def local_index_map(Dg, g0, g1, G_total):
    """Positions, in the FULL flat layout [globals | u.mean (G_total) | u.info (G_total)], of the
    entries of a shard's local layout [globals | u.mean (g0:g1) | u.info (g0:g1)]."""
    return np.concatenate([np.arange(Dg), Dg + np.arange(g0, g1),
                           Dg + G_total + np.arange(g0, g1)]).astype(np.int64)


class PeerAllReduce(object):
    """Sum of small fp64 device buffers over the ranks through NVLink peer memory
    (csrc/p2p.cu): one kernel per rank pushes its block into a window of every peer, waits for
    theirs and adds them in rank order -- bitwise identical on all ranks, one NVLink traversal,
    in-stream behind the producer (no NCCL stream hand-over).  Collective constructor: every rank
    of ``process_group`` must call it.  ``PeerAllReduce.create`` returns None when the ranks are
    not one-process-per-GPU on one box or a window cannot be mapped; callers then use NCCL."""

    def __init__(self, handle, lib, max_elems, rank, world):
        self._h, self._lib = handle, lib
        self.max_elems, self.rank, self.world = int(max_elems), rank, world

    @classmethod
    def create(cls, max_elems, process_group=None):
        import ctypes
        import os
        import socket
        import torch
        import torch.distributed as dist
        from . import _native as nat
        if os.environ.get("LRVB_P2P_ALLREDUCE", "1") == "0" or not torch.cuda.is_available():
            return None
        if dist.get_backend(process_group) != "nccl":
            return None
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        if world < 2 or world > 16:
            return None
        lib = nat.load()
        h = ctypes.c_void_p()
        ok = lib.lrvb_p2p_create(ctypes.byref(h), rank, world, int(max_elems)) == 0
        nbytes = lib.lrvb_p2p_handle_bytes()
        blob = ctypes.create_string_buffer(nbytes)
        ok = ok and lib.lrvb_p2p_export(h, blob) == 0
        infos = [None] * world
        dist.all_gather_object(infos, (socket.gethostname(), torch.cuda.current_device(), bool(ok),
                                       bytes(blob.raw)), group=process_group)
        same_box = len({i[0] for i in infos}) == 1 and len({i[1] for i in infos}) == world
        ok = ok and same_box and all(i[2] for i in infos)
        if ok:
            ok = lib.lrvb_p2p_connect(h, b"".join(i[3] for i in infos)) == 0
        oks = [None] * world
        dist.all_gather_object(oks, bool(ok), group=process_group)   # also: every window is mapped
        if not all(oks):
            if h.value:
                lib.lrvb_p2p_destroy(h)
            return None
        return cls(h, lib, max_elems, rank, world)

    def fits(self, t):
        import torch
        # one-shot: every rank receives (world - 1) * n lines; beyond ~200k doubles in flight per
        # rank NCCL's bandwidth-oriented algorithms win (profiles/r01_peer_allreduce_latency.txt)
        return (t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()
                and t.numel() <= self.max_elems and t.numel() * (self.world - 1) <= 200000)

    def all_reduce_(self, t):
        """In-place sum over the ranks on torch's current stream."""
        from . import _native as nat
        nat.check(self._lib.lrvb_p2p_allreduce_sum(self._h, nat.ptr(t), t.numel(), nat.stream_ptr()))
        return t

    def status(self, wait=True):
        """0, or 1 + r when rank r missed the deadline (sticky; the results since are NaN and
        ``all_reduce_`` raises RuntimeError).  ``wait=False`` reads the host word without
        synchronising the stream."""
        import ctypes
        from . import _native as nat
        s = ctypes.c_int32()
        if wait:
            nat.check(self._lib.lrvb_p2p_status(self._h, ctypes.byref(s), nat.stream_ptr()))
        else:
            nat.check(self._lib.lrvb_p2p_status_nowait(self._h, ctypes.byref(s)))
        return s.value

    def set_timeout(self, seconds):
        from . import _native as nat
        nat.check(self._lib.lrvb_p2p_set_timeout(self._h, float(seconds)))

    def set_stats(self, enable=True):
        """Start (and reset) / stop the in-kernel accounting of the time spent waiting for peers."""
        from . import _native as nat
        nat.check(self._lib.lrvb_p2p_set_stats(self._h, 1 if enable else 0, nat.stream_ptr()))

    def stats(self):
        """dict(calls, wait_us_total, wait_us_max) since ``set_stats`` (synchronises)."""
        import ctypes
        from . import _native as nat
        out = (ctypes.c_double * 3)()
        nat.check(self._lib.lrvb_p2p_get_stats(self._h, out, nat.stream_ptr()))
        return dict(calls=int(out[0]), wait_us_total=float(out[1]), wait_us_max=float(out[2]))

    def close(self):
        if self._h is not None and self._h.value:
            self._lib.lrvb_p2p_destroy(self._h)
        self._h = None


class ShardedLogisticGLMM(object):
    _lrvb_device_model = True

    def __init__(self, local, g0, g1, G_total, process_group=None, min_info=0.0, min_shape=0.0,
                 min_rate=0.0, name="glmm_par"):
        import torch
        import torch.distributed as dist
        from .GammaParams import GammaParam
        from .NormalParams import UVNParam, UVNParamVector
        from .ParameterDictionary import ModelParamsDict
        self.local = local
        self.pg = process_group
        self.rank = dist.get_rank(process_group)
        self.world = dist.get_world_size(process_group)
        self.g0, self.g1, self.G = int(g0), int(g1), int(G_total)
        self.K, self.Dg = local.K, local.Dg
        self.D = self.Dg + 2 * self.G
        self.device = local.device
        self.N = local.N
        assert local.G == self.g1 - self.g0
        self._map = torch.from_numpy(local_index_map(self.Dg, g0, g1, G_total)).to(self.device)
        sizes = [None] * self.world
        dist.all_gather_object(sizes, (self.g0, self.g1), group=process_group)
        self.group_ranges = sizes
        self.glmm_par = ModelParamsDict(name)
        self.glmm_par.push_param(UVNParam("mu", min_info=min_info))
        self.glmm_par.push_param(GammaParam("tau", min_shape=min_shape, min_rate=min_rate))
        self.glmm_par.push_param(UVNParamVector("beta", self.K, min_info=min_info))
        self.glmm_par.push_param(UVNParamVector("u", self.G, min_info=min_info))
        self.lower_bounds = dict(mu_info=min_info, tau_shape=min_shape, tau_rate=min_rate,
                                 beta_info=min_info, u_info=min_info)
        self._cache = dict(x=None, order=-1, coords=None)
        self._sinv = None
        # small replicated blocks are summed through NVLink peer memory when the ranks are the GPUs
        # of one box (collective decision, identical on every rank); otherwise NCCL / gloo
        self._peer = None
        self._full_input = hasattr(local, "set_shard")
        if self._full_input:
            local.set_shard(self.g0, self.G)
        if getattr(local, "_h", None) is not None and getattr(self.device, "type", "") == "cuda":
            self._peer = PeerAllReduce.create(max(1 + self.Dg + self.Dg * self.Dg, 4096), process_group)

    # ---- construction ----------------------------------------------------------------------
    @classmethod
    def from_local_shard(cls, X, y, g_local, num_local_groups, process_group=None, **kw):
        """Every rank passes ITS shard with group ids local to the shard (0..num_local_groups)."""
        import torch.distributed as dist
        from .GLMM import LogisticGLMM
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        sizes = [None] * world
        dist.all_gather_object(sizes, int(num_local_groups), group=process_group)
        g0 = int(sum(sizes[:rank]))
        bounds_kw = {k: kw[k] for k in ("min_info", "min_shape", "min_rate") if k in kw}
        local = LogisticGLMM(X, y, g_local, num_groups=int(num_local_groups),
                             include_global_terms=(rank == 0), **kw)
        return cls(local, g0, g0 + int(num_local_groups), int(sum(sizes)), process_group,
                   **bounds_kw)

    @classmethod
    def from_full(cls, X, y, groups, num_groups, process_group=None, weights=None,
                  local_factory=None, **kw):
        """Every rank passes the FULL (host) data set; each keeps its group-aligned shard."""
        import torch.distributed as dist
        rank, world = dist.get_rank(process_group), dist.get_world_size(process_group)
        X, y = np.asarray(X, dtype=np.float64), np.asarray(y, dtype=np.float64).reshape(-1)
        g = np.asarray(groups).astype(np.int64).reshape(-1)
        order = np.argsort(g, kind="stable")
        counts = np.bincount(g, minlength=int(num_groups))
        bounds = partition_groups(counts, world)
        g0, g1 = int(bounds[rank]), int(bounds[rank + 1])
        csum = np.concatenate([[0], np.cumsum(counts)])
        sel = order[csum[g0]:csum[g1]]
        wl = None if weights is None else np.asarray(weights, dtype=np.float64).reshape(-1)[sel]
        if local_factory is None:
            from .GLMM import LogisticGLMM

            def local_factory(Xl, yl, gl, Gl, wl_, include_global, **k2):
                return LogisticGLMM(Xl, yl, gl, weights=wl_, num_groups=Gl,
                                    include_global_terms=include_global, **k2)
        local = local_factory(X[sel], y[sel], g[sel] - g0, g1 - g0, wl, rank == 0, **kw)
        bounds_kw = {k: kw[k] for k in ("min_info", "min_shape", "min_rate") if k in kw}
        return cls(local, g0, g1, int(num_groups), process_group, **bounds_kw)

    # ---- helpers -----------------------------------------------------------------------------
    def _allreduce(self, t):
        if self._peer is not None and self._peer.fits(t):
            return self._peer.all_reduce_(t)
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.pg)
        return t

    def to_local(self, v_full):
        """Full-layout vector(s) (..., D) -> this rank's local layout (..., Dg + 2 G_local)."""
        return v_full.index_select(-1, self._map).contiguous()

    def from_local(self, v_local):
        """Local-layout vector(s) (..., Dg + 2 G_local) -> full vector(s) (..., D), identical on every
        rank (globals taken as they are -- they are replicated -- locals all-gathered): ONE all_gather
        whatever the number of vectors."""
        import torch
        import torch.distributed as dist
        Dg, Gl = self.Dg, self.g1 - self.g0
        lead = tuple(v_local.shape[:-1])
        v2 = v_local.reshape(-1, Dg + 2 * Gl)
        n = v2.shape[0]
        gmax = max(b - a for a, b in self.group_ranges)
        pad = torch.zeros(n, 2, gmax, dtype=v_local.dtype, device=v_local.device)
        pad[:, 0, :Gl] = v2[:, Dg:Dg + Gl]
        pad[:, 1, :Gl] = v2[:, Dg + Gl:]
        gathered = [torch.empty_like(pad) for _ in range(self.world)]
        dist.all_gather(gathered, pad, group=self.pg)
        out = torch.empty(n, self.D, dtype=v_local.dtype, device=v_local.device)
        out[:, :Dg] = v2[:, :Dg]
        for (a, b), t in zip(self.group_ranges, gathered):
            out[:, Dg + a:Dg + b] = t[:, 0, :b - a]
            out[:, Dg + self.G + a:Dg + self.G + b] = t[:, 1, :b - a]
        return out.reshape(lead + (self.D,))

    def _dev(self, x):
        import torch
        if is_torch(x):
            return x.to(self.device, torch.float64).reshape(-1)
        return torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64))).reshape(
            -1).to(self.device)

    def _same_point(self, x, coords):
        c = self._cache
        return c["x"] is not None and c["coords"] == coords and c["x"].matches(x)

    def invalidate(self):
        self._cache = dict(x=None, order=-1, coords=None)
        self._sinv = None
        self.local.invalidate() if hasattr(self.local, "invalidate") else None

    # ---- the model interface used by Objective / ConjugateGradientSolver / LRVB --------------
    def evaluate(self, x, order, coords="free", force=False):
        if not force and self._cache["order"] >= order and self._same_point(x, coords):
            return
        n_in = x.numel() if is_torch(x) else np.asarray(x).size
        if n_in != self.D:
            raise ValueError("Wrong size for parameter {}.  Expected {}, got {}".format(
                self.glmm_par.name, self.D, n_in))
        if self._full_input:
            # the shard's kernels read their entries out of the full vector: no gather kernel
            self.local.evaluate(x, order, coords, force=True)
        else:
            self.local.evaluate(self.to_local(self._dev(x)), order, coords, force=True)
        Dg = self.Dg
        n = 1 + (Dg if order >= 1 else 0) + (Dg * Dg if order >= 2 else 0)
        buf = self.local._out_global
        self._allreduce(buf[:n])            # on the compute stream, behind the eval; `buf` is the handle's
        #                                     own buffer, so the cached global block A is reduced too
        self._sinv = None
        self._cache = dict(x=PointKey(x), order=int(order), coords=coords)

    def kl_tensor(self):
        return self.local._out_global[0]

    def grad_local_layout(self):
        import torch
        return torch.cat([self.local._out_global[1:1 + self.Dg], self.local._grad_local])

    def grad_tensor(self):
        return self.from_local(self.grad_local_layout())

    def hvp_local_layout(self, v_local):
        """H v in the local layout: rank-private local rows, all-reduced global rows."""
        out = self.local.hvp_cached(v_local, include_A=(self.rank == 0))
        self._allreduce(out[:self.Dg])
        return out

    def hvp(self, v_full):
        return self.from_local(self.hvp_local_layout(self.to_local(self._dev(v_full))))

    def hessian_csr(self):
        """This rank's part of the distributed sparse Hessian (local layout, device CSR)."""
        return self.local.hessian_csr()

    def hessian_csr_global(self):
        """Full (D, D) scipy CSR gathered on every rank (parity tests / host API only)."""
        import scipy.sparse
        import torch.distributed as dist
        loc = self.local.hessian_csr().to_scipy().tocoo()
        m = self._map.cpu().numpy()
        rows, cols, vals = m[loc.row], m[loc.col], loc.data
        if self.rank != 0:   # the global block is replicated: keep rank 0's copy only
            keep = ~((loc.row < self.Dg) & (loc.col < self.Dg))
            rows, cols, vals = rows[keep], cols[keep], vals[keep]
        pieces = [None] * self.world
        dist.all_gather_object(pieces, (rows, cols, vals), group=self.pg)
        R = np.concatenate([p[0] for p in pieces])
        C = np.concatenate([p[1] for p in pieces])
        V = np.concatenate([p[2] for p in pieces])
        H = scipy.sparse.csr_matrix((V, (R, C)), (self.D, self.D))
        H.sort_indices()
        return H

    # ---- solves ----------------------------------------------------------------------------------
    def _dot(self, a, b, extra=None):
        """Global dot product of local-layout vectors (globals counted once); ``extra`` lets a
        second pair share the same all-reduce."""
        import torch
        Dg = self.Dg
        parts = [torch.dot(a[Dg:], b[Dg:])]
        if extra is not None:
            parts.append(torch.dot(extra[0][Dg:], extra[1][Dg:]))
        t = self._allreduce(torch.stack(parts))
        res = [t[0] + torch.dot(a[:Dg], b[:Dg])]
        if extra is not None:
            res.append(t[1] + torch.dot(extra[0][:Dg], extra[1][:Dg]))
        return res

    def _precond(self, r, which):
        import torch
        if not which:
            return r.clone()
        A, _, L = self.local.blocks()
        Dg, Gl = self.Dg, self.g1 - self.g0
        z = torch.empty_like(r)
        z[:Dg] = r[:Dg] / torch.diagonal(A)
        det = L[:, 0] * L[:, 2] - L[:, 1] * L[:, 1]
        rm, ri = r[Dg:Dg + Gl], r[Dg + Gl:]
        z[Dg:Dg + Gl] = (L[:, 2] * rm - L[:, 1] * ri) / det
        z[Dg + Gl:] = (-L[:, 1] * rm + L[:, 0] * ri) / det
        return z

    def cg_local_layout(self, b, x0=None, precond=0, rtol=1e-8, maxiter=0):
        """scipy.sparse.linalg.cg's iteration (ConjugateGradient.py:81-85) on sharded vectors."""
        import torch
        if isinstance(precond, str):
            if precond != "block_jacobi":
                raise ValueError("the sharded CG takes preconditioner None or 'block_jacobi'; got %r "
                                 "(use LinearResponseCovariances(method='schur') for the exact solve)" % precond)
            precond = 1
        elif precond is None:
            precond = 0
        elif not isinstance(precond, int):
            raise ValueError("the sharded CG takes preconditioner None or 'block_jacobi'")
        if maxiter <= 0:
            maxiter = 10 * self.D
        if self._peer is not None and self.Dg + 1 <= self._peer.max_elems:
            # device-resident iteration, two peer all-reduces per step (lrvb_glmm_cg_sharded)
            import ctypes
            from . import _native as nat
            b = b.contiguous()
            x = torch.empty_like(b)
            info, iters = ctypes.c_int32(), ctypes.c_int32()
            nat.check(self.local._lib.lrvb_glmm_cg_sharded(
                self.local._h, self._peer._h, nat.ptr(b), nat.ptr(None if x0 is None else x0.contiguous()),
                int(precond), float(rtol), int(min(maxiter, 2000000000)), 1 if self.rank == 0 else 0,
                nat.ptr(x), ctypes.byref(info), ctypes.byref(iters), nat.stream_ptr()))
            return x, info.value, iters.value
        bnrm = torch.sqrt(self._dot(b, b)[0]).item()
        if bnrm == 0.0:
            return b.clone(), 0, 0
        atol = rtol * bnrm
        if x0 is None:
            x = torch.zeros_like(b)
            r = b.clone()
        else:
            x = x0.clone()
            r = b - self.hvp_local_layout(x)
        rho_prev, p = None, None
        rnorm = torch.sqrt(self._dot(r, r)[0]).item()
        for it in range(maxiter):
            if rnorm < atol:
                return x, 0, it
            z = self._precond(r, precond)
            rho = self._dot(r, z)[0]
            if it > 0:
                p = z + (rho / rho_prev) * p
            else:
                p = z.clone()
            q = self.hvp_local_layout(p)
            alpha = rho / self._dot(p, q)[0]
            x += alpha * p
            r -= alpha * q
            rho_prev = rho
            rnorm = torch.sqrt(self._dot(r, r)[0]).item()
        return x, maxiter, maxiter

    def cg(self, b_full, x0_full=None, precond=0, rtol=1e-8, maxiter=0):
        b = self.to_local(self._dev(b_full))
        x0 = None if x0_full is None else self.to_local(self._dev(x0_full))
        x, info, iters = self.cg_local_layout(b, x0, precond, rtol, maxiter)
        return self.from_local(x), info, iters

    def max_abs_diagonal(self):
        import torch
        import torch.distributed as dist
        t = torch.tensor([self.local.max_abs_diagonal()], dtype=torch.float64, device=self.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.pg)
        return float(t.item())

    def add_diagonal_(self, lam):
        # A is a replica on every rank (only rank 0's copy enters the Schur complement and the HVP)
        self.local.add_diagonal_(lam)
        self._sinv = None

    def global_covariance(self):
        """(H^-1)_gg: all-reduce of the per-rank Schur pieces, then the small SPD inverse."""
        if self._sinv is None:
            S = self.local.schur_cached(include_A=(self.rank == 0))
            self._allreduce(S)
            self._sinv = self.local.spd_inverse_(S)
        return self._sinv

    def solve(self, b_full):
        """H^-1 b for b (D,) or (nrhs, D), full layout in and out."""
        import torch
        b = self._dev(b_full).reshape(-1, self.D)
        bl = self.to_local(b)
        Sinv = self.global_covariance()
        rhs = self.local.solve_reduce_rhs(bl, include_bg=(self.rank == 0))
        self._allreduce(rhs)
        xl = self.local.solve_finish(Sinv, rhs, bl)
        out = self.from_local(xl)           # one all_gather for all right-hand sides
        shape = tuple(b_full.shape) if hasattr(b_full, "shape") else (self.D,)
        return out.reshape(shape)

    def local_cov(self, Sinv):
        """LRVB covariances of this rank's groups' (u.mean, u.info), (G_local, 3)."""
        return self.local.local_cov(Sinv)

    def _no_prediction(self, *args, **kwargs):
        raise NotImplementedError("prediction of a sharded model: build a single-GPU LogisticGLMM of the job "
                                  "and use LogisticGLMM.predict / LinearResponseCovariances.get_prediction_variances")

    predict = prediction_jacobian = _no_prediction

    def approximate_loo(self, *args, **kwargs):
        raise NotImplementedError("approximate LOO of a sharded model: build a single-GPU LogisticGLMM of the job "
                                  "and use LinearResponseCovariances.get_approximate_loo")

    def approximate_logo(self, *args, **kwargs):
        raise NotImplementedError("approximate LOGO of a sharded model: build a single-GPU LogisticGLMM of the job "
                                  "and use LinearResponseCovariances.get_approximate_logo")

    def third_derivative_contraction(self, *args, **kwargs):
        raise NotImplementedError("the third derivative of a sharded model: build a single-GPU LogisticGLMM of the job "
                                  "and use LinearResponseCovariances.get_approximate_max_influence")

    def moment_jacobian(self, free):
        import scipy.sparse
        free = np.asarray(free, dtype=np.float64).reshape(-1)
        K, G, Dg = self.K, self.G, self.Dg
        a = np.exp(free[2]) + self.lower_bounds["tau_shape"]
        b = np.exp(free[3]) + self.lower_bounds["tau_rate"]
        rows = [0, 1, 1] + list(range(2, 2 + K)) + list(range(2 + K, 2 + K + G))
        cols = [0, 2, 3] + list(range(4, 4 + K)) + list(range(Dg, Dg + G))
        vals = [1.0, np.exp(free[2]) / b, -a / (b * b) * np.exp(free[3])] + [1.0] * (K + G)
        return scipy.sparse.csr_matrix((vals, (rows, cols)), (2 + K + G, self.D))
