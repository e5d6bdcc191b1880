"""The Poisson GLMM on the device (GLMM.PoissonGLMM, lrvb_glmm_create_poisson, k_obs_pois / k_pois_influence of
csrc/pois.cuh) against the numpy oracle (oracle/poisson_oracle.py): KL, gradient, CSR Hessian and HVP in free and
vector coordinates for every Gram kernel class, Newton to the optimum with the LRVB covariances there, the weight
cross-Hessian, the IJ covariance, determinism, and the refused calls and rejected data."""
import numpy as np
import pytest
import torch

from helpers import assert_close
from oracle import glmm_oracle as go
from oracle import ij_oracle as ij
from oracle import poisson_oracle as pois

pytestmark = pytest.mark.gpu

# K <= 24: the nine k_gram_mid instantiations of the IJ lookup; 25 .. 104 k_gram_mid; 105, 130 k_gram_big; 200
# k_gram_wide; 256 the largest K (k_gram_big).  The lanes per row of k_obs_pois change at K = 9, 17, 33, 65, 129.
KS = [3, 6, 8, 11, 14, 16, 19, 22, 24, 25, 62, 63, 104, 105, 130, 200, 256]


def _case(K, N, G, seed, shuffle, ragged, empty, weights, offset, bounds):
    X, y, g, off = pois.make_poisson_data(N, K, G - empty, seed, offset=offset)
    rng = np.random.default_rng(seed + 1)
    if ragged:
        g = np.sort(rng.integers(0, G - empty, size=N)).astype(np.int64)
    if empty:
        g = np.sort(rng.choice(G, size=G - empty, replace=False))[g]
    w = None
    if weights:
        w = rng.uniform(0.5, 1.5, N)
        w[rng.choice(N, size=max(1, N // 20), replace=False)] = 0.0
    if shuffle:
        p = rng.permutation(N)
        X, y, g = X[p], y[p], g[p]
        w = None if w is None else w[p]
        off = None if off is None else off[p]
    free = go.make_free(4 + 2 * K + 2 * G, seed)
    return dict(X=X, y=y, g=g, w=w, off=off, K=K, G=G, N=N, free=free, bounds=bounds)


def _oracle(case, w=None):
    o = np.argsort(case["g"], kind="stable")
    b = case["bounds"]
    w = case["w"] if w is None else w
    return pois.PoissonOracle(case["X"][o], case["y"][o], case["g"][o],
                              offset=None if case["off"] is None else case["off"][o],
                              weights=None if w is None else w[o], G=case["G"], bounds=go.GLMMBounds(b, b, b, b, b))


def _model(vb, case):
    b = case["bounds"]
    return vb.PoissonGLMM(case["X"], case["y"], case["g"], offset=case["off"], weights=case["w"],
                          num_groups=case["G"], min_info=b, min_shape=b, min_rate=b)


def _kcase(K):
    i = KS.index(K)
    return _case(K, 1500 if K <= 64 else 12 * K + 7, 20, 4100 + K, shuffle=i % 2 == 0, ragged=i % 3 == 0,
                 empty=2 if i % 2 else 0, weights=i % 2 == 1, offset=i % 3 != 1, bounds=0.05 if i % 4 == 1 else 0.0)


@pytest.fixture(scope="module", params=KS)
def setup(request, vb):
    case = _kcase(request.param)
    model = _model(vb, case)
    return case, _oracle(case), model, vb.Objective(model.glmm_par, model)


def test_value_gradient_hessian_hvp(setup):
    case, oracle, model, obj = setup
    x = case["free"]
    assert_close(obj.fun_free(x), oracle.kl(x), what="KL")
    ge = oracle.kl_grad(x)
    assert_close(obj.fun_free_grad(x), ge, scale=np.abs(ge).max() * 1e-3, what="grad")
    H, He = obj.fun_free_hessian(x), oracle.kl_hessian_csr(x)
    np.testing.assert_array_equal(H.indptr, He.indptr)
    np.testing.assert_array_equal(H.indices, He.indices)
    assert_close(H.data, He.data, scale=np.abs(He.data).max() * 1e-6, what="hessian data")
    v = np.random.default_rng(5).standard_normal(x.size)
    hve = oracle.kl_hvp(x, v)
    assert_close(obj.fun_free_hvp(x, v), hve, scale=np.abs(hve).max() * 1e-3, what="hvp")


def test_vector_coordinates(setup):
    case, oracle, model, obj = setup
    vec = oracle.free_to_vector(case["free"])
    kl, gv, blk = oracle.vector_derivs(vec, hessian=True)
    assert_close(obj.fun_vector(vec), kl, what="KL(vector)")
    assert_close(obj.fun_vector_grad(vec), gv, scale=np.abs(gv).max() * 1e-3, what="grad(vector)")
    Hd, He = obj.fun_vector_hessian(vec).toarray(), oracle.blocks_to_dense(oracle.lay, blk)
    assert_close(Hd, He, scale=np.abs(He).max() * 1e-6, what="hessian(vector)")
    v = np.random.default_rng(6).standard_normal(vec.size)
    assert_close(obj.fun_vector_hvp(vec, v), He @ v, scale=np.abs(He @ v).max() * 1e-3, what="hvp(vector)")
    assert_close(obj.fun_free(case["free"]), oracle.kl(case["free"]), what="KL after vector")


def test_weight_cross_hessian(setup):
    case, oracle, model, obj = setup
    x, N = case["free"], case["N"]
    w0 = np.ones(N) if case["w"] is None else case["w"]
    rng = np.random.default_rng(7)
    dw = rng.standard_normal(N)
    obj.fun_free_grad(x)
    ref = _oracle(case, w0 + dw).kl_grad(x) - _oracle(case, w0).kl_grad(x)
    assert_close(model.weight_cross_matvec(dw).cpu().numpy(), ref, scale=np.abs(ref).max() * 1e-3, what="C dw")
    v = rng.standard_normal(x.size)
    obj.fun_free(x)
    got = model.weight_cross_rmatvec(v).cpu().numpy()
    g0 = _oracle(case, w0).kl_grad(x)
    for n in rng.choice(N, size=8, replace=False):
        e = np.zeros(N)
        e[n] = 1.0
        col = _oracle(case, w0 + e).kl_grad(x) - g0
        assert abs(got[n] - col @ v) <= 1e-12 + 1e-9 * max(abs(col @ v), np.abs(col).max())


def test_determinism(setup):
    case, oracle, model, obj = setup
    x = torch.as_tensor(case["free"], device="cuda")
    model.evaluate(x, 2, force=True)
    a = model._out_global.clone(), model._grad_local.clone(), model.obs_weights().clone()
    model.evaluate(x, 2, force=True)
    b = model._out_global, model._grad_local, model.obs_weights()
    assert all(torch.equal(p, q) for p, q in zip(a, b))


@pytest.mark.timeout(900)
@pytest.mark.parametrize("K", [3, 16, 24, 50, 130])
def test_newton_lrvb_and_ij_at_the_optimum(vb, K):
    case = _case(K, 2500 if K <= 50 else 30 * K, 25, 4700 + K, shuffle=True, ragged=True, empty=2, weights=True,
                 offset=True, bounds=0.0)
    model = _model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    oracle = _oracle(case)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=1e-9)
    assert res.success, res.message
    xr = pois.newton_optimum(oracle, case["free"])
    assert_close(xo, xr, rtol=1e-7, scale=np.abs(xr).max() * 1e-3, what="optimum")
    Hinv = np.linalg.inv(oracle.kl_hessian_dense(xo))
    Dg = model.Dg
    for method in ("schur", "cg") if K <= 24 else ("schur",):
        lr = vb.LinearResponseCovariances(obj, xo, method=method, cg_tol=1e-12)
        assert_close(lr.get_global_covariance(), Hinv[:Dg, :Dg], rtol=1e-7,
                     scale=np.abs(Hinv[:Dg, :Dg]).max() * 1e-3, what="global covariance " + method)
    lr = vb.LinearResponseCovariances(obj, xo)
    J = model.moment_jacobian(xo)
    ref = J @ Hinv @ J.T
    assert_close(lr.get_lr_covariance(), ref, rtol=1e-8, scale=np.abs(ref).max() * 1e-3, what="moment covariance")
    fac = lr.get_lr_covariance_factors(J)
    assert_close(fac.diagonal(), np.diag(ref), rtol=1e-8, scale=np.abs(ref).max() * 1e-3, what="factored diagonal")
    for unit in ("row", "group"):
        got = lr.get_ij_covariance(unit)
        ref_ij = ij.ij_covariance_dense(oracle, xo, unit)[:Dg, :Dg]
        assert got.n_units == ij.n_units(oracle, unit)
        assert_close(got.global_cov, ref_ij, rtol=1e-8, scale=np.abs(ref_ij).max() * 1e-3, what="IJ " + unit)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("N,K", [(400003, 6), (100001, 50)])
def test_many_tiles_per_cta(vb, N, K):
    """More tiles per CTA than pipeline stages (the ring wraps) and a partial last tile."""
    case = _case(K, N, 300, 4900 + K, shuffle=False, ragged=True, empty=3, weights=True, offset=True, bounds=0.0)
    model = _model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    oracle = _oracle(case)
    x = case["free"]
    assert_close(obj.fun_free(x), oracle.kl(x), what="KL")
    ge = oracle.kl_grad(x)
    assert_close(obj.fun_free_grad(x), ge, scale=np.abs(ge).max() * 1e-3, what="grad")
    H, He = obj.fun_free_hessian(x), oracle.kl_hessian_csr(x)
    np.testing.assert_array_equal(H.indices, He.indices)
    assert_close(H.data, He.data, scale=np.abs(He.data).max() * 1e-6, what="hessian data")


def test_no_observations(vb):
    X = np.zeros((0, 4))
    model = vb.PoissonGLMM(X, np.zeros(0), np.zeros(0, dtype=np.int64), num_groups=3)
    oracle = pois.PoissonOracle(X, np.zeros(0), np.zeros(0, dtype=np.int64), G=3)
    obj = vb.Objective(model.glmm_par, model)
    x = go.make_free(model.D, 9)
    assert_close(obj.fun_free(x), oracle.kl(x), what="KL")
    H, He = obj.fun_free_hessian(x), oracle.kl_hessian_csr(x)
    np.testing.assert_array_equal(H.indices, He.indices)
    assert_close(H.data, He.data, scale=np.abs(He.data).max() * 1e-6, what="hessian data")


def test_rejected_data(vb):
    X, y, g, off = pois.make_poisson_data(300, 4, 5, 77, offset=True)
    for bad in (-1.0, np.nan, np.inf):
        yb = y.copy()
        yb[17] = bad
        with pytest.raises(ValueError, match="y must be finite and >= 0"):
            vb.PoissonGLMM(X, yb, g, offset=off)
    ob = off.copy()
    ob[5] = np.nan
    with pytest.raises(ValueError, match="offset must be finite"):
        vb.PoissonGLMM(X, y, g, offset=ob)
    with pytest.raises(ValueError, match="offset"):
        vb.PoissonGLMM(X, y, g, offset=off[:-1])
    yf = y + 0.25                       # non-integer counts are accepted
    vb.PoissonGLMM(X, yf, g, offset=off)


def test_refused_calls(vb):
    from lrvb_b200 import _native as nat
    case = _case(5, 400, 6, 91, shuffle=False, ragged=False, empty=0, weights=False, offset=False, bounds=0.0)
    model = _model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    x = case["free"]
    obj.fun_free_hessian(x)
    lr = vb.LinearResponseCovariances(obj, x)
    Xn, gn = case["X"][:4], case["g"][:4]
    for call in (lambda: model.predict(x, Xn, gn), lambda: lr.get_prediction_variances(Xn, gn),
                 lambda: lr.get_approximate_loo(), lambda: lr.get_approximate_logo(),
                 lambda: lr.get_approximate_max_influence(0), lambda: model.third_derivative_contraction(x),
                 lambda: model.approximate_loo(None, None, None), lambda: model.approximate_logo(None)):
        with pytest.raises(NotImplementedError, match="Poisson|poisson"):
            call()
    # the C entry points refuse before touching their arguments
    lib, h = nat.load(), model._h
    d = torch.zeros(max(model.D, model.Dg * model.Dg, 6 * model.N), dtype=torch.float64, device="cuda")
    p, s = nat.ptr(d), nat.stream_ptr()
    gi = torch.zeros(4, dtype=torch.int32, device="cuda")
    rcs = [lib.lrvb_glmm_predict(h, p, p, model.K, nat.ptr(gi), None, 4, p, s),
           lib.lrvb_glmm_predict_lr(h, p, p, p, p, model.K, nat.ptr(gi), None, 4, p, s),
           lib.lrvb_glmm_loo(h, p, p, p, p, s),
           lib.lrvb_glmm_logo(h, p, p, p, p, p, s),
           lib.lrvb_glmm_third_contract(h, p, p, p, s)]
    for rc in rcs:
        assert rc == nat.LRVB_EINVAL
    torch.cuda.synchronize()
    assert "Poisson" in nat.last_error()
