"""Prediction on new rows (csrc/predict.cu): LogisticGLMM.predict against the numpy oracle, the LRVB
variances of LinearResponseCovariances.get_prediction_variances against diag(J H^-1 J^T) with the dense
inverse of the oracle Hessian and against the factored path, at scale, determinism and input errors."""
import numpy as np
import pytest
import torch

from helpers import assert_close, make_case, make_model, make_oracle
from oracle import predict_oracle as po

pytestmark = pytest.mark.gpu

FIELDS = ("eta_mean", "eta_var_mfvb", "prob", "prob_var_mfvb")


def _bounds(case):
    b = case["bounds"]
    return dict(mu_info=b, beta_info=b, u_info=b)


def _new_rows(case, M, seed):
    """M rows in random order with every kind of group id: -1, ids with training rows, ids without."""
    rng = np.random.default_rng(seed)
    X = 0.7 * rng.standard_normal((M, case["K"]))
    g = rng.integers(-1, case["G"], size=M)
    empty = np.setdiff1d(np.arange(case["G"]), case["g"])
    if M >= 3:
        g[:3] = [-1, int(empty[0]) if empty.size else 0, case["G"] - 1]
        rng.shuffle(g)
    return X, g


def _oracle_predict(case, x, X, g):
    return po.predict(x, X, g, case["K"], case["G"], case["gh_x"], case["gh_w"], _bounds(case))


@pytest.mark.parametrize("K", [1, 5, 20, 50, 130, 200, 256])
@pytest.mark.parametrize("Q,bounds", [(4, 0.0), (8, 0.1)])
def test_predict_matches_oracle(vb, K, Q, bounds):
    case = make_case(N=1500, K=K, G=40, Q=Q, seed=500 + K + Q, shuffle=True, bounds=bounds, empty_groups=3)
    model = make_model(vb, case)
    x = case["free"]
    for M in (0, 1, 37, 100_003):
        X, g = _new_rows(case, M, seed=M + K)
        got = model.predict(x, X, g)
        ref = _oracle_predict(case, x, X, g)
        for f in FIELDS:
            assert isinstance(getattr(got, f), np.ndarray) and getattr(got, f).shape == (M,)
            assert_close(getattr(got, f), ref[f], what="%s K=%d M=%d" % (f, K, M))
        assert got.prob_var_lr is None and got.eta_var_lr is None
    # CUDA tensors in, CUDA tensors out
    X, g = _new_rows(case, 37, seed=9)
    got = model.predict(torch.from_numpy(x).cuda(), torch.from_numpy(X).cuda(), torch.from_numpy(g).cuda())
    assert got.prob.is_cuda
    assert_close(got.prob.cpu().numpy(), _oracle_predict(case, x, X, g)["prob"], what="prob (torch)")


def _optimum(vb, case):
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=1e-7)
    assert res.success, res.message
    return model, obj, xo


@pytest.mark.timeout(900)
@pytest.mark.parametrize("name,kw", [
    ("c1", dict(N=5000, K=5, G=100, Q=4, seed=1001)),
    ("k20", dict(N=20000, K=20, G=200, Q=8, seed=2001)),
    ("k50", dict(N=6000, K=50, G=60, Q=8, seed=3001)),
    ("k130", dict(N=4000, K=130, G=20, Q=4, seed=23)),
    ("k200", dict(N=12_000, K=200, G=30, Q=8, seed=4001)),
])
def test_lr_variances_at_the_optimum(vb, name, kw):
    case = make_case(**kw)
    oracle = make_oracle(case)
    model, obj, xo = _optimum(vb, case)
    Hinv = np.linalg.inv(oracle.kl_hessian_dense(xo))
    lr = vb.LinearResponseCovariances(obj, xo)
    X, g = _new_rows(case, 301, seed=kw["seed"])
    got = lr.get_prediction_variances(X, g)
    ref = _oracle_predict(case, xo, X, g)
    for f in FIELDS:
        assert_close(getattr(got, f), ref[f], what=f)
    for quantity, field in (("prob", "prob_var_lr"), ("eta", "eta_var_lr")):
        J = po.prediction_jacobian(xo, X, g, case["K"], case["G"], case["gh_x"], case["gh_w"], _bounds(case),
                                   quantity=quantity)
        Jm = model.prediction_jacobian(xo, X, g, quantity=quantity)
        assert_close(Jm.toarray(), J.toarray(), scale=np.abs(J.data).max() * 1e-3, what="jacobian " + quantity)
        var = po.lr_variances(J, Hinv)
        assert_close(getattr(got, field), var, rtol=1e-8, scale=np.abs(var).max() * 1e-3, what=field)
        fac = lr.get_lr_covariance_factors(Jm).diagonal()
        assert_close(getattr(got, field), fac, rtol=1e-8, scale=np.abs(fac).max() * 1e-3,
                     what=field + " vs factored")
    # the LR variances never fall below zero and the MFVB ones stay positive
    assert np.all(got.prob_var_lr > 0) and np.all(got.prob_var_mfvb > 0)


@pytest.fixture(scope="module")
def c2_optimum(vb):
    case = make_case(N=400_000, K=20, G=10_000, Q=8, seed=2100)
    model, obj, xo = _optimum(vb, case)
    return case, model, vb.LinearResponseCovariances(obj, xo), xo


@pytest.mark.timeout(900)
def test_lr_variances_at_scale(c2_optimum):
    case, model, lr, xo = c2_optimum
    M = 1_000_000
    Xh, gh = _new_rows(case, M, seed=77)
    X, g = torch.from_numpy(Xh).cuda(), torch.from_numpy(gh).cuda()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    got = lr.get_prediction_variances(X, g)
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    limit = X.nbytes + g.nbytes + 6 * 8 * M + 16 * 8 * case["G"] * case["K"]
    assert growth < limit, (growth, limit)
    idx = np.random.default_rng(5).choice(M, size=1000, replace=False)
    for quantity, field in (("prob", "prob_var_lr"), ("eta", "eta_var_lr")):
        J = model.prediction_jacobian(xo, Xh[idx], gh[idx], quantity=quantity)
        fac = lr.get_lr_covariance_factors(J).diagonal()
        v = getattr(got, field).cpu().numpy()[idx]
        assert_close(v, fac, rtol=1e-8, scale=np.abs(fac).max() * 1e-3, what=field)
    ref = _oracle_predict(case, xo, Xh[idx], gh[idx])
    for f in FIELDS:
        assert_close(getattr(got, f).cpu().numpy()[idx], ref[f], what=f)


def test_determinism(c2_optimum):
    case, model, lr, xo = c2_optimum
    M = 200_003
    Xh, gh = _new_rows(case, M, seed=78)
    a = lr.get_prediction_variances(Xh, gh)
    b = lr.get_prediction_variances(Xh, gh)
    perm = np.random.default_rng(6).permutation(M)
    c = lr.get_prediction_variances(Xh[perm], gh[perm])
    p = model.predict(xo, Xh, gh)
    q = model.predict(xo, Xh[perm], gh[perm])
    for f in a._fields:
        np.testing.assert_array_equal(getattr(a, f), getattr(b, f), err_msg=f)
        np.testing.assert_array_equal(getattr(c, f), getattr(a, f)[perm], err_msg=f)
    for f in FIELDS:
        np.testing.assert_array_equal(getattr(q, f), getattr(p, f)[perm], err_msg=f)
        np.testing.assert_array_equal(getattr(p, f), getattr(a, f), err_msg=f)


def test_input_errors(vb, c2_optimum, tmp_path):
    case, model, lr, xo = c2_optimum
    K, G = case["K"], case["G"]
    X = np.zeros((5, K))
    with pytest.raises(ValueError):
        model.predict(xo, np.zeros((5, K + 1)), np.zeros(5, dtype=np.int64))
    with pytest.raises(ValueError):
        lr.get_prediction_variances(np.zeros((5, K - 1)), np.zeros(5, dtype=np.int64))
    for bad in ([0, 0, 0, 0, G], [0, -2, 0, 0, 0]):
        with pytest.raises(ValueError):
            model.predict(xo, X, np.array(bad))
        with pytest.raises(ValueError):
            lr.get_prediction_variances(X, torch.tensor(bad, device="cuda"))
    with pytest.raises(ValueError):
        model.predict(xo, X, np.array([0, 0.5, 0, 0, 0]))
    with pytest.raises(ValueError):
        model.predict(xo, X, np.zeros(4, dtype=np.int64))

    import torch.distributed as dist
    from lrvb_b200.distributed import ShardedLogisticGLMM
    dist.init_process_group("gloo", init_method="file://" + str(tmp_path / "store"), rank=0, world_size=1)
    try:
        small = make_case(N=2000, K=3, G=10, Q=4, seed=11)
        sharded = ShardedLogisticGLMM.from_full(small["X"], small["y"], small["g"], small["G"], num_gh_points=4)
        obj = vb.Objective(sharded.glmm_par, sharded)
        with pytest.raises(NotImplementedError):
            sharded.predict(small["free"], np.zeros((2, 3)), np.zeros(2, dtype=np.int64))
        with pytest.raises(NotImplementedError):
            vb.LinearResponseCovariances(obj, small["free"]).get_prediction_variances(
                np.zeros((2, 3)), np.zeros(2, dtype=np.int64))
    finally:
        dist.destroy_process_group()


def test_c_abi_status_codes(vb):
    """The entry points report misuse themselves (the Python layer checks first, a C caller has only these)."""
    from lrvb_b200 import _native as nat
    case = make_case(N=600, K=6, G=8, Q=4, seed=12)
    model = make_model(vb, case)
    lib, h, st = model._lib, model._h, nat.stream_ptr()
    K, G, M = 6, 8, 33
    buf = torch.zeros(M * K + 1, dtype=torch.float64, device="cuda")
    X, Xmis = buf[:M * K], buf[1:]
    g = torch.zeros(M, dtype=torch.int32, device="cuda")
    free = torch.from_numpy(case["free"]).cuda()
    out = torch.empty(6, M, dtype=torch.float64, device="cuda")
    sinv = torch.eye(model.Dg, dtype=torch.float64, device="cuda")
    cross = torch.zeros(G, 2, 2 * K, dtype=torch.float64, device="cuda")
    lcov = torch.zeros(G, 3, dtype=torch.float64, device="cuda")
    P = nat.ptr

    def pred(Xt=X, k=K, m=M, f=free):
        return lib.lrvb_glmm_predict(h, P(f), P(Xt), k, P(g), None, m, P(out), st)

    def pred_lr(Xt=X, k=K, m=M):
        return lib.lrvb_glmm_predict_lr(h, P(sinv), P(cross), P(lcov), P(Xt), k, P(g), None, m, P(out), st)

    # no Hessian cached yet: the LR pieces are refused, the MFVB prediction needs only the free point
    assert pred_lr() == nat.LRVB_ESTATE
    assert lib.lrvb_glmm_predict_cross(h, P(sinv), P(cross), st) == nat.LRVB_ESTATE
    assert pred() == nat.LRVB_OK
    model.evaluate(case["free"], 2)
    assert lib.lrvb_glmm_predict_cross(h, P(sinv), P(cross), st) == nat.LRVB_OK
    assert pred_lr() == nat.LRVB_OK
    for call in (pred, pred_lr):
        assert call(k=K + 1) == nat.LRVB_EINVAL
        assert call(m=-1) == nat.LRVB_EINVAL
        assert call(Xt=Xmis) == nat.LRVB_EINVAL
        assert "aligned" in nat.last_error()
    assert pred(f=None) == nat.LRVB_EINVAL
    assert lib.lrvb_glmm_predict(None, P(free), P(X), K, P(g), None, M, P(out), st) == nat.LRVB_EINVAL
    torch.cuda.synchronize()
