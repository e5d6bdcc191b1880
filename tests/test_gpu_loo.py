"""Approximate leave-one-out cross-validation (LinearResponseCovariances.get_approximate_loo, csrc/predict.cu
lrvb_glmm_loo): against the dense numpy oracle at the optimum, against the per-row weight-sensitivity path, against
exact refits without a row, and its determinism, return types and errors."""
import numpy as np
import pytest
import torch

from helpers import assert_close, make_case, make_model, make_oracle
from oracle import loo_oracle as lo
from oracle import predict_oracle as po

pytestmark = pytest.mark.gpu

FIELDS = ("lpd", "lpd_loo", "eta_mean_loo", "eta_var_loo")


def _bounds(case):
    b = case["bounds"]
    return dict(mu_info=b, beta_info=b, u_info=b)


def _weighted_case(zero_rows=6, **kw):
    """make_case with weights, some of them 0; returns (case, the rows of weight 0 in caller order)."""
    case = make_case(weights=True, **kw)
    zero = np.random.default_rng(kw["seed"] + 1).choice(case["N"], size=zero_rows, replace=False)
    case["w"][zero] = 0.0
    return case, zero


def _optimum(vb, case, gtol=1e-7):
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=gtol)
    assert res.success, res.message
    return model, obj, xo


def _oracle_loo(case, xo):
    """The oracle's result in the caller's row order (the oracle holds the rows group-sorted)."""
    r = lo.approximate_loo(make_oracle(case), xo)
    order = np.argsort(case["g"], kind="stable")
    for f in FIELDS:
        v = np.empty_like(r[f])
        v[order] = r[f]
        r[f] = v
    return r


def _check_against_oracle(got, ref, what):
    for f in FIELDS:
        assert isinstance(getattr(got, f), np.ndarray) and getattr(got, f).shape == ref[f].shape
        assert_close(getattr(got, f), ref[f], what="%s %s" % (f, what))
    assert got.n_invalid == ref["n_invalid"] == 0
    assert_close(got.elpd_loo, ref["elpd_loo"], what="elpd_loo " + what)
    assert_close(got.elpd_loo_se, ref["elpd_loo_se"], what="elpd_loo_se " + what)
    # p_loo is a difference of two sums of size ~elpd: judged against that scale
    assert_close(got.p_loo, ref["p_loo"], scale=abs(ref["elpd_loo"]), what="p_loo " + what)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("K", [1, 5, 20, 24, 25, 50, 130, 200])
def test_matches_oracle_at_the_optimum(vb, K):
    N = 3000 if K <= 50 else 40 * K
    case, zero = _weighted_case(N=N, K=K, G=30, Q=8 if K % 2 else 4, seed=700 + K, shuffle=True)
    model, obj, xo = _optimum(vb, case)
    assert model.perm is not None
    got = vb.LinearResponseCovariances(obj, xo).get_approximate_loo()
    _check_against_oracle(got, _oracle_loo(case, xo), "K=%d" % K)
    # weight-zero rows are already held out: no shift at all
    np.testing.assert_array_equal(got.lpd_loo[zero], got.lpd[zero])
    pred = model.predict(xo, case["X"][zero], case["g"][zero])
    assert_close(got.eta_mean_loo[zero], pred.eta_mean, what="eta_mean of w = 0 rows")


def _shifts_by_weight_sensitivity(vb, obj, model, case, xo, rows):
    """(dz_m, dz_v) of `rows` (caller order): get_dinput_dhyper_times(-w_n e_n) through the row's moment Jacobians."""
    ws = vb.WeightSensitivityLinearApproximation(obj, xo)
    w = np.ones(case["N"]) if case["w"] is None else case["w"]
    dm, dv = [], []
    for n in rows:
        diff = np.zeros(case["N"])
        diff[n] = -w[n]
        dtheta = np.asarray(ws.get_dinput_dhyper_times(diff))
        Jm = model.prediction_jacobian(xo, case["X"][n:n + 1], case["g"][n:n + 1], quantity="eta")
        _, Jv = lo.moment_jacobians(xo, case["X"][n:n + 1], case["g"][n:n + 1], case["K"], case["G"], _bounds(case))
        dm.append((Jm @ dtheta)[0])
        dv.append((Jv @ dtheta)[0])
    return np.array(dm), np.array(dv)


def _check_shifts(vb, obj, model, lr, case, xo, rows):
    a = lr.get_approximate_loo()
    dm, dv = _shifts_by_weight_sensitivity(vb, obj, model, case, xo, rows)
    b = lr.get_approximate_loo()       # the weight-sensitivity calls in between leave W alone
    for f in a._fields:
        np.testing.assert_array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(b, f)), err_msg=f)
    pred = model.predict(xo, case["X"][rows], case["g"][rows])
    got_m = b.eta_mean_loo[rows] - pred.eta_mean
    got_v = b.eta_var_loo[rows] - pred.eta_var_mfvb
    assert_close(got_m, dm, scale=1e-3 * np.abs(dm).max(), what="dz_m")
    assert_close(got_v, dv, scale=1e-3 * np.abs(dv).max(), what="dz_v")


@pytest.mark.timeout(900)
@pytest.mark.parametrize("K", [5, 130])
def test_matches_weight_sensitivity_path(vb, K):
    case, _ = _weighted_case(N=4000 if K < 62 else 6000, K=K, G=25, Q=6, seed=800 + K, shuffle=True)
    model, obj, xo = _optimum(vb, case)
    lr = vb.LinearResponseCovariances(obj, xo)
    rows = np.random.default_rng(K).choice(case["N"], size=10, replace=False)
    _check_shifts(vb, obj, model, lr, case, xo, rows)


@pytest.fixture(scope="module")
def c2_optimum(vb):
    case = make_case(N=1_000_000, K=20, G=10_000, Q=8, seed=2200, shuffle=True)
    model, obj, xo = _optimum(vb, case)
    return case, model, obj, vb.LinearResponseCovariances(obj, xo), xo


@pytest.mark.timeout(900)
def test_matches_weight_sensitivity_path_at_c2(vb, c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    rows = np.random.default_rng(3).choice(case["N"], size=10, replace=False)
    _check_shifts(vb, obj, model, lr, case, xo, rows)


def test_determinism_and_types(c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    a, b = lr.get_approximate_loo(), lr.get_approximate_loo()
    for f in a._fields:
        np.testing.assert_array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(b, f)), err_msg=f)
    assert a.n_invalid == 0 and np.isfinite(a.elpd_loo) and np.isfinite(a.elpd_loo_se)
    assert isinstance(a.elpd_loo, float) and isinstance(a.n_invalid, int)
    import lrvb_b200 as vb
    t = vb.LinearResponseCovariances(obj, torch.from_numpy(xo).cuda()).get_approximate_loo()
    assert isinstance(t, vb.ApproximateLOO)
    for f in FIELDS:
        v = getattr(t, f)
        assert torch.is_tensor(v) and v.is_cuda and v.shape == (case["N"],)
        np.testing.assert_array_equal(v.cpu().numpy(), getattr(a, f), err_msg=f)


@pytest.mark.timeout(900)
def test_close_to_exact_refits(vb):
    """IJ error << the LOO effect: |lpd_loo - lpd_exact| <= 0.1 |lpd - lpd_exact| + 1e-8 on the 8 rows of largest
    |w l_m|, each refitted without its row."""
    case = make_case(N=3000, K=4, G=30, Q=8, seed=4242)
    model, obj, xo = _optimum(vb, case, gtol=1e-10)
    got = vb.LinearResponseCovariances(obj, xo).get_approximate_loo()
    assert model.perm is None
    W_m = model.obs_weights()[0].cpu().numpy()
    rows = np.argsort(-np.abs(W_m), kind="stable")[:8]
    for n in rows:
        w = np.ones(case["N"])
        w[n] = 0.0
        m2 = vb.LogisticGLMM(case["X"], case["y"], case["g"], gh_x=case["gh_x"], gh_w=case["gh_w"], weights=w,
                             num_groups=case["G"])
        x2, res = vb.OptimizationUtils.minimize_objective_newton(vb.Objective(m2.glmm_par, m2), xo, maxiter=60,
                                                                 gtol=1e-10)
        assert res.success, res.message
        p = po.predict(x2, case["X"][n:n + 1], case["g"][n:n + 1], case["K"], case["G"], case["gh_x"],
                       case["gh_w"], _bounds(case))
        exact = lo.log_predictive_density(p["eta_mean"], p["eta_var_mfvb"], case["y"][n:n + 1], case["gh_x"],
                                          case["gh_w"])[0]
        err, effect = abs(got.lpd_loo[n] - exact), abs(got.lpd[n] - exact)
        assert err <= 0.1 * effect + 1e-8, (int(n), got.lpd[n], got.lpd_loo[n], exact)


def test_errors(vb, tmp_path):
    case = make_case(N=600, K=6, G=8, Q=4, seed=13)
    y = case["y"].copy()
    y[17] = 0.5
    bad = vb.LogisticGLMM(case["X"], y, case["g"], gh_x=case["gh_x"], gh_w=case["gh_w"], num_groups=case["G"])
    lr = vb.LinearResponseCovariances(vb.Objective(bad.glmm_par, bad), case["free"])
    with pytest.raises(ValueError):
        lr.get_approximate_loo()

    import torch.distributed as dist
    from lrvb_b200.distributed import ShardedLogisticGLMM
    dist.init_process_group("gloo", init_method="file://" + str(tmp_path / "store"), rank=0, world_size=1)
    try:
        small = make_case(N=2000, K=3, G=10, Q=4, seed=11)
        sharded = ShardedLogisticGLMM.from_full(small["X"], small["y"], small["g"], small["G"], num_gh_points=4)
        obj = vb.Objective(sharded.glmm_par, sharded)
        with pytest.raises(NotImplementedError):
            sharded.approximate_loo(None, None, None)
        with pytest.raises(NotImplementedError):
            vb.LinearResponseCovariances(obj, small["free"]).get_approximate_loo()
    finally:
        dist.destroy_process_group()


def test_c_abi_status_codes(vb):
    from lrvb_b200 import _native as nat
    case = make_case(N=600, K=6, G=8, Q=4, seed=12)
    model = make_model(vb, case)
    lib, h, st, P = model._lib, model._h, nat.stream_ptr(), nat.ptr
    sinv = torch.eye(model.Dg, dtype=torch.float64, device="cuda")
    cross = torch.zeros(model.G, 2, 2 * model.K, dtype=torch.float64, device="cuda")
    lcov = torch.ones(model.G, 3, dtype=torch.float64, device="cuda")
    out = torch.empty(4, model.N, dtype=torch.float64, device="cuda")

    def loo(hh=h, s=sinv, c=cross, l=lcov, o=out):
        return lib.lrvb_glmm_loo(hh, P(s), P(c), P(l), P(o), st)

    assert loo() == nat.LRVB_ESTATE          # no order-2 evaluation yet
    model.evaluate(case["free"], 1)
    assert loo() == nat.LRVB_ESTATE          # order 1 caches no Hessian
    model.evaluate(case["free"], 2)
    assert loo() == nat.LRVB_OK
    assert loo(hh=None) == nat.LRVB_EINVAL
    for kw in (dict(s=None), dict(c=None), dict(l=None), dict(o=None)):
        assert loo(**kw) == nat.LRVB_EINVAL, kw
        assert "NULL" in nat.last_error()
    torch.cuda.synchronize()
