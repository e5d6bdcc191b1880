"""Approximate leave-one-group-out cross-validation and group influence (LinearResponseCovariances.get_approximate_logo,
csrc/logo.cu lrvb_glmm_logo): against the dense numpy oracle at the optimum, against the weight-sensitivity path one
group at a time, end to end through model.predict, and its determinism, return types and errors."""
import numpy as np
import pytest
import torch

from helpers import assert_close, make_case, make_model, make_oracle
from oracle import logo_oracle as lg
from oracle import loo_oracle as lo

pytestmark = pytest.mark.gpu

ROW_FIELDS = ("lpd_logo", "eta_mean_logo", "eta_var_logo")
GROUP_FIELDS = ("elpd_logo_group", "cooks_distance", "delta_global")


def _optimum(vb, case, gtol=1e-7):
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=gtol)
    assert res.success, res.message
    return model, obj, xo


def _case(K, N, seed, G=30, empty=3):
    """Shuffled rows, ragged groups, `empty` groups without rows, weights with zeros and one group (the returned
    id) whose rows all have weight 0."""
    case = make_case(N=N, K=K, G=G, Q=8 if K % 2 else 4, seed=seed, shuffle=True, ragged=True, weights=True,
                     empty_groups=empty)
    rng = np.random.default_rng(seed + 1)
    case["w"][rng.choice(N, size=6, replace=False)] = 0.0
    sizes = np.bincount(case["g"], minlength=G)
    dead = int(np.nonzero(sizes > 0)[0][0])
    case["w"][case["g"] == dead] = 0.0
    return case, dead


def _oracle_logo(case, xo):
    """The oracle's result with its rows in the caller's order (the oracle holds them group-sorted)."""
    r = lg.approximate_logo(make_oracle(case), xo)
    order = np.argsort(case["g"], kind="stable")
    for f in ROW_FIELDS:
        v = np.empty_like(r[f])
        v[order] = r[f]
        r[f] = v
    return r


@pytest.mark.timeout(900)
@pytest.mark.parametrize("K", [1, 5, 20, 24, 25, 50, 130, 200])
def test_matches_oracle_at_the_optimum(vb, K):
    case, dead = _case(K, 3000 if K <= 50 else 40 * K, 900 + K)
    model, obj, xo = _optimum(vb, case)
    assert model.perm is not None
    got = vb.LinearResponseCovariances(obj, xo).get_approximate_logo()
    ref = _oracle_logo(case, xo)
    for f in ROW_FIELDS + GROUP_FIELDS:
        v = getattr(got, f)
        assert isinstance(v, np.ndarray) and v.shape == ref[f].shape, f
        # delta and Cook's distance of a group are judged against the largest over the groups
        scale = np.abs(ref[f]).max() if f in ("cooks_distance", "delta_global") else None
        assert_close(v, ref[f], scale=scale, what="%s K=%d" % (f, K))
    assert_close(got.elpd_logo, ref["elpd_logo"], what="elpd_logo")
    assert_close(got.elpd_logo_se, ref["elpd_logo_se"], what="elpd_logo_se")
    empty = np.bincount(case["g"], minlength=case["G"]) == 0
    assert empty.sum() == 3
    for g in list(np.nonzero(empty)[0]) + [dead]:
        assert np.all(got.delta_global[g] == 0.0) and got.cooks_distance[g] == 0.0, g
    assert np.all(got.elpd_logo_group[empty] == 0.0)


def _check_against_weight_sensitivity(vb, obj, model, case, xo, lr, groups):
    a = lr.get_approximate_logo()
    ws = vb.WeightSensitivityLinearApproximation(obj, xo)
    w = np.ones(case["N"]) if case["w"] is None else case["w"]
    Dg, G = model.Dg, model.G
    for g in groups:
        diff = np.where(case["g"] == g, -w, 0.0)
        dtheta = np.asarray(ws.get_dinput_dhyper_times(diff))
        assert_close(a.delta_global[g], dtheta[:Dg], scale=np.abs(dtheta[:Dg]).max(), what="delta group %d" % g)
        # end to end: the globals at theta + delta_g, q(u_g) at its closed form, through model.predict
        free = np.array(xo, dtype=np.float64)
        free[:Dg] += a.delta_global[g]
        lb = case["bounds"]
        info = max((np.exp(free[2]) + lb) / (np.exp(free[3]) + lb), lb)
        free[Dg + g] = free[0]
        free[Dg + G + g] = np.log(info - lb)
        rows = np.nonzero(case["g"] == g)[0]
        p = model.predict(free, case["X"][rows], case["g"][rows])
        assert_close(a.eta_mean_logo[rows], p.eta_mean, what="eta_mean group %d" % g)
        assert_close(a.eta_var_logo[rows], p.eta_var_mfvb, what="eta_var group %d" % g)
        lpd = lo.log_predictive_density(p.eta_mean, p.eta_var_mfvb, case["y"][rows], case["gh_x"], case["gh_w"])
        assert_close(a.lpd_logo[rows], lpd, what="lpd group %d" % g)
    b = lr.get_approximate_logo()      # the weight-sensitivity calls in between leave W alone
    for f in a._fields:
        np.testing.assert_array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(b, f)), err_msg=f)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("K", [5, 130])
def test_matches_weight_sensitivity_path(vb, K):
    case = make_case(N=4000 if K < 62 else 6000, K=K, G=25, Q=6, seed=1000 + K, shuffle=True, weights=True)
    model, obj, xo = _optimum(vb, case)
    lr = vb.LinearResponseCovariances(obj, xo)
    groups = np.random.default_rng(K).choice(case["G"], size=5, replace=False)
    _check_against_weight_sensitivity(vb, obj, model, case, xo, lr, groups)


@pytest.fixture(scope="module")
def c2_optimum(vb):
    case = make_case(N=1_000_000, K=20, G=10_000, Q=8, seed=2200, shuffle=True)
    model, obj, xo = _optimum(vb, case)
    return case, model, obj, vb.LinearResponseCovariances(obj, xo), xo


@pytest.mark.timeout(900)
def test_matches_weight_sensitivity_path_at_c2(vb, c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    groups = np.random.default_rng(3).choice(case["G"], size=5, replace=False)
    _check_against_weight_sensitivity(vb, obj, model, case, xo, lr, groups)


def test_determinism_and_types(c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    a, b = lr.get_approximate_logo(), lr.get_approximate_logo()
    for f in a._fields:
        np.testing.assert_array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(b, f)), err_msg=f)
    assert isinstance(a.elpd_logo, float) and isinstance(a.elpd_logo_se, float)
    assert np.isfinite(a.elpd_logo) and np.isfinite(a.elpd_logo_se)
    assert np.all(np.isfinite(a.lpd_logo)) and np.all(a.cooks_distance >= 0)
    assert a.delta_global.shape == (case["G"], model.Dg)
    import lrvb_b200 as vb
    t = vb.LinearResponseCovariances(obj, torch.from_numpy(xo).cuda()).get_approximate_logo()
    assert isinstance(t, vb.ApproximateLOGO)
    for f in ROW_FIELDS + GROUP_FIELDS:
        v = getattr(t, f)
        assert torch.is_tensor(v) and v.is_cuda, f
        np.testing.assert_array_equal(v.cpu().numpy(), getattr(a, f), err_msg=f)


def test_errors(vb, tmp_path):
    case = make_case(N=600, K=6, G=8, Q=4, seed=13)
    y = case["y"].copy()
    y[17] = 0.5
    bad = vb.LogisticGLMM(case["X"], y, case["g"], gh_x=case["gh_x"], gh_w=case["gh_w"], num_groups=case["G"])
    lr = vb.LinearResponseCovariances(vb.Objective(bad.glmm_par, bad), case["free"])
    with pytest.raises(ValueError):
        lr.get_approximate_logo()

    import torch.distributed as dist
    from lrvb_b200.distributed import ShardedLogisticGLMM
    dist.init_process_group("gloo", init_method="file://" + str(tmp_path / "store"), rank=0, world_size=1)
    try:
        small = make_case(N=2000, K=3, G=10, Q=4, seed=11)
        sharded = ShardedLogisticGLMM.from_full(small["X"], small["y"], small["g"], small["G"], num_gh_points=4)
        obj = vb.Objective(sharded.glmm_par, sharded)
        with pytest.raises(NotImplementedError):
            sharded.approximate_logo(None)
        with pytest.raises(NotImplementedError):
            vb.LinearResponseCovariances(obj, small["free"]).get_approximate_logo()
    finally:
        dist.destroy_process_group()


def test_c_abi_status_codes(vb):
    from lrvb_b200 import _native as nat
    case = make_case(N=600, K=6, G=8, Q=4, seed=12)
    model = make_model(vb, case)
    lib, h, st, P = model._lib, model._h, nat.stream_ptr(), nat.ptr
    sinv = torch.eye(model.Dg, dtype=torch.float64, device="cuda")
    pinv = torch.eye(model.K, dtype=torch.float64, device="cuda")
    delta = torch.empty(model.G, model.Dg, dtype=torch.float64, device="cuda")
    grp = torch.empty(2, model.G, dtype=torch.float64, device="cuda")
    out = torch.empty(3, model.N, dtype=torch.float64, device="cuda")

    def logo(hh=h, s=sinv, p=pinv, d=delta, g=grp, o=out):
        return lib.lrvb_glmm_logo(hh, P(s), P(p), P(d), P(g), P(o), st)

    assert logo() == nat.LRVB_ESTATE          # no order-2 evaluation yet
    model.evaluate(case["free"], 1)
    assert logo() == nat.LRVB_ESTATE          # order 1 caches no Hessian
    model.evaluate(case["free"], 2)
    assert logo() == nat.LRVB_OK
    assert logo(hh=None) == nat.LRVB_EINVAL
    for kw in (dict(s=None), dict(p=None), dict(d=None), dict(g=None), dict(o=None)):
        assert logo(**kw) == nat.LRVB_EINVAL, kw
        assert "NULL" in nat.last_error()
    torch.cuda.synchronize()
