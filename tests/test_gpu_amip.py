"""The approximate maximum influence perturbation (LinearResponseCovariances.get_approximate_max_influence, csrc/amip.cu
lrvb_glmm_third_contract): against the dense numpy oracle at the optimum, against the weight-sensitivity and LOGO
paths, against exact refits without the selected rows or groups, at C2 size, and its errors."""
import numpy as np
import pytest
import torch

from helpers import assert_close, make_case, make_model, make_oracle
from oracle import amip_oracle as am
from oracle import glmm_oracle as go

pytestmark = pytest.mark.gpu


def _optimum(vb, case, gtol=1e-7):
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=gtol)
    assert res.success, res.message
    return model, obj, xo


def _case(K, N, seed, G=30, empty=3):
    """Shuffled rows, ragged groups, `empty` groups without rows, weights with zeros and one group whose rows all
    have weight 0 (the case mix of test_gpu_logo.py)."""
    case = make_case(N=N, K=K, G=G, Q=8 if K % 2 else 4, seed=seed, shuffle=True, ragged=True, weights=True,
                     empty_groups=empty)
    rng = np.random.default_rng(seed + 1)
    case["w"][rng.choice(N, size=6, replace=False)] = 0.0
    sizes = np.bincount(case["g"], minlength=G)
    case["w"][case["g"] == int(np.nonzero(sizes > 0)[0][0])] = 0.0
    return case


def _check_drops(got, ref, to_caller, what):
    for name in am.TARGETS:
        g, r = got.targets[name], ref[name]
        assert g.n_drop == r["n_drop"], (what, name, g.n_drop, r["n_drop"])
        np.testing.assert_array_equal(g.dropped, to_caller(r["dropped"]), err_msg="%s %s" % (what, name))
        if r["n_drop"] is None:
            assert g.fraction is None and g.predicted_estimate is None and g.predicted_sd is None
            continue
        assert_close(g.fraction, r["fraction"], what="%s %s fraction" % (what, name))
        assert_close(g.predicted_estimate, r["predicted_estimate"], what="%s %s estimate" % (what, name))
        assert_close(g.predicted_sd, r["predicted_sd"], what="%s %s sd" % (what, name))


@pytest.mark.timeout(900)
@pytest.mark.parametrize("K", [1, 5, 20, 24, 25, 50, 130, 200])
def test_matches_oracle_at_the_optimum(vb, K):
    case = _case(K, 3000 if K <= 50 else 40 * K, 1900 + K)
    model, obj, xo = _optimum(vb, case)
    assert model.perm is not None
    lr = vb.LinearResponseCovariances(obj, xo)
    oracle = make_oracle(case)
    Hinv = np.linalg.inv(oracle.kl_hessian_dense(xo))
    c = K // 2 if K % 2 else np.random.default_rng(K).standard_normal(K)
    order = np.argsort(case["g"], kind="stable")        # oracle row j is the caller's row order[j]

    def rows_to_caller(v):
        out = np.empty_like(v)
        out[order] = v
        return out

    ref = am.influences(oracle, xo, c, Hinv)
    # the device pass itself, at the oracle's a
    t, q = model.third_derivative_contraction(torch.from_numpy(ref["a"]).cuda())
    assert_close(t.cpu().numpy(), ref["t"], scale=np.abs(ref["t"]).max(), what="t K=%d" % K)
    assert_close(q.cpu().numpy(), rows_to_caller(ref["q"]), scale=np.abs(ref["q"]).max(), what="q K=%d" % K)
    for unit in ("row", "group"):
        got = lr.get_approximate_max_influence(c, unit=unit, max_fraction=0.5)
        r = am.approximate_max_influence(oracle, xo, c, unit=unit, max_fraction=0.5, Hinv=Hinv)
        assert_close(got.estimate, r["estimate"], what="estimate")
        assert_close(got.sd_lr, r["sd_lr"], what="sd_lr")
        assert got.z == r["z"]
        conv = rows_to_caller if unit == "row" else (lambda v: v)
        for f in ("mean_shift", "sd_shift"):
            v = getattr(got, f)
            assert isinstance(v, np.ndarray)
            assert_close(v, conv(r[f]), scale=np.abs(r[f]).max(), what="%s %s K=%d" % (f, unit, K))
        _check_drops(got, r["targets"], (lambda d: order[d]) if unit == "row" else (lambda d: d), "%s K=%d" % (unit, K))
        if unit == "row":
            assert np.all(got.mean_shift[case["w"] == 0] == 0) and np.all(got.sd_shift[case["w"] == 0] == 0)
        else:
            empty = np.bincount(case["g"], minlength=case["G"]) == 0
            assert np.all(got.mean_shift[empty] == 0) and np.all(got.sd_shift[empty] == 0)


@pytest.mark.timeout(900)
def test_mean_shift_matches_weight_sensitivity_and_logo(vb):
    case = make_case(N=4000, K=5, G=25, Q=6, seed=1950, shuffle=True, weights=True)
    model, obj, xo = _optimum(vb, case)
    lr = vb.LinearResponseCovariances(obj, xo)
    c = np.array([0.3, -1.0, 0.0, 2.0, 0.5])
    chat = np.zeros(model.D)
    chat[4:4 + model.K] = c
    rows = lr.get_approximate_max_influence(c, unit="row")
    infl = np.asarray(vb.WeightSensitivityLinearApproximation(obj, xo).get_dhyper_influence(chat))
    ref = -case["w"] * infl
    assert_close(rows.mean_shift, ref, scale=np.abs(ref).max(), what="row mean_shift")
    groups = lr.get_approximate_max_influence(c, unit="group")
    ref = lr.get_approximate_logo().delta_global[:, 4:4 + model.K] @ c
    assert_close(groups.mean_shift, ref, scale=np.abs(ref).max(), what="group mean_shift")


def _refit_case(N, K, G, seed):
    X, y, g = go.make_glmm_data(N, K, G, seed)
    return dict(X=X, y=y, g=g, w=None, gh_x=np.polynomial.hermite.hermgauss(8)[0],
                gh_w=np.polynomial.hermite.hermgauss(8)[1], G=G, K=K, N=N, free=go.make_free(4 + 2 * K + 2 * G, seed),
                bounds=0.0)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("unit,seed,G", [("row", 62, 12), ("row", 61, 12), ("group", 63, 20)])
def test_close_to_exact_refits(vb, unit, seed, G):
    """Every target the search reaches on the least significant coefficient of a 600-row model, refitted by device
    Newton with the selected rows' or groups' weights set to 0: |predicted - refit| <= 0.35 |refit - original| for
    the estimate and <= 0.55 for sd_lr.  Measured with these seeds (DESIGN.md 3e): estimate 0.31, 0.12, 0.33, 0.05
    and sd 0.47, 0.17, 0.51, 0.08 of the change; in each of these cases the refit moves further than the first-order
    step predicts."""
    case = _refit_case(600, 3, G, seed)
    model, obj, xo = _optimum(vb, case, gtol=1e-10)
    lr = vb.LinearResponseCovariances(obj, xo)
    sd = np.sqrt(np.diag(lr.get_global_covariance()))[4:7]
    k = int(np.argmin(np.abs(xo[4:7] / sd)))
    r = lr.get_approximate_max_influence(k, unit=unit, max_fraction=0.3 if unit == "group" else 0.1)
    reached = [d for d in r.targets.values() if d.n_drop is not None]
    assert reached
    for d in reached:
        w = np.ones(case["N"])
        w[d.dropped if unit == "row" else np.isin(case["g"], d.dropped)] = 0.0
        c2 = dict(case, w=w)
        m2, o2, x2 = _optimum(vb, c2, gtol=1e-10)
        est2 = x2[4 + k]
        sd2 = np.sqrt(vb.LinearResponseCovariances(o2, x2).get_global_covariance()[4 + k, 4 + k])
        assert abs(d.predicted_estimate - est2) <= 0.35 * abs(est2 - r.estimate), (d, est2)
        assert abs(d.predicted_sd - sd2) <= 0.55 * abs(sd2 - r.sd_lr), (d, sd2)


@pytest.fixture(scope="module")
def c2_optimum(vb):
    case = make_case(N=1_000_000, K=20, G=10_000, Q=8, seed=2300, shuffle=True)
    model, obj, xo = _optimum(vb, case)
    return case, model, obj, vb.LinearResponseCovariances(obj, xo), xo


@pytest.mark.timeout(900)
def test_c2_determinism_memory_and_types(vb, c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    for unit in ("row", "group"):
        a = lr.get_approximate_max_influence(3, unit=unit)
        torch.cuda.synchronize()
        mem = torch.cuda.memory_allocated()
        b = lr.get_approximate_max_influence(3, unit=unit)
        torch.cuda.synchronize()
        # nothing of the call stays allocated beyond its results
        assert torch.cuda.memory_allocated() - mem <= 8 * (2 * case["N"] + 2 * model.D) + (1 << 20)
        assert a.estimate == b.estimate and a.sd_lr == b.sd_lr
        for f in ("mean_shift", "sd_shift"):
            np.testing.assert_array_equal(getattr(a, f), getattr(b, f), err_msg=f)
            assert np.all(np.isfinite(getattr(a, f)))
        for name in am.TARGETS:
            assert a.targets[name].n_drop == b.targets[name].n_drop
            np.testing.assert_array_equal(a.targets[name].dropped, b.targets[name].dropped)
    model.evaluate(xo, 2)
    x = torch.from_numpy(np.random.default_rng(5).standard_normal(model.D)).cuda()
    t1, q1 = model.third_derivative_contraction(x)
    t2, q2 = model.third_derivative_contraction(x)
    assert torch.equal(t1, t2) and torch.equal(q1, q2)
    assert bool(torch.isfinite(t1).all()) and bool(torch.isfinite(q1).all())
    t = vb.LinearResponseCovariances(obj, torch.from_numpy(xo).cuda()).get_approximate_max_influence(3, unit="group")
    assert isinstance(t, vb.ApproximateMaxInfluence) and isinstance(t.targets["sign"], vb.DropResult)
    assert torch.is_tensor(t.mean_shift) and t.mean_shift.is_cuda
    np.testing.assert_array_equal(t.mean_shift.cpu().numpy(), b.mean_shift)


def test_errors(vb, tmp_path):
    case = make_case(N=600, K=6, G=8, Q=4, seed=13)
    model = make_model(vb, case)
    lr = vb.LinearResponseCovariances(vb.Objective(model.glmm_par, model), case["free"])
    for c in (6, -1, 2.0, True, np.zeros(6), np.ones(5), np.ones((6, 1)), [1, 2, np.nan, 0, 0, 0], "a"):
        with pytest.raises(ValueError):
            lr.get_approximate_max_influence(c)
    for kw in (dict(unit="rows"), dict(level=1.0), dict(level=0.0), dict(max_fraction=0.0),
               dict(max_fraction=1.5)):
        with pytest.raises(ValueError):
            lr.get_approximate_max_influence(0, **kw)
    with pytest.raises(ValueError):
        model.third_derivative_contraction(np.zeros(model.D + 1))

    import torch.distributed as dist
    from lrvb_b200.distributed import ShardedLogisticGLMM
    dist.init_process_group("gloo", init_method="file://" + str(tmp_path / "store"), rank=0, world_size=1)
    try:
        small = make_case(N=2000, K=3, G=10, Q=4, seed=11)
        sharded = ShardedLogisticGLMM.from_full(small["X"], small["y"], small["g"], small["G"], num_gh_points=4)
        obj = vb.Objective(sharded.glmm_par, sharded)
        with pytest.raises(NotImplementedError):
            sharded.third_derivative_contraction(None)
        with pytest.raises(NotImplementedError):
            vb.LinearResponseCovariances(obj, small["free"]).get_approximate_max_influence(0)
    finally:
        dist.destroy_process_group()


def test_c_abi_status_codes(vb):
    from lrvb_b200 import _native as nat
    case = make_case(N=600, K=6, G=8, Q=4, seed=12)
    model = make_model(vb, case)
    lib, h, st, P = model._lib, model._h, nat.stream_ptr(), nat.ptr
    a = torch.ones(model.D, dtype=torch.float64, device="cuda")
    t = torch.empty(model.D, dtype=torch.float64, device="cuda")
    q = torch.empty(model.N, dtype=torch.float64, device="cuda")

    def call(hh=h, aa=a, tt=t, qq=q):
        return lib.lrvb_glmm_third_contract(hh, P(aa), P(tt), P(qq), st)

    assert call() == nat.LRVB_ESTATE          # no evaluation yet
    model.evaluate(np.abs(case["free"]) + 1.0, 0, "vector")
    assert call() == nat.LRVB_ESTATE          # vector coordinates
    model.evaluate(case["free"], 0, "free")
    assert call() == nat.LRVB_OK
    assert call(hh=None) == nat.LRVB_EINVAL
    for kw in (dict(aa=None), dict(tt=None), dict(qq=None)):
        assert call(**kw) == nat.LRVB_EINVAL, kw
        assert "NULL" in nat.last_error()
    torch.cuda.synchronize()
