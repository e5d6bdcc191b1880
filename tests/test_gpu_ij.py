"""The infinitesimal-jackknife bootstrap covariance of the globals (LinearResponseCovariances.get_ij_covariance,
csrc/ij.cu lrvb_glmm_ij_meat): against the numpy oracle at the optimum for every Gram kernel class, against the row
shifts of the AMIP path and the group shifts of the LOGO path at C2 size, its determinism, that it leaves the cached
state alone, and its errors."""
import numpy as np
import pytest
import torch

from helpers import assert_close, make_case, make_model, make_oracle
from oracle import ij_oracle as ij

pytestmark = pytest.mark.gpu

FIELDS = ("global_cov", "moment_cov", "beta_cov", "beta_se_ij", "beta_se_lr")


def _optimum(vb, case, gtol=1e-7):
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=gtol)
    assert res.success, res.message
    return model, obj, xo


def _case(K, N, seed, bounds, G=30, empty=3):
    """The LOGO case mix: shuffled rows, ragged groups, `empty` groups without rows, weights with zeros and one group
    whose rows all have weight 0."""
    case = make_case(N=N, K=K, G=G, Q=8 if K % 2 else 4, seed=seed, shuffle=True, ragged=True, weights=True,
                     empty_groups=empty, bounds=bounds)
    rng = np.random.default_rng(seed + 1)
    case["w"][rng.choice(N, size=6, replace=False)] = 0.0
    sizes = np.bincount(case["g"], minlength=G)
    case["w"][case["g"] == int(np.nonzero(sizes > 0)[0][0])] = 0.0
    return case


# every k_gram_mid shape of K <= 24 (T2 = 1 .. 6), then k_gram_mid, k_gram_big and k_gram_wide
KS = [1, 4, 5, 8, 12, 16, 20, 24, 25, 50, 104, 130, 200]


@pytest.mark.timeout(900)
@pytest.mark.parametrize("K", KS)
def test_matches_oracle_at_the_optimum(vb, K):
    bounds = 0.05 if KS.index(K) % 2 else 0.0
    case = _case(K, 3000 if K <= 50 else 40 * K, 1900 + K, bounds)
    model, obj, xo = _optimum(vb, case)
    lr = vb.LinearResponseCovariances(obj, xo)
    oracle = make_oracle(case)
    Dg = model.Dg
    for unit in ("row", "group"):
        meat, s = model.ij_meat(unit)
        rm, rs = ij.meat_arrowhead(oracle, xo, unit)
        assert torch.equal(meat, meat.t()), unit
        assert_close(meat.cpu().numpy(), rm, scale=np.abs(rm).max(), what="meat %s K=%d" % (unit, K))
        assert_close(s.cpu().numpy(), rs, scale=np.abs(rs).max(), what="sum %s K=%d" % (unit, K))
        jac = model.moment_jacobian(xo)[:2 + K, :Dg].toarray()
        for centered in (True, False):
            got = lr.get_ij_covariance(unit, centered)
            ref = ij.ij_covariance_dense(oracle, xo, unit, centered)[:Dg, :Dg]
            assert got.unit == unit and got.n_units == ij.n_units(oracle, unit)
            want = dict(global_cov=ref, moment_cov=jac @ ref @ jac.T, beta_cov=ref[4:4 + K, 4:4 + K],
                        beta_se_ij=np.sqrt(np.diag(ref)[4:4 + K]),
                        beta_se_lr=np.sqrt(np.diag(np.linalg.inv(oracle.kl_hessian_dense(xo)))[4:4 + K]))
            for f in FIELDS:
                v = getattr(got, f)
                assert isinstance(v, np.ndarray) and v.shape == want[f].shape, f
                assert_close(v, want[f], scale=np.abs(want[f]).max(),
                             what="%s %s centered=%s K=%d" % (f, unit, centered, K))
            assert np.array_equal(got.global_cov, got.global_cov.T)


@pytest.fixture(scope="module")
def c2_optimum(vb):
    case = make_case(N=1_000_000, K=20, G=10_000, Q=8, seed=2300, shuffle=True, weights=True)
    case["w"][np.random.default_rng(1).choice(case["N"], size=1000, replace=False)] = 0.0
    model, obj, xo = _optimum(vb, case)
    return case, model, obj, vb.LinearResponseCovariances(obj, xo), xo


@pytest.mark.timeout(900)
def test_rows_match_the_amip_row_shifts_at_c2(c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    cov = lr.get_ij_covariance("row", centered=False)
    assert cov.n_units == case["N"] - 1000
    for c in (np.eye(model.K)[0], np.random.default_rng(2).standard_normal(model.K)):
        shift = lr.get_approximate_max_influence(c, "row").mean_shift
        assert_close(c @ cov.beta_cov @ c, np.sum(shift * shift), what="c^T beta_cov c")


@pytest.mark.timeout(900)
def test_groups_match_the_logo_shifts_at_c2(c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    cov = lr.get_ij_covariance("group", centered=False)
    d = lr.get_approximate_logo().delta_global
    ref = d.T @ d
    assert_close(cov.global_cov, ref, scale=np.abs(ref).max(), what="global_cov against delta^T delta")


def test_determinism_types_and_state_at_c2(vb, c2_optimum):
    case, model, obj, lr, xo = c2_optimum
    rng = np.random.default_rng(4)
    v = torch.from_numpy(rng.standard_normal(model.D)).cuda()
    rhs = torch.from_numpy(rng.standard_normal(model.D)).cuda()

    def state():
        h = lr.get_hessian_at_opt()
        out = [np.asarray(h.data), np.asarray(h.indices), np.asarray(h.indptr)]
        out += [model.hvp(v).cpu().numpy(), lr.hinv(rhs).cpu().numpy()]
        out += [np.asarray(f) for f in lr.get_approximate_loo()]
        out += [np.asarray(f) for f in lr.get_approximate_logo()]
        return out

    before = state()
    for unit in ("row", "group"):
        a, b = model.ij_meat(unit), model.ij_meat(unit)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), unit
        x, y = lr.get_ij_covariance(unit), lr.get_ij_covariance(unit)
        for f in FIELDS:
            np.testing.assert_array_equal(getattr(x, f), getattr(y, f), err_msg=f)
    after = state()
    for i, (p, q) in enumerate(zip(before, after)):
        np.testing.assert_array_equal(p, q, err_msg="state item %d" % i)
    t = vb.LinearResponseCovariances(obj, torch.from_numpy(xo).cuda()).get_ij_covariance("group")
    assert isinstance(t, vb.IJCovariance) and isinstance(t.n_units, int)
    for f in FIELDS:
        val = getattr(t, f)
        assert torch.is_tensor(val) and val.is_cuda, f
        np.testing.assert_array_equal(val.cpu().numpy(), getattr(x, f), err_msg=f)


def test_errors(vb, tmp_path):
    case = make_case(N=600, K=6, G=8, Q=4, seed=13, weights=True)
    model = make_model(vb, case)
    lr = vb.LinearResponseCovariances(vb.Objective(model.glmm_par, model), case["free"])
    with pytest.raises(ValueError, match="unit must be"):
        lr.get_ij_covariance("cluster")
    with pytest.raises(ValueError, match="unit must be"):
        model.ij_meat("rows")
    case["w"][:] = 0.0
    zero = make_model(vb, case)
    lz = vb.LinearResponseCovariances(vb.Objective(zero.glmm_par, zero), case["free"])
    for unit in ("row", "group"):
        with pytest.raises(ValueError, match="non-zero weight"):
            lz.get_ij_covariance(unit)

    import torch.distributed as dist
    from lrvb_b200.distributed import ShardedLogisticGLMM
    dist.init_process_group("gloo", init_method="file://" + str(tmp_path / "store"), rank=0, world_size=1)
    try:
        small = make_case(N=2000, K=3, G=10, Q=4, seed=11)
        sharded = ShardedLogisticGLMM.from_full(small["X"], small["y"], small["g"], small["G"], num_gh_points=4)
        obj = vb.Objective(sharded.glmm_par, sharded)
        with pytest.raises(NotImplementedError):
            sharded.ij_meat("row")
        with pytest.raises(NotImplementedError):
            vb.LinearResponseCovariances(obj, small["free"]).get_ij_covariance()
    finally:
        dist.destroy_process_group()


def test_c_abi_status_codes(vb):
    from lrvb_b200 import _native as nat
    case = make_case(N=600, K=6, G=8, Q=4, seed=12)
    model = make_model(vb, case)
    lib, h, st, P = model._lib, model._h, nat.stream_ptr(), nat.ptr
    meat = torch.empty(model.Dg, model.Dg, dtype=torch.float64, device="cuda")
    s = torch.empty(model.Dg, dtype=torch.float64, device="cuda")

    def call(hh=h, u=0, m=meat, v=s):
        return lib.lrvb_glmm_ij_meat(hh, u, P(m), P(v), st)

    assert call() == nat.LRVB_ESTATE          # no order-2 evaluation yet
    model.evaluate(case["free"], 1)
    assert call() == nat.LRVB_ESTATE          # order 1 caches no Hessian
    model.evaluate(case["free"], 2)
    assert call() == nat.LRVB_OK and call(u=1) == nat.LRVB_OK
    assert call(hh=None) == nat.LRVB_EINVAL
    assert call(u=2) == nat.LRVB_EINVAL and "unit" in nat.last_error()
    for kw in (dict(m=None), dict(v=None)):
        assert call(**kw) == nat.LRVB_EINVAL, kw
        assert "NULL" in nat.last_error()
    torch.cuda.synchronize()
