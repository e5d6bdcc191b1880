"""GPU parity of the weight cross-Hessian operator (SURVEY.md 8(f) rank 1): the CUDA products
C dw and C^T v against the CPU oracle.  KL is linear in the observation weights, so
C dw = grad KL(w + dw) - grad KL(w) exactly; the columns of C come from unit vectors."""
import numpy as np
import pytest

from helpers import assert_close, make_case, make_model
from oracle import glmm_oracle as go

pytestmark = pytest.mark.gpu

CASES = {
    "small_shuffled": dict(N=257, K=5, G=9, Q=6, seed=31, ragged=True, shuffle=True, weights=True),
    "k33_bounds": dict(N=300, K=33, G=7, Q=8, seed=32, bounds=0.05),
    "multistage": dict(N=70001, K=12, G=40, Q=4, seed=33, ragged=True),
    # K > 62: the wide-model observation kernel (lane = column dot products, transposing butterflies)
    "k80_wide": dict(N=903, K=80, G=10, Q=6, seed=34, weights=True, bounds=0.05),
    "k200_wide_ragged": dict(N=777, K=200, G=9, Q=8, seed=35, ragged=True),
    "k65_odd": dict(N=300, K=65, G=5, Q=5, seed=36),
    # the last K of the fused two-slot pass and the first of k_obs<1> + k_group<1> / k_obs_influence_wide
    "k62_fused_two_slot": dict(N=400, K=62, G=6, Q=8, seed=37, weights=True),
    "k63_obs_group": dict(N=400, K=63, G=6, Q=8, seed=38),
    # k_obs with one tile buffer (K >= 220) and the most quadrature nodes
    "k226_one_buffer_q64": dict(N=600, K=226, G=6, Q=64, seed=39, ragged=True),
}


def _oracle(case, w):
    order = np.argsort(case["g"], kind="stable")
    b = case["bounds"]
    return go.GLMMOracle(case["X"][order], case["y"][order], case["g"][order], case["gh_x"],
                         case["gh_w"], weights=w[order], G=case["G"], bounds=go.GLMMBounds(b, b, b, b, b))


@pytest.fixture(scope="module", params=sorted(CASES))
def setup(request, vb):
    case = make_case(**CASES[request.param])
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    return case, model, obj


def test_matvec_is_the_gradient_difference(setup):
    case, model, obj = setup
    x, N = case["free"], case["N"]
    w0 = np.ones(N) if case["w"] is None else case["w"]
    rng = np.random.default_rng(3)
    dw = rng.standard_normal(N)
    obj.fun_free_grad(x)
    got = model.weight_cross_matvec(dw).cpu().numpy()
    ref = _oracle(case, w0 + dw).kl_grad(x) - _oracle(case, w0).kl_grad(x)
    assert_close(got, ref, scale=np.abs(ref).max() * 1e-3, what="C dw")


def test_rmatvec_matches_columns_of_c(setup):
    case, model, obj = setup
    x, N = case["free"], case["N"]
    rng = np.random.default_rng(4)
    v = rng.standard_normal(x.size)
    obj.fun_free(x)
    got = model.weight_cross_rmatvec(v).cpu().numpy()
    assert got.shape == (N,)
    w0 = np.ones(N) if case["w"] is None else case["w"]
    g0 = _oracle(case, w0).kl_grad(x)
    idx = rng.choice(N, size=min(N, 12), replace=False)
    for n in idx:
        e = np.zeros(N)
        e[n] = 1.0
        col = _oracle(case, w0 + e).kl_grad(x) - g0          # column n of C
        assert abs(got[n] - col @ v) <= 1e-12 + 1e-9 * max(abs(col @ v), np.abs(col).max())
    # adjointness of the two device products
    dw = rng.standard_normal(N)
    lhs = float(model.weight_cross_matvec(dw).cpu().numpy() @ v)
    rhs = float(got @ dw)
    assert abs(lhs - rhs) <= 1e-9 * max(1.0, abs(lhs))


def test_linear_approximation_of_the_optimum(setup, vb):
    case, model, obj = setup
    if case["N"] > 1000:
        pytest.skip("dense reference solve only for small cases")
    x, N = case["free"], case["N"]
    w0 = np.ones(N) if case["w"] is None else case["w"]
    Hd = _oracle(case, w0).kl_hessian_dense(x)
    if np.linalg.eigvalsh(Hd).min() <= 0:
        pytest.skip("Hessian not PD at this (non-optimal) point")
    sens = vb.WeightSensitivityLinearApproximation(obj, x)
    rng = np.random.default_rng(5)
    dw = 0.1 * rng.standard_normal(N)
    cdw = _oracle(case, w0 + dw).kl_grad(x) - _oracle(case, w0).kl_grad(x)
    ref = -np.linalg.solve(Hd, cdw)
    got = sens.get_dinput_dhyper_times(dw)
    assert_close(got, ref, rtol=1e-8, scale=np.abs(ref).max() * 1e-3, what="dinput/dhyper dw")
    pred = sens.predict_input_par_from_hyperparameters(w0 + dw)
    assert_close(pred, x + ref, rtol=1e-8, scale=np.abs(x).max() * 1e-3, what="prediction")
    v = rng.standard_normal(x.size)
    infl = sens.get_dhyper_influence(v)
    assert abs(float(infl @ dw) - float(v @ ref)) <= 1e-8 * max(1.0, abs(float(v @ ref)))
    if x.size * N <= 40000:
        S = sens.get_dinput_dhyper()
        assert S.shape == (x.size, N)
        assert_close(S @ dw, ref, rtol=1e-8, scale=np.abs(ref).max() * 1e-3, what="dense S dw")
