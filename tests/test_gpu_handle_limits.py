"""Kernel launch limits are properties of the library, not of one handle: the dynamic shared-memory limit of a
kernel belongs to the kernel on a device and is shared by every model there.  Models of different widths in one
process, created one after the other, must keep computing what they computed alone; a model on a second device must
compute what the same model computes on the first; and every kernel of the library is compiled exactly once."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import make_case, make_model

# K = 200: k_obs (about 205 KB of shared memory) and k_gram_wide; K = 50: k_obs_fused, k_gram_mid and a CSR export
# above 48 KB; K = 5: the one-pass order-2 kernel.  The wider models need the larger limits and are created first.
WIDTHS = (200, 50, 5)
FULL = (200, 50)      # the on-demand passes: weight cross products, LR prediction, LOO, LOGO


def _case(K):
    return make_case(N=20000, K=K, G=300, Q=8, seed=900 + K, weights=True, shuffle=True)


def _host(v):
    """A tensor, array or scalar result as a host array of its own."""
    import torch
    return v.detach().cpu().numpy().copy() if torch.is_tensor(v) else np.array(v)


def _fit(vb, case):
    model = make_model(vb, case)
    obj = vb.Objective(model.glmm_par, model)
    xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=1e-7)
    assert res.success, res.message
    return model, xo


def _record(model, xo, case, full):
    """Everything the model computes at xo, as host arrays; the evaluation is forced to run again."""
    model.evaluate(xo, 2, force=True)
    A, B, L = model.blocks()
    r = dict(kl=_host(model.kl_tensor()), grad=_host(model.grad_tensor()), A=_host(A), B=_host(B), L=_host(L))
    csr = model.hessian_csr()
    r.update(csr_values=_host(csr.values), csr_col=_host(csr.col_indices), csr_crow=_host(csr.crow_indices))
    if full:
        rng = np.random.default_rng(case["K"])
        r["wc_matvec"] = _host(model.weight_cross_matvec(rng.standard_normal(case["N"])))
        r["wc_rmatvec"] = _host(model.weight_cross_rmatvec(rng.standard_normal(model.D)))
        Sinv = model.global_covariance()
        cross, lcov = model.prediction_cross(Sinv), model.local_cov(Sinv)
        Xp, gp = rng.standard_normal((500, case["K"])), rng.integers(0, case["G"], size=500)
        results = dict(predict=model.predict_lr(Sinv, cross, lcov, Xp, gp),
                       loo=model.approximate_loo(Sinv, cross, lcov), logo=model.approximate_logo(Sinv))
        for name, res in results.items():
            for f in res._fields:
                r["%s_%s" % (name, f)] = _host(getattr(res, f))
    return r


def _assert_bitwise_equal(got, ref, what):
    assert got.keys() == ref.keys(), what
    for k in ref:
        a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(ref[k])
        assert a.shape == b.shape and a.tobytes() == b.tobytes(), "%s: %s differs" % (what, k)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_later_handles_keep_earlier_handles_running(vb):
    models, records = {}, {}
    for K in WIDTHS:
        case = _case(K)
        model, xo = _fit(vb, case)
        models[K] = (model, xo, case)
        records[K] = _record(model, xo, case, K in FULL)
    for K in reversed(WIDTHS):
        model, xo, case = models[K]
        _assert_bitwise_equal(_record(model, xo, case, K in FULL), records[K], "K = %d" % K)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_second_device_computes_what_the_first_does(vb):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    case = _case(50)
    got = []
    for dev in (0, 1):
        with torch.cuda.device(dev):
            model, xo = _fit(vb, case)
            Sinv = model.global_covariance()
            cross, lcov = model.prediction_cross(Sinv), model.local_cov(Sinv)
            rng = np.random.default_rng(7)
            pred = model.predict_lr(Sinv, cross, lcov, rng.standard_normal((500, 50)), rng.integers(0, 300, 500))
            logo = model.approximate_logo(Sinv)
            got.append(dict(xo=_host(xo), prob_var_lr=_host(pred.prob_var_lr), eta_var_lr=_host(pred.eta_var_lr),
                            lpd_logo=_host(logo.lpd_logo), delta_global=_host(logo.delta_global),
                            elpd_logo=_host(logo.elpd_logo)))
    _assert_bitwise_equal(got[1], got[0], "device 1 against device 0")


def test_every_kernel_is_compiled_once():
    from lrvb_b200 import _native as nat
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(nat.LIB_PATH) or not os.path.exists(cuobjdump):
        pytest.skip("needs the built library and cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", nat.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = [line.split("Function :", 1)[1].strip() for line in sass.splitlines() if "Function :" in line]
    assert len(names) > 100
    twice = sorted({n for n in names if names.count(n) > 1})
    assert not twice, "kernels compiled in more than one object: %s" % twice
