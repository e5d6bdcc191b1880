"""Timing of approximate leave-one-group-out cross-validation (lrvb_glmm_logo, csrc/logo.cu): CUDA-event medians of
the whole device call and, from torch.profiler in a separate window, the medians of its three passes (k_logo_grad,
the two k_logo_gemm products, k_logo_rows).  In the same run: lrvb_glmm_loo on the same model, the DGEMM rate
bench.measure_dgemm_tflops measures, the rate of the Delta = -V S^-1 product at C4's shape (G = 100k, Dg = 404), the
card's name and power limit and, at C2, the per-group reference path (``get_dinput_dhyper_times`` with one group's
weights dropped) extrapolated to G.

    python tools/logo_time.py [--reps 10] [--out FILE]

The C2, C3 and K = 200 models are fitted by device Newton first: the passes read the Hessian and W of the optimum."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def pass_medians(torch, fn, reps):
    """Median device time (ms) of each pass of lrvb_glmm_logo over `reps` calls, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    ev = sorted((e.time_range.start, e.name, e.time_range.elapsed_us()) for e in prof.events() if "k_logo_" in e.name)
    gemm = [t for _, n, t in ev if "k_logo_gemm" in n]
    out = dict(grad=[t for _, n, t in ev if "k_logo_grad" in n], gemm_delta=gemm[0::2], gemm_cook=gemm[1::2],
               rows=[t for _, n, t in ev if "k_logo_rows" in n])
    return {k: float(np.median(v)) * 1e-3 for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import lrvb_b200 as vb
    from lrvb_b200 import _native as nat
    from bench import measure_dgemm_tflops
    from helpers import make_case, make_model
    from predict_time import card, events_median

    if not torch.cuda.is_available():
        raise SystemExit("logo_time.py needs the GPU")
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    dgemm = measure_dgemm_tflops(torch)
    emit(dict(card=card(), dgemm_tflops=dgemm))

    def buffers(model):
        return (torch.empty(model.G, model.Dg, dtype=torch.float64, device="cuda"),
                torch.empty(2, model.G, dtype=torch.float64, device="cuda"),
                torch.empty(3, model.N, dtype=torch.float64, device="cuda"))

    # the Delta = -V S^-1 product at C4's shape: an order-2 evaluation and a small SPD S^-1 (the rate does not depend
    # on the values)
    case = make_case(N=1_000_000, K=200, G=100_000, Q=8, seed=5500)
    model = make_model(vb, case)
    del case["X"]
    model.evaluate(case["free"], 2)
    sinv = 1e-6 * torch.eye(model.Dg, dtype=torch.float64, device="cuda")
    pinv = torch.eye(model.K, dtype=torch.float64, device="cuda")
    delta, grp, out = buffers(model)
    lib, h, st = model._lib, model._h, nat.stream_ptr()

    def f_c4():
        nat.check(lib.lrvb_glmm_logo(h, nat.ptr(sinv), nat.ptr(pinv), nat.ptr(delta), nat.ptr(grp), nat.ptr(out), st))

    p = pass_medians(torch, f_c4, args.reps)
    flops = 2.0 * model.G * model.Dg * model.Dg
    emit(dict(config="C4-shape product", G=model.G, Dg=model.Dg, gemm_delta_ms=p["gemm_delta"],
              gemm_delta_tflops=flops / (p["gemm_delta"] * 1e-3) / 1e12,
              gemm_delta_share_of_dgemm=flops / (p["gemm_delta"] * 1e-3) / 1e12 / dgemm, passes_ms=p))
    del model, delta, grp, out, sinv, pinv
    torch.cuda.empty_cache()

    configs = [  # (name, N, K, G, seed)
        ("C2", 1_000_000, 20, 10_000, 2200),
        ("C3", 10_000_000, 50, 100_000, 3300),
        ("K200", 1_000_000, 200, 1_000, 4400),
    ]
    for name, N, K, G, seed in configs:
        case = make_case(N=N, K=K, G=G, Q=8, seed=seed)
        model = make_model(vb, case)
        del case["X"]
        obj = vb.Objective(model.glmm_par, model)
        xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=400, gtol=1e-7)
        lr = vb.LinearResponseCovariances(obj, xo)
        # Where Newton stops short of gtol (C3), the last iterate is timed, with the Levenberg damping of
        # minimize_objective_newton on the cached Hessian if S is not positive definite there (as tools/loo_time.py).
        damping = 0.0
        while True:
            try:
                sinv = model.global_covariance()
                break
            except np.linalg.LinAlgError:
                lam = 1e-3 * model.max_abs_diagonal() if damping == 0.0 else 9.0 * damping
                model.add_diagonal_(lam)
                damping += lam
        pinv = model.spd_inverse_(sinv[4:4 + K, 4:4 + K].clone())
        lcov = model.local_cov(sinv)
        cross = model.prediction_cross(sinv)
        delta, grp, out = buffers(model)
        out4 = torch.empty(4, N, dtype=torch.float64, device="cuda")
        lib, h, st = model._lib, model._h, nat.stream_ptr()

        def f_logo():
            nat.check(lib.lrvb_glmm_logo(h, nat.ptr(sinv), nat.ptr(pinv), nat.ptr(delta), nat.ptr(grp), nat.ptr(out),
                                         st))

        def f_loo():
            nat.check(lib.lrvb_glmm_loo(h, nat.ptr(sinv), nat.ptr(cross), nat.ptr(lcov), nat.ptr(out4), st))

        # alternate the two so that both see the same state of the card
        tg, tl = [], []
        for _ in range(3):
            tg.append(events_median(torch, f_logo, args.reps))
            tl.append(events_median(torch, f_loo, args.reps))
        t_logo = float(np.median([t[0] for t in tg]))
        t_loo = float(np.median([t[0] for t in tl]))
        p = pass_medians(torch, f_logo, args.reps)
        flops = 2.0 * G * model.Dg * model.Dg
        r = lr.get_approximate_logo()
        te = events_median(torch, lr.get_approximate_logo, args.reps)
        d = dict(config=name, N=N, K=K, G=G, newton_success=bool(res.success), newton_iterations=int(res.nit),
                 grad_inf_norm=float(res.grad_inf_norm), hessian_damping=damping,
                 logo_ms=t_logo, logo_ms_runs=[t[0] for t in tg], loo_ms=t_loo, loo_ms_runs=[t[0] for t in tl],
                 logo_over_loo=t_logo / t_loo, passes_ms=p,
                 gemm_delta_tflops=flops / (p["gemm_delta"] * 1e-3) / 1e12,
                 gemm_delta_share_of_dgemm=flops / (p["gemm_delta"] * 1e-3) / 1e12 / dgemm,
                 python_call_ms=te[0], elpd_logo=r.elpd_logo, elpd_logo_se=r.elpd_logo_se)
        if name == "C2":
            # the per-group reference path: one weight cross-Hessian product and one H^-1 solve per dropped group
            ws = vb.WeightSensitivityLinearApproximation(obj, xo)
            gs = np.sort(case["g"])
            ts = []
            for g in range(4):
                diff = np.where(gs == g, -1.0, 0.0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ws.get_dinput_dhyper_times(diff)
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            per_group = float(np.median(ts[1:]))
            d.update(per_group_reference_s=per_group, per_group_reference_extrapolated_s=per_group * G,
                     speedup_over_per_group=per_group * G / (te[0] * 1e-3))
        emit(d)
        del out4, delta, grp, out, model, obj, lr, sinv, pinv, lcov, cross
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
