"""Timing of approximate leave-one-out cross-validation (lrvb_glmm_loo, csrc/predict.cu) with CUDA events, next to
lrvb_glmm_predict_lr over the same rows (the model's own group-sorted training X) in the same run: the median of
--reps launches after a warm-up, their ratio, rows/s and the share of the DGEMM rate bench.measure_dgemm_tflops
measures in the same run, counting 4K^2 + 16K flops per row as tools/predict_time.py does.  Also the end-to-end
``LinearResponseCovariances.get_approximate_loo`` call and, at C2, the per-row reference path
(``WeightSensitivityLinearApproximation.get_dinput_dhyper_times`` on a few rows) extrapolated to N.

    python tools/loo_time.py [--reps 10] [--out FILE]

The models are fitted by device Newton first: the pass reads the Hessian and W of the optimum."""
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
        raise SystemExit("loo_time.py needs the GPU")
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    dgemm = measure_dgemm_tflops(torch)
    emit(dict(card=card(), dgemm_tflops=dgemm))
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
        # Where Newton stops short of gtol (C3, N = 10M, G = 100k: |grad| ~ 10 after 400 steps), the last iterate is timed, with the
        # Levenberg damping of minimize_objective_newton on the cached Hessian if S is not positive definite there.
        # The pass reads and computes the same either way; the record says which point was timed.
        damping = 0.0
        while True:
            try:
                sinv = model.global_covariance()
                break
            except np.linalg.LinAlgError:
                lam = 1e-3 * model.max_abs_diagonal() if damping == 0.0 else 9.0 * damping
                model.add_diagonal_(lam)
                damping += lam
        lcov = model.local_cov(sinv)
        cross = model.prediction_cross(sinv)
        out4 = torch.empty(4, N, dtype=torch.float64, device="cuda")
        out6 = torch.empty(6, N, dtype=torch.float64, device="cuda")
        lib, h, st = model._lib, model._h, nat.stream_ptr()

        def f_loo():
            nat.check(lib.lrvb_glmm_loo(h, nat.ptr(sinv), nat.ptr(cross), nat.ptr(lcov), nat.ptr(out4), st))

        def f_lr():   # the same rows, already group-sorted: no visiting order needed
            nat.check(lib.lrvb_glmm_predict_lr(h, nat.ptr(sinv), nat.ptr(cross), nat.ptr(lcov), nat.ptr(model.X), K,
                                               nat.ptr(model.g), None, N, nat.ptr(out6), st))

        # alternate the two kernels so that both see the same state of the card
        tl, tp = [], []
        for _ in range(3):
            tl.append(events_median(torch, f_loo, args.reps))
            tp.append(events_median(torch, f_lr, args.reps))
        t_loo = float(np.median([t[0] for t in tl]))
        t_lr = float(np.median([t[0] for t in tp]))
        r = lr.get_approximate_loo()
        te = events_median(torch, lr.get_approximate_loo, args.reps)
        flops = (4.0 * K * K + 16.0 * K) * N
        d = dict(config=name, N=N, K=K, G=G, newton_success=bool(res.success), newton_iterations=int(res.nit),
                 grad_inf_norm=float(res.grad_inf_norm), hessian_damping=damping,
                 loo_ms=t_loo, loo_ms_runs=[t[0] for t in tl], predict_lr_ms=t_lr, predict_lr_ms_runs=[t[0] for t in tp],
                 loo_over_predict_lr=t_loo / t_lr, loo_rows_per_s=N / (t_loo * 1e-3),
                 loo_tflops=flops / (t_loo * 1e-3) / 1e12, loo_share_of_dgemm=flops / (t_loo * 1e-3) / 1e12 / dgemm,
                 predict_lr_share_of_dgemm=flops / (t_lr * 1e-3) / 1e12 / dgemm,
                 python_call_ms=te[0], elpd_loo=r.elpd_loo, p_loo=r.p_loo, n_invalid=r.n_invalid)
        if name == "C2":
            # the per-row reference path: one weight cross-Hessian product and one H^-1 solve per dropped row
            ws = vb.WeightSensitivityLinearApproximation(obj, xo)
            w = np.zeros(N)
            ts = []
            for n in range(4):
                w[:] = 0.0
                w[n] = -1.0
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ws.get_dinput_dhyper_times(w)
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            per_row = float(np.median(ts[1:]))
            d.update(per_row_reference_s=per_row, per_row_reference_extrapolated_s=per_row * N,
                     speedup_over_per_row=per_row * N / (te[0] * 1e-3))
        emit(d)
        del out4, out6, model, obj, lr, sinv, lcov, cross
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
