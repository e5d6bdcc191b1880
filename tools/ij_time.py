"""Timing of the infinitesimal-jackknife bootstrap covariance (lrvb_glmm_ij_meat, csrc/ij.cu): CUDA-event medians of
the device call for rows and for groups, of lrvb_glmm_logo and of an order-2 evaluation of the same model (three
alternating rounds), the per-kernel medians of the row call from torch.profiler with the IJ Gram kernel's share of the
DGEMM rate bench.measure_dgemm_tflops measures, the Python call, the card's name and power limit and, at C2, the
per-unit reference path (``get_dinput_dhyper_times`` with one row's or one group's weight dropped) extrapolated to N
and G.

    python tools/ij_time.py [--reps 10] [--out FILE]

The models are fitted by device Newton first; where Newton stops short (C3) the last iterate is timed, with the
Levenberg damping of minimize_objective_newton on the cached Hessian if S is not positive definite there."""
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


def kernel_medians(torch, fn, reps):
    """Median device time (ms) per kernel name of `fn` over `reps` calls, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    by = {}
    for e in prof.events():
        if e.device_type.name != "CUDA" or "Memset" in e.name or "Memcpy" in e.name:
            continue
        key = e.name.split("(")[0].split("<")[0].replace("void ", "").replace("lrvb::", "")
        by.setdefault(key, []).append(e.time_range.elapsed_us())
    return {k: float(np.median(v)) * 1e-3 * (len(v) / reps) for k, v in by.items()}


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
        raise SystemExit("ij_time.py needs the GPU")
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
        xd = torch.from_numpy(np.asarray(xo)).cuda()
        lr = vb.LinearResponseCovariances(obj, xd)
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
        Dg = model.Dg
        meat = torch.empty(Dg, Dg, dtype=torch.float64, device="cuda")
        s = torch.empty(Dg, dtype=torch.float64, device="cuda")
        delta = torch.empty(G, Dg, dtype=torch.float64, device="cuda")
        grp = torch.empty(2, G, dtype=torch.float64, device="cuda")
        out = torch.empty(3, N, dtype=torch.float64, device="cuda")
        lib, h, st = model._lib, model._h, nat.stream_ptr()

        def f_row():
            nat.check(lib.lrvb_glmm_ij_meat(h, 0, nat.ptr(meat), nat.ptr(s), st))

        def f_group():
            nat.check(lib.lrvb_glmm_ij_meat(h, 1, nat.ptr(meat), nat.ptr(s), st))

        def f_logo():
            nat.check(lib.lrvb_glmm_logo(h, nat.ptr(sinv), nat.ptr(pinv), nat.ptr(delta), nat.ptr(grp), nat.ptr(out),
                                         st))

        def f_eval():      # an order-2 evaluation at the same point (replaces a damped Hessian by the undamped one)
            nat.check(lib.lrvb_glmm_eval(h, nat.ptr(xd), 2, None, None, st))

        # the Python calls first: they compute S^-1 from the cached (possibly damped) Hessian, which f_eval replaces
        py_row = events_median(torch, lambda: lr.get_ij_covariance("row"), args.reps)[0]
        py_group = events_median(torch, lambda: lr.get_ij_covariance("group"), args.reps)[0]
        runs = dict(row=[], group=[], logo=[], eval=[])
        for _ in range(3):
            runs["row"].append(events_median(torch, f_row, args.reps)[0])
            runs["group"].append(events_median(torch, f_group, args.reps)[0])
            runs["logo"].append(events_median(torch, f_logo, args.reps)[0])
            runs["eval"].append(events_median(torch, f_eval, args.reps)[0])
        kern = kernel_medians(torch, f_row, args.reps)
        gram = {k: v for k, v in kern.items() if k.startswith("k_gram_")}
        gram_ms = sum(gram.values())
        flops = 2.0 * N * (2 * K) * (2 * K + 1) / 2.0       # the packed upper triangle, as the evaluation's Gram
        med = {k: float(np.median(v)) for k, v in runs.items()}
        t_eval = med["eval"]
        d = dict(config=name, N=N, K=K, G=G, newton_success=bool(res.success), newton_iterations=int(res.nit),
                 grad_inf_norm=float(res.grad_inf_norm), hessian_damping=damping,
                 row_ms=med["row"], group_ms=med["group"], logo_ms=med["logo"], eval_order2_ms=t_eval,
                 runs_ms=runs, row_over_eval=med["row"] / t_eval,
                 group_over_logo=med["group"] / med["logo"], row_kernels_ms=kern, gram_ms=gram_ms,
                 gram_tflops=flops / (gram_ms * 1e-3) / 1e12 if gram_ms else None,
                 gram_share_of_dgemm=flops / (gram_ms * 1e-3) / 1e12 / dgemm if gram_ms else None,
                 python_row_ms=py_row, python_group_ms=py_group)
        if name == "C2":
            # the per-unit reference path: one weight cross-Hessian product and one H^-1 solve per unit
            ws = vb.WeightSensitivityLinearApproximation(obj, xo)
            gs = np.sort(case["g"])
            tr, tg = [], []
            for u in range(4):
                for which, ts in ((np.arange(N) == u, tr), (gs == u, tg)):
                    diff = np.where(which, -1.0, 0.0)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    ws.get_dinput_dhyper_times(diff)
                    torch.cuda.synchronize()
                    ts.append(time.perf_counter() - t0)
            pr, pg = float(np.median(tr[1:])), float(np.median(tg[1:]))
            d.update(per_row_reference_s=pr, per_row_reference_extrapolated_s=pr * N,
                     per_group_reference_s=pg, per_group_reference_extrapolated_s=pg * G)
        emit(d)
        del meat, s, delta, grp, out, model, obj, lr, sinv, pinv
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
