"""Timing of prediction on new rows (csrc/predict.cu) with CUDA events: lrvb_glmm_predict (MFVB outputs),
lrvb_glmm_predict_lr (the LR pass) and lrvb_glmm_predict_cross (the once-per-optimum precompute), each
warmed up and then the median of --reps launches; rows/s and, for the LR pass, the share of the DGEMM rate
bench.measure_dgemm_tflops measures in the same run, counting 4K^2 + 16K flops per row (the quadratic
form over beta and the cross terms).  Also times the factored path at M = 1M, K = 20
(prediction_jacobian -> get_lr_covariance_factors(J).diagonal()) and the end-to-end Python call.

    python tools/predict_time.py [--reps 10] [--out FILE]

The models are fitted by device Newton first (the LR pieces need a positive definite Hessian)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the measurement still stands; say what is missing
        return "unknown (%s)" % e


def events_median(torch, fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times)), float(np.min(times)), float(np.max(times))


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

    if not torch.cuda.is_available():
        raise SystemExit("predict_time.py needs the GPU")
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    dgemm = measure_dgemm_tflops(torch)
    emit(dict(card=card(), dgemm_tflops=dgemm))
    configs = [  # (K, M, fitted model: N, G)
        (20, 10_000_000, 200_000, 2_000),
        (50, 10_000_000, 100_000, 1_000),
        (200, 1_000_000, 20_000, 100),
    ]
    for K, M, N, G in configs:
        case = make_case(N=N, K=K, G=G, Q=8, seed=900 + K)
        model = make_model(vb, case)
        obj = vb.Objective(model.glmm_par, model)
        xo, res = vb.OptimizationUtils.minimize_objective_newton(obj, case["free"], maxiter=60, gtol=1e-7)
        lr = vb.LinearResponseCovariances(obj, xo)
        rng = np.random.default_rng(K)
        X = torch.from_numpy(0.7 * rng.standard_normal((M, K))).cuda()
        g = torch.from_numpy(rng.integers(-1, G, size=M)).cuda()
        g32 = g.to(torch.int32)
        order = torch.sort(g, stable=True)[1].contiguous()
        sinv = model.global_covariance()
        lcov = model.local_cov(sinv)
        cross = model.prediction_cross(sinv)
        out4 = torch.empty(4, M, dtype=torch.float64, device="cuda")
        out6 = torch.empty(6, M, dtype=torch.float64, device="cuda")
        lib, h, st = model._lib, model._h, nat.stream_ptr()
        xf = torch.from_numpy(np.asarray(xo, dtype=np.float64)).cuda()

        def f_pred():
            nat.check(lib.lrvb_glmm_predict(h, nat.ptr(xf), nat.ptr(X), K, nat.ptr(g32), None, M, nat.ptr(out4), st))

        def f_lr():
            nat.check(lib.lrvb_glmm_predict_lr(h, nat.ptr(sinv), nat.ptr(cross), nat.ptr(lcov), nat.ptr(X), K,
                                               nat.ptr(g32), nat.ptr(order), M, nat.ptr(out6), st))

        def f_lr_unsorted():
            nat.check(lib.lrvb_glmm_predict_lr(h, nat.ptr(sinv), nat.ptr(cross), nat.ptr(lcov), nat.ptr(X), K,
                                               nat.ptr(g32), None, M, nat.ptr(out6), st))

        def f_cross():
            nat.check(lib.lrvb_glmm_predict_cross(h, nat.ptr(sinv), nat.ptr(cross), st))

        def f_call():
            lr._pred_blocks = None
            lr.get_prediction_variances(X, g)

        tp = events_median(torch, f_pred, args.reps)
        tl = events_median(torch, f_lr, args.reps)
        tu = events_median(torch, f_lr_unsorted, args.reps)
        tc = events_median(torch, f_cross, args.reps)
        te = events_median(torch, f_call, args.reps)
        flops = (4.0 * K * K + 16.0 * K) * M
        emit(dict(K=K, M=M, G=G, newton_success=bool(res.success),
                  predict_ms=tp[0], predict_rows_per_s=M / (tp[0] * 1e-3),
                  predict_GBps=(M * (8 * K + 4) + 4 * 8 * M) / (tp[0] * 1e-3) / 1e9,
                  lr_ms=tl[0], lr_ms_min_max=tl[1:], lr_rows_per_s=M / (tl[0] * 1e-3),
                  lr_tflops=flops / (tl[0] * 1e-3) / 1e12, lr_share_of_dgemm=flops / (tl[0] * 1e-3) / 1e12 / dgemm,
                  lr_unsorted_ms=tu[0], cross_precompute_ms=tc[0], python_call_ms=te[0]))
        if K == 20:
            # the factored path on 1M of the rows: host Jacobian, then W = Jg - Jl T (M x Dg) and diag(W S^-1 W^T)
            Mf = 1_000_000
            Xh, gh = X[:Mf].cpu().numpy(), g[:Mf].cpu().numpy()
            tf = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                J = model.prediction_jacobian(xo, Xh, gh)
                t1 = time.perf_counter()
                lr.get_lr_covariance_factors(J).diagonal()
                t2 = time.perf_counter()
                tf.append((t1 - t0, t2 - t1))
            ti = events_median(torch, lambda: lr.get_prediction_variances(X[:Mf], g[:Mf]), args.reps)
            emit(dict(K=K, M=Mf, factored_jacobian_s=tf[-1][0], factored_diagonal_s=tf[-1][1],
                      factored_total_s=sum(tf[-1]), fused_python_call_ms=ti[0],
                      speedup=sum(tf[-1]) / (ti[0] * 1e-3)))
        del X, g, g32, order, out4, out6
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
