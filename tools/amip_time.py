"""Timing of the approximate maximum influence perturbation (LinearResponseCovariances.get_approximate_max_influence,
csrc/amip.cu lrvb_glmm_third_contract): CUDA-event medians of the whole Python call for rows and for groups, of the
approximate-LOO call on the same model (the yardstick), and of the device pass lrvb_glmm_third_contract alone, with
the median of its row kernel k_amip_rows from torch.profiler in a separate window and that kernel's share of the HBM
peak (7.7 TB/s) on the bytes it must read and write: X, the group ids, the weights, q and the two row coefficients.
Also the card's name and power limit.

    python tools/amip_time.py [--reps 10] [--out FILE]

The C2, C3 and K = 200 models are fitted by device Newton first: the call reads the Hessian of the optimum."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM_TBS = 7.7


def kernel_median(torch, fn, reps, name):
    """Median device time (ms) of kernel `name` over `reps` calls of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    return float(np.median([e.time_range.elapsed_us() for e in prof.events() if name in e.name])) * 1e-3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import lrvb_b200 as vb
    from lrvb_b200 import _native as nat
    from helpers import make_case, make_model
    from predict_time import card, events_median

    if not torch.cuda.is_available():
        raise SystemExit("amip_time.py needs the GPU")
    lines = []

    def emit(d):
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    emit(dict(card=card()))
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
        # minimize_objective_newton on the cached Hessian if S is not positive definite there (as tools/logo_time.py).
        damping = 0.0
        while True:
            try:
                model.global_covariance()
                break
            except np.linalg.LinAlgError:
                lam = 1e-3 * model.max_abs_diagonal() if damping == 0.0 else 9.0 * damping
                model.add_diagonal_(lam)
                damping += lam
        lr.get_approximate_loo()
        r_row = lr.get_approximate_max_influence(0, unit="row")
        r_grp = lr.get_approximate_max_influence(0, unit="group")
        a = torch.from_numpy(np.random.default_rng(seed).standard_normal(model.D)).cuda()
        t = torch.empty(model.D, dtype=torch.float64, device="cuda")
        q = torch.empty(N, dtype=torch.float64, device="cuda")
        lib, h, st = model._lib, model._h, nat.stream_ptr()

        def f_pass():
            nat.check(lib.lrvb_glmm_third_contract(h, nat.ptr(a), nat.ptr(t), nat.ptr(q), st))

        def f_row():
            lr.get_approximate_max_influence(0, unit="row")

        def f_grp():
            lr.get_approximate_max_influence(0, unit="group")

        # alternate the calls so that all see the same state of the card
        runs = dict(row=[], group=[], loo=[], pass_=[])
        for _ in range(3):
            runs["row"].append(events_median(torch, f_row, args.reps)[0])
            runs["group"].append(events_median(torch, f_grp, args.reps)[0])
            runs["loo"].append(events_median(torch, lr.get_approximate_loo, args.reps)[0])
            runs["pass_"].append(events_median(torch, f_pass, args.reps)[0])
        med = {k: float(np.median(v)) for k, v in runs.items()}
        k_rows = kernel_median(torch, f_pass, args.reps, "k_amip_rows")
        nbytes = 8.0 * N * K + 4.0 * N + 8.0 * N + 8.0 * N + 16.0 * N
        emit(dict(config=name, N=N, K=K, G=G, newton_success=bool(res.success), newton_iterations=int(res.nit),
                  grad_inf_norm=float(res.grad_inf_norm), hessian_damping=damping,
                  amip_row_call_ms=med["row"], amip_group_call_ms=med["group"], loo_call_ms=med["loo"],
                  row_over_loo=med["row"] / med["loo"], group_over_loo=med["group"] / med["loo"],
                  third_contract_ms=med["pass_"], k_amip_rows_ms=k_rows,
                  k_amip_rows_hbm_share=nbytes / (k_rows * 1e-3) / (HBM_TBS * 1e12),
                  runs_ms={k: v for k, v in runs.items()},
                  estimate=r_row.estimate, sd_lr=r_row.sd_lr,
                  n_drop_row={k: v.n_drop for k, v in r_row.targets.items()},
                  n_drop_group={k: v.n_drop for k, v in r_grp.targets.items()}))
        del model, obj, lr, a, t, q
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
