"""Timing of the Poisson GLMM evaluation beside the logistic one on the same X: CUDA-event medians of an order-2
evaluation of each (alternating rounds), and k_obs_pois alone (the observation-pass events of lrvb_glmm_set_timing)
as a fraction of the HBM peak, with its bytes counted from the shapes.  C2 (N = 1M, K = 20, G = 10k) and C3
(N = 10M, K = 50, G = 100k), logistic with Q = 8 as in bench.py; the data are generated on the device.

    python tools/poisson_time.py [--reps 20] [--rounds 3] [--out profiles/r08_poisson_time.jsonl]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM_PEAK = 7.7e12      # bytes/s, HGX B200 data sheet, one GPU
CONFIGS = {"C2": dict(N=1_000_000, K=20, G=10_000), "C3": dict(N=10_000_000, K=50, G=100_000)}


def obs_pois_bytes(N, K, order=2):
    """DRAM bytes k_obs_pois must move at order 2 without weights or offset: X, y, g read, rows 0-4 of W written."""
    return N * (8 * K + 8 + 4) + N * 8 * (5 if order >= 2 else 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_poisson_time.jsonl"))
    args = ap.parse_args()
    import ctypes
    import torch
    import lrvb_b200 as vb
    from lrvb_b200 import _native as nat
    from predict_time import card, events_median

    if not torch.cuda.is_available():
        raise SystemExit("poisson_time.py needs the GPU")
    gpu = card()
    lines = []
    for name, c in CONFIGS.items():
        N, K, G = c["N"], c["K"], c["G"]
        gen = torch.Generator(device="cuda").manual_seed(8)
        X = torch.randn(N, K, dtype=torch.float64, device="cuda", generator=gen) / np.sqrt(K)
        g = torch.arange(N, device="cuda") * G // N
        eta = X @ (0.3 * torch.randn(K, dtype=torch.float64, device="cuda", generator=gen))
        y_cnt = torch.poisson(torch.exp(eta), generator=gen)
        y_bin = torch.bernoulli(torch.sigmoid(eta), generator=gen)
        pm = vb.PoissonGLMM(X, y_cnt, g, num_groups=G)
        lm = vb.LogisticGLMM(X, y_bin, g, num_gh_points=8, num_groups=G)
        x = (0.1 * torch.randn(pm.D, dtype=torch.float64, device="cuda", generator=gen)).contiguous()
        res = {"pois": [], "logit": [], "obs_pois": []}
        for _ in range(args.rounds):
            for key, m in (("pois", pm), ("logit", lm)):
                res[key].append(events_median(torch, lambda m=m: m.evaluate(x, 2, force=True), args.reps)[0])
            nat.check(pm._lib.lrvb_glmm_set_timing(pm._h, 1))
            ms = []
            for _ in range(args.reps):
                pm.evaluate(x, 2, force=True)
                ms3 = (ctypes.c_float * 3)()
                nat.check(pm._lib.lrvb_glmm_last_timing(pm._h, ms3))
                ms.append(ms3[1])
            nat.check(pm._lib.lrvb_glmm_set_timing(pm._h, 0))
            res["obs_pois"].append(float(np.median(ms)))
        t_obs = float(np.median(res["obs_pois"]))
        nbytes = obs_pois_bytes(N, K)
        d = dict(config=name, N=N, K=K, G=G, gpu=gpu,
                 eval_order2_ms_poisson=float(np.median(res["pois"])),
                 eval_order2_ms_logistic_q8=float(np.median(res["logit"])),
                 k_obs_pois_ms=t_obs, k_obs_pois_bytes=nbytes,
                 k_obs_pois_hbm_fraction=nbytes / (t_obs * 1e-3) / HBM_PEAK,
                 rounds=res)
        print(json.dumps(d))
        lines.append(d)
        del pm, lm, X, y_cnt, y_bin
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
