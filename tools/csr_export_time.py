"""CUDA-event time of a first CSR export -- ``hessian_csr`` right after an order-2 evaluation, on a fresh
pattern (the full export of lrvb_glmm_hessian_csr: a model's first step, and every step of a model below
the refill threshold) -- and of the device step (evaluation + ``hessian_csr``, as bench.py times it) at the
shapes of bench.py's workloads.  The inputs are bench.py's seeded data and point; L2 is flushed (256 MiB
write) before every evaluation, outside the events.  Prints one JSON line per workload, with the card's
name and power limit.  A/B of two library builds: run it once per build with LRVB_LIB_PATH, alternating.

    python tools/csr_export_time.py [--reps 30] [--workloads c1,c2,c3,c4] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import lrvb_b200 as vb  # noqa: E402
from lrvb_b200 import _native as nat  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def timed(fn, before, reps):
    """CUDA-event times (ms) of fn() over reps calls; before() runs ahead of each, outside the events."""
    ts = []
    for _ in range(reps):
        before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
        del out
    return np.asarray(ts)


def run(name, reps, flush, lib):
    wl = bench.WORKLOADS[name]
    dev = torch.device("cuda", 0)
    X, y, g = bench.synth_shard(torch, wl["N"], wl["K"], wl["G"], 2000, dev)
    model = vb.LogisticGLMM(X, y, g, num_gh_points=wl["Q"], num_groups=wl["G"])
    del X, y, g
    gen = torch.Generator(device=dev)
    gen.manual_seed(7)
    x = 0.1 * torch.randn(model.D, dtype=torch.float64, device=dev, generator=gen)

    def evaluate():
        flush.zero_()
        model.evaluate(x, 2, force=True)

    def first_export():
        model._csr_pattern = None        # a fresh pattern: hessian_csr runs the full export
        return model.hessian_csr()

    def step():
        model.evaluate(x, 2, force=True)
        return model.hessian_csr()

    for _ in range(3):
        evaluate()
        first_export()
    torch.cuda.synchronize()
    n0 = lib.lrvb_launch_count()
    first = timed(first_export, evaluate, reps)
    launches = (lib.lrvb_launch_count() - n0) // reps
    for _ in range(3):
        flush.zero_()
        step()
    torch.cuda.synchronize()
    steps = timed(step, flush.zero_, reps)
    nnz = int(model.hessian_csr().nnz)
    res = {"workload": name, "D": int(model.D), "nnz": nnz, "reps": reps,
           "first_export_ms": {"median": float(np.median(first)), "mean": float(first.mean()),
                               "min": float(first.min())},
           "launches_per_eval_and_first_export": int(launches),
           "step_ms": {"median": float(np.median(steps)), "mean": float(steps.mean()), "min": float(steps.min())}}
    del model, x
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--workloads", default="c1,c2,c3,c4")
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("csr_export_time.py needs a CUDA device")
    torch.cuda.set_device(0)
    lib = nat.load()
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")
    gpu = card()
    lines = []
    for name in args.workloads.split(","):
        res = run(name, args.reps, flush, lib)
        res.update(lib=nat.LIB_PATH, card=gpu)
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
