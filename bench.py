#!/usr/bin/env python
"""bench.py -- logistic-GLMM observations/sec for one fused ELBO + gradient + sparse-Hessian
evaluation (BASELINE.json metric) on N B200s, plus the end-to-end number through the public
Objective API, the rooflines of the dominant kernels, parity against the CPU oracle on the very
data that is timed, and the CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c1|c2|c3|c4|c5] [--no-target] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A step = one pass of the hot path over one batch of synthetic observations already resident in
HBM: lrvb_glmm_eval(order 2) [+ the all-reduce of the packed (KL, global gradient, global Hessian
block) over the NVLink peer windows when N > 1] + device CSR assembly of the arrowhead Hessian.

The headline line (`value`) is BASELINE.json configs[1] (C2: N=1M, K=20, G=10k, Q=8) on one GPU;
with N > 1 every rank holds a C2-sized shard (weak scaling; groups are rank-private, the replicated
blocks all-reduced).  The same JSON line carries `target_config`: BASELINE.json configs[2] (C3:
N=10M, K=50, G=100k) -- whole on one GPU at N = 1, and at N > 1 the SAME 10M problem cut into
group-aligned shards by distributed.partition_groups (strong scaling), timed next to a 1-GPU run of
the whole problem on rank 0 in the same process so that the speed-up is measured on one box.
Prints ONE JSON line.  --steps is the number of timed steps behind `value` / `ms_per_step` (for c5: timed
launches per family).  The other timed loops -- e2e, the per-kernel durations, target_config -- run bounded
counts of their own, reported in their sections, so that C4's 150 ms steps keep a run short.  With
--dump-outputs DIR the results of the last timed step are also written as .npy files: the inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # observations, fixed effects, groups, Gauss-Hermite points
    "c1": dict(N=5_000, K=5, G=100, Q=4, name="logistic GLMM N=5k K=5 G=100 Q=4 (BASELINE configs[0])"),
    "c2": dict(N=1_000_000, K=20, G=10_000, Q=8,
               name="logistic GLMM N=1M K=20 G=10k Q=8 per GPU (BASELINE configs[1])"),
    "c3": dict(N=10_000_000, K=50, G=100_000, Q=8,
               name="logistic GLMM N=10M K=50 G=100k Q=8 (BASELINE configs[2])"),
    "c4": dict(N=10_000_000, K=200, G=100_000, Q=8,
               name="logistic GLMM N=10M K=200 G=100k Q=8 (BASELINE configs[3])"),
}
METRIC = "GLMM obs/sec for ELBO+grad+sparse Hessian"
UNIT = "obs/s"
CPU_SAMPLE = dict(N=500_000, G=5_000)   # bounded sample of the workload for the CPU arm
DUMP_BYTES = 64 * 10 ** 6               # --dump-outputs: all .npy files together


# ------------------------------------------------------------------------------------------
class ClockSampler(object):
    """SM clock / throttle reasons sampled DURING the timed region, in-process through NVML
    (a thread polling every few ms; spawning nvidia-smi stalls the GPU for milliseconds and its
    100 ms period misses a short timed region).  Falls back to one nvidia-smi query."""
    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
               ("hw_power_brake_slowdown", 0x80), ("sw_power_cap", 0x4))

    def __init__(self, index, period_s=0.002):
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.power = [], set(), []
        self.handle, self.nvml, self.max_mhz = None, None, None
        self._stop = threading.Event()
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception as exc:       # noqa: BLE001
            self.error = "NVML unavailable: %s" % exc

    def _poll(self):
        nv = self.nvml
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                for name, bit in self.REASONS:
                    if mask & bit:
                        self.reasons.add(name)
                if len(self.samples) % 32 == 1:    # the power query is the slow one: sparse
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
            except Exception:          # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()

    def stop(self):
        if self.thread is not None:
            self._stop.set()
            self.thread.join(timeout=2)
        if self.samples:
            return dict(sm_mhz=float(np.median(self.samples)), sm_max_mhz=self.max_mhz,
                        reasons=sorted(self.reasons), samples=len(self.samples),
                        power_w_max=max(self.power) if self.power else None, source="nvml")
        try:
            out = subprocess.run(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=clocks.sm,clocks.max.sm",
                 "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
            a, b2 = [float(v) for v in out.strip().split(",")[:2]]
            return dict(sm_mhz=a, sm_max_mhz=b2, reasons=[], samples=1,
                        source="nvidia-smi after the timed region (NVML polling failed)")
        except Exception:              # noqa: BLE001
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["clock sampling unavailable"], samples=0)


def synth_shard(torch, N, K, G, seed, device):
    """Seeded synthetic shard on the device (SURVEY.md 8d): X ~ N(0,1), balanced group-sorted ids,
    y ~ Bernoulli(sigmoid(X beta + u_g))."""
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    X = torch.randn(N, K, dtype=torch.float64, device=device, generator=gen)
    base, rem = divmod(N, G)
    counts = torch.full((G,), base, dtype=torch.int64, device=device)
    counts[:rem] += 1
    g = torch.repeat_interleave(torch.arange(G, device=device), counts)
    beta = 0.5 * torch.randn(K, dtype=torch.float64, device=device, generator=gen)
    u = 0.3 + 0.5 * torch.randn(G, dtype=torch.float64, device=device, generator=gen)
    p = torch.sigmoid(X @ beta + u[g])
    y = (torch.rand(N, dtype=torch.float64, device=device, generator=gen) < p).double()
    return X, y, g


def measure_dgemm_tflops(torch, n=8192, reps=5):
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(2):
        a @ b
    best = float("inf")
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        a @ b
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def cpu_oracle_step(sample, K, Q, seed=123):
    """One CPU pass (oracle port) over a bounded sample: KL + gradient + arrowhead blocks + CSR."""
    from oracle import glmm_oracle as go
    Ns, Gs = sample["N"], sample["G"]
    X, y, g = go.make_glmm_data(Ns, K, Gs, seed)
    gh_x, gh_w = np.polynomial.hermite.hermgauss(Q)
    o = go.GLMMOracle(X, y, g, gh_x, gh_w, G=Gs)
    x = go.make_free(o.lay.D, seed)

    def step():
        t = time.perf_counter()
        H = o.kl_hessian_csr(x)     # kl_blocks (value, gradient, Hessian blocks) + CSR emission
        return time.perf_counter() - t, H.nnz
    return step


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(n) if n else 1
    except Exception:
        return os.cpu_count() or 1


def _hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0   # B200_PROFILING.md fallback


def _hbm_peak_source():
    return ("MEASURED_PEAKS.json hbm_gbs (burst copy)" if os.path.exists(
        os.path.join(ROOT, "MEASURED_PEAKS.json")) else "B200_PROFILING.md fallback")


# ------------------------------------------------------------------------------------------
def run_reference(args, wl):
    """--impl reference: the reference's CPU path for this metric (oracle port -- the reference
    itself needs autograd<1.4, not installable here; see DESIGN.md), rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "c5":
        import bench_ef
        return bench_ef.run_reference(args)
    ns = min(CPU_SAMPLE["N"], wl["N"])
    sample_cfg = dict(N=ns, G=max(1, wl["G"] * ns // wl["N"]))
    step = cpu_oracle_step(sample_cfg, wl["K"], wl["Q"])
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    times = [step()[0] for _ in range(args.steps)]
    ms = 1e3 * float(np.mean(times))
    value = sample_cfg["N"] / (ms * 1e-3)
    cores = blas_threads()
    sample = ("N=%d obs, K=%d, G=%d, Q=%d per step: a %s sample of the per-GPU workload; obs/s is "
              "rate-normalised (the work is linear in N at fixed N/G)") % (
        sample_cfg["N"], wl["K"], sample_cfg["G"], wl["Q"],
        "1/%d" % (wl["N"] // sample_cfg["N"]) if wl["N"] > sample_cfg["N"] else "full-size")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"], "cpu_sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample,
                         "note": "numpy analytic restatement of the reference path (oracle/); "
                                 "BLAS parts use %d threads, elementwise parts 1" % cores},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
class Ctx(object):
    pass


def _gather_floats(ctx, vals):
    """(world, len(vals)) array of per-rank values on every rank."""
    t = ctx.torch.tensor([float(v) for v in vals], dtype=ctx.torch.float64, device=ctx.device)
    if ctx.world == 1:
        return t.cpu().numpy()[None, :]
    out = [ctx.torch.empty_like(t) for _ in range(ctx.world)]
    ctx.dist.all_gather(out, t)
    return ctx.torch.stack(out).cpu().numpy()


def make_model(ctx, wl, mode):
    """mode 'single': the whole workload on this GPU.  'weak': this rank's own workload-sized shard.
    'strong': this rank's group-aligned shard of ONE workload-sized problem (distributed.partition_groups
    over the balanced synthetic groups)."""
    torch, vb = ctx.torch, ctx.vb
    N, K, G, Q = wl["N"], wl["K"], wl["G"], wl["Q"]
    if mode == "single":
        X, y, g = synth_shard(torch, N, K, G, seed=1000 * 2, device=ctx.device)
        model = vb.LogisticGLMM(X, y, g, num_gh_points=Q, num_groups=G)
        return model, model, N
    from lrvb_b200 import distributed as vbd
    if mode == "weak":
        X, y, g = synth_shard(torch, N, K, G, seed=1000 * 2 + ctx.rank, device=ctx.device)
        model = vbd.ShardedLogisticGLMM.from_local_shard(X, y, g, num_local_groups=G, num_gh_points=Q)
        return model, model.local, N
    # strong: cut the G balanced groups of the N-observation problem exactly as from_full would
    base, rem = divmod(N, G)
    counts = np.full(G, base, dtype=np.int64)
    counts[:rem] += 1
    bounds = vbd.partition_groups(counts, ctx.world)
    g0, g1 = int(bounds[ctx.rank]), int(bounds[ctx.rank + 1])
    Nl = int(counts[g0:g1].sum())
    X, y, g = synth_shard(torch, Nl, K, g1 - g0, seed=1000 * 3 + ctx.rank, device=ctx.device)
    model = vbd.ShardedLogisticGLMM.from_local_shard(X, y, g, num_local_groups=g1 - g0, num_gh_points=Q)
    return model, model.local, Nl


def last_step_outputs(torch, model, csr):
    """What a caller of the timed step receives -- KL, gradient and sparse Hessian of the last evaluation --
    as float64 host arrays.  The Hessian goes out as COO triplets (row, col, value) in CSR order.  When all
    of them would take the total past DUMP_BYTES (C3, C4), entry positions drawn with a fixed seed stand in
    for them: two builds that produce the same pattern write the same positions."""
    kl = model.kl_tensor().reshape(1).cpu().numpy()
    grad = model.grad_tensor().cpu().numpy()
    crow, val = csr.crow_indices.long(), csr.values
    nnz = val.numel()
    room = (DUMP_BYTES - 8 * (kl.size + grad.size) - 4096) // 24     # 4096: the five .npy headers
    if nnz <= room:
        pos = torch.arange(nnz, device=val.device)
    else:
        pos = torch.from_numpy(np.unique(np.random.default_rng(0).integers(0, nnz, size=room))).to(val.device)
    row = torch.searchsorted(crow, pos, right=True) - 1
    return {"kl": kl, "grad": grad, "hessian_row": row.double().cpu().numpy(),
            "hessian_col": csr.col_indices[pos].double().cpu().numpy(), "hessian_value": val[pos].cpu().numpy()}


def write_outputs(path, outputs):
    os.makedirs(path, exist_ok=True)
    for name, arr in outputs.items():
        np.save(os.path.join(path, name + ".npy"), arr)
    print("outputs of the last timed step: %s (%s)" % (
        path, ", ".join("%s %d" % (n, a.size) for n, a in outputs.items())), file=sys.stderr)


def time_workload(ctx, wl, mode, steps, warmup, sampler=None, kernel_steps=30, dump=False):
    """Device-timed steps of one workload.  Returns a dict (identical on every rank for the reduced
    entries).  Timing discipline: garbage collector off and every rank synchronised BEFORE the last
    barrier; one untimed step after the barrier (the first collective after a barrier pays a
    re-synchronisation); then straight into the timed loop.  L2 flushed (256 MiB write) before every
    timed step, outside the events.  With ``dump`` the result carries ``outputs``: the last timed
    step's results on the host (last_step_outputs)."""
    torch, dist, lib, nat = ctx.torch, ctx.dist, ctx.lib, ctx.nat
    sharded = mode in ("weak", "strong")
    model, local, N_local = make_model(ctx, wl, mode)
    D = model.D
    gen = torch.Generator(device=ctx.device)
    gen.manual_seed(7)
    x_dev = 0.1 * torch.randn(D, dtype=torch.float64, device=ctx.device, generator=gen)
    if sharded:
        dist.broadcast(x_dev, 0)
    flush = ctx.flush
    peer = getattr(model, "_peer", None) if sharded else None

    def device_step():
        model.evaluate(x_dev, 2, force=True)
        return model.hessian_csr()

    csr = None
    for _ in range(max(warmup, 3)):
        flush.zero_()
        csr = device_step()                 # keep the previous result alive as the timed loop does:
    torch.cuda.synchronize()                # the allocator then owns both ping-pong result blocks
    if sampler is not None:
        sampler.start()
    for _ in range(3):                      # the sampler thread's first NVML calls happen untimed (every
        flush.zero_()                       # rank runs these steps: they contain a collective)
        csr = device_step()
    if peer is not None:
        peer.set_stats(True)
    gc.collect()
    gc.disable()                            # no collector pauses from here to the end of the timed loop
    torch.cuda.synchronize()
    if sharded:
        dist.barrier()
    flush.zero_()
    csr = device_step()                     # untimed: re-synchronises the ranks on the device
    torch.cuda.synchronize()
    if peer is not None:
        peer.set_stats(True)                # reset: count the timed steps only
    launches0 = lib.lrvb_launch_count()
    step_ms = []
    for _ in range(steps):
        flush.zero_()                       # L2 flush (126 MB L2 < 256 MiB), outside the timing
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        csr = device_step()
        e1.record()
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1))
    torch.cuda.synchronize()
    gc.enable()
    outputs = last_step_outputs(torch, local, csr) if dump else None
    launches = (lib.lrvb_launch_count() - launches0) // max(1, steps)
    wait = peer.stats() if peer is not None else None
    if peer is not None:
        peer.set_stats(False)
    if sharded:
        dist.barrier()
    clocks = sampler.stop() if sampler is not None else None
    sm = np.asarray(step_ms)
    per_rank = _gather_floats(ctx, [sm.mean(), np.median(sm), sm.min(), sm.max(), N_local,
                                    (wait["wait_us_total"] / max(1, wait["calls"])) if wait else 0.0,
                                    wait["wait_us_max"] if wait else 0.0]) if sharded else \
        np.asarray([[sm.mean(), np.median(sm), sm.min(), sm.max(), N_local, 0.0, 0.0]])
    ms_per_step = float(per_rank[:, 0].max())          # max over ranks of the per-rank mean
    n_total = int(per_rank[:, 4].sum())
    res = dict(ms_per_step=ms_per_step, value=n_total / (ms_per_step * 1e-3), n_total=n_total,
               n_local=N_local, launches=int(launches), nnz=int(csr.nnz), D=int(D), clocks=clocks,
               median_ms_max_over_ranks=float(per_rank[:, 1].max()),
               per_rank_ms={"mean": [round(v, 5) for v in per_rank[:, 0]],
                            "median": [round(v, 5) for v in per_rank[:, 1]],
                            "max": [round(v, 5) for v in per_rank[:, 3]]},
               model=model, local=local, x_dev=x_dev, mode=mode, outputs=outputs)
    if sharded:
        res["collective_wait_us"] = {
            "mean_per_call_max_over_ranks": float(per_rank[:, 5].max()),
            "mean_per_call_by_rank": [round(v, 2) for v in per_rank[:, 5]],
            "largest_single_wait_us": float(per_rank[:, 6].max()),
            "calls_per_step": (wait["calls"] // max(1, steps)) if wait else 0,
            "how": "inside k_p2p_allreduce: %globaltimer before / after the poll loops, maximum over the "
                   "elements of a call; the time a rank waited for its slowest peer (inter-rank skew + one "
                   "NVLink traversal)" if peer is not None else "NCCL path: not measured"}
    if ctx.rank == 0:
        s2 = np.sort(sm)
        worst = np.argsort(step_ms)[-3:][::-1]
        print("[%s %s] step ms (rank 0): min %.4f median %.4f p90 %.4f max %.4f mean %.4f; slowest %s; "
              "max-over-ranks mean %.4f" % (
                  wl["name"][:28], mode, s2[0], s2[len(s2) // 2], s2[int(0.9 * (len(s2) - 1))], s2[-1],
                  sm.mean(), ", ".join("#%d %.3f" % (i, step_ms[i]) for i in worst), ms_per_step),
              file=sys.stderr)

    # per-kernel durations for the rooflines: a separate loop, because the CUDA events the library
    # records between its kernels cut the chain of programmatic dependent launches
    ms3 = (ctypes.c_float * 3)()
    eval_ms, obs_ms, gram_ms = [], [], []
    nat.check(lib.lrvb_glmm_set_timing(local._h, 1))
    for i in range(min(steps, kernel_steps) + 3):
        flush.zero_()
        csr = device_step()
        torch.cuda.synchronize()
        if i >= 3:
            nat.check(lib.lrvb_glmm_last_timing(local._h, ms3))
            eval_ms.append(ms3[0]); obs_ms.append(ms3[1]); gram_ms.append(ms3[2])
    nat.check(lib.lrvb_glmm_set_timing(local._h, 0))
    res.update(eval_ms=float(np.mean(eval_ms)), obs_ms=float(np.mean(obs_ms)), gram_ms=float(np.mean(gram_ms)))
    del csr
    return res


def rooflines(res, wl, peak_tf, traffic):
    """Rooflines of the two kernels that carry the step -- the fused per-observation pass (HBM roofline
    per SURVEY.md 8(d): 8K + 12 algorithmic bytes per observation) and the packed Gram kernel (FP64
    tensor roofline: 4K^2 + 2K flops per observation) -- and of the whole step.  `roofline` is the
    kernel with the larger measured duration; the other is reported beside it."""
    K, Q, N = wl["K"], wl["Q"], res["n_local"]
    flops_per_obs = 4 * K * K + 2 * K
    bytes_per_obs = 8 * K + 12
    step_flops = 4 * K * K + 18 * K + 12 * Q          # SURVEY.md 8(d) total per observation
    gms, oms = res["gram_ms"], res["obs_ms"]
    hbm = _hbm_peak()
    if gms == 0.0 and oms > 0.0:
        # one-pass kernel (csrc/fused.cuh): quadrature, group sums and the packed Gram in one launch; it is
        # bound by the FP64 pipe (DFMA + DMMA share it), so its roofline is the FP64 tensor peak against ALL
        # algorithmic flops of an observation (SURVEY.md 8(d): 4K^2 + 18K + 12Q)
        roofline = {"bound": "tensor",
                    "kernel": "lrvb::k_fused_eval (one pass over X: quadrature warps + DMMA.8x8x4 warps per SM "
                              "sub-partition, TMA rings)",
                    "achieved": N * step_flops / (oms * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                    "traffic": traffic.get("k_fused_dram_bytes"),
                    "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (FP64 is not in MEASURED_PEAKS.json); "
                                   "DMMA.8x8x4 microbenchmark: 37.1 TF",
                    "kernel_ms": oms, "flops_per_obs": step_flops,
                    "hbm": {"achieved": N * bytes_per_obs / (oms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                            "bytes_per_obs": bytes_per_obs, "peak_source": _hbm_peak_source(),
                            "frac": N * bytes_per_obs / (oms * 1e-3) / 1e9 / hbm}}
        roofline["frac"] = roofline["achieved"] / peak_tf
    else:
        gram_kernel = ("lrvb::k_gram_small (DMMA.8x8x4, packed [x|s] triangle per warp)" if K < 16 else
                       "lrvb::k_gram_mid (DMMA.8x8x4, packed [x|s] triangle per warp / warp team)" if K <= 104 else
                       "lrvb::k_gram_wide (DMMA.8x8x4, 4-5 tile column blocks against each other, 8 warps x 25 "
                       "accumulator tiles; k_group runs beside it on a side stream and is inside kernel_ms)" if (K % 8 == 0 and 176 <= K <= 240
                                                and os.environ.get("LRVB_GRAM_WIDE", "1") != "0") else
                       "lrvb::k_gram_big (DMMA.8x8x4, packed [x|s] rectangles)")
        roof_gram = {"bound": "tensor", "kernel": gram_kernel,
                     "achieved": N * flops_per_obs / (gms * 1e-3) / 1e12 if gms > 0 else None, "peak": peak_tf,
                     "unit": "TFLOP/s", "traffic": traffic.get("k_gram_dram_bytes"),
                     "peak_source": "cuBLAS DGEMM 8192^3 measured in this run (FP64 is not in "
                                    "MEASURED_PEAKS.json); DMMA.8x8x4 microbenchmark: 37.1 TF",
                     "kernel_ms": gms, "flops_per_obs": flops_per_obs}
        roof_gram["frac"] = roof_gram["achieved"] / peak_tf if gms > 0 else None
        roof_obs = {"bound": "hbm",
                    "kernel": "lrvb::k_obs_fused<2> (quadrature + per-group sums, TMA ring per warp)"
                    if K <= 62 else "lrvb::k_obs<2>",
                    "achieved": N * bytes_per_obs / (oms * 1e-3) / 1e9 if oms > 0 else None, "peak": hbm,
                    "unit": "GB/s", "traffic": traffic.get("k_obs_dram_bytes"),
                    "peak_source": _hbm_peak_source(), "kernel_ms": oms, "bytes_per_obs": bytes_per_obs,
                    "note": "bound by fp64 instruction throughput (exp / log1p chains of the quadrature), not by "
                            "HBM; see profiles/"}
        roof_obs["frac"] = roof_obs["achieved"] / hbm if oms > 0 else None
        roofline = dict(roof_obs if oms >= gms else roof_gram)
        roofline["other_kernel"] = roof_gram if oms >= gms else roof_obs
    roofline["eval_ms"] = res["eval_ms"]
    t = res["ms_per_step"] * 1e-3
    hbm_s = N * bytes_per_obs / (hbm * 1e9)
    fl_s = N * step_flops / (peak_tf * 1e12)
    roofline["step_frac"] = max(hbm_s, fl_s) / t
    roofline["step_frac_how"] = ("max(N (8K+12) B / HBM peak, N (4K^2+18K+12Q) flop / DGEMM peak) / ms_per_step "
                                 "= max(%.4f, %.4f) ms / %.4f ms" % (hbm_s * 1e3, fl_s * 1e3, t * 1e3))
    roofline["traffic_source"] = traffic.get("source")
    return roofline


def cov_entry(ctx, model, K, G_local, peak_tf, ncov=20):
    """Second half of the metric: wall time of the global-parameter LRVB covariance (H^-1)[:Dg,:Dg] of the
    cached Hessian by the Schur complement of the local blocks: DMMA Gram over the border matrix
    [+ all-reduce of S when sharded] + SPD inverse; device timed, max over ranks."""
    torch, dist = ctx.torch, ctx.dist
    sharded = hasattr(model, "local")
    for _ in range(3):
        if sharded:
            model._sinv = None
        model.global_covariance()
    torch.cuda.synchronize()
    if sharded:
        dist.barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(ncov):
        if sharded:
            model._sinv = None              # the sharded model caches the result: recompute
        model.global_covariance()
    c1.record()
    c1.synchronize()
    cov_ms = float(_gather_floats(ctx, [c0.elapsed_time(c1) / ncov])[:, 0].max()) if sharded \
        else c0.elapsed_time(c1) / ncov
    Dg = 4 + 2 * K
    world = ctx.world if sharded else 1
    flops = world * G_local * (2 * Dg * Dg + 8 * Dg) + Dg ** 3
    tf = flops / (cov_ms * 1e-3) / 1e12
    return {"ms": cov_ms, "what": "(H^-1)[:Dg,:Dg] of the cached Hessian: Schur complement (DMMA) "
            "[+ sum over ranks] + SPD inverse, device time, max over ranks", "Dg": Dg,
            "algorithmic_flops": flops, "achieved_tflops": tf, "peak_tflops": peak_tf,
            "frac": tf / peak_tf,
            "bound": "latency (work far below one wave of the tensor pipe)" if Dg < 128 else "tensor / latency"}


def cov_cg_entry(ctx, res, max_seconds=40.0):
    """BASELINE configs[3]: the global-parameter LRVB covariance by CONJUGATE GRADIENT with device Hessian-
    vector products (ConjugateGradient.py:81-105), one solve per global parameter, block-Jacobi
    preconditioner, rtol 1e-8 -- next to the Schur path.  Columns are solved until `max_seconds` of device
    time are spent; the total is extrapolated from the per-solve mean when not all Dg columns were run."""
    torch = ctx.torch
    model, x_dev = res["model"], res["x_dev"]
    model.evaluate(x_dev, 2)
    Dg, D = model.Dg, model.D
    sinv = model.global_covariance()
    e = torch.zeros(D, dtype=torch.float64, device=ctx.device)
    iters, ms, err = [], [], 0.0
    t_all = 0.0
    for i in range(Dg):
        e.zero_()
        e[i] = 1.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        x, info, it = model.cg(e, None, precond="block_jacobi", rtol=1e-8)
        e1.record()
        e1.synchronize()
        t = e0.elapsed_time(e1)
        ms.append(t); iters.append(it)
        t_all += t
        err = max(err, float(((x[:Dg] - sinv[i]).abs().max() / sinv.abs().max()).item()))
        if info != 0:
            break
        if t_all > 1e3 * max_seconds:
            break
    n = len(ms)
    return {"what": "(H^-1)[:Dg,:Dg] column by column: device CG (scipy.sparse.linalg.cg semantics, rtol 1e-8, "
                    "block-Jacobi M), Hessian-vector products on the cached arrowhead blocks",
            "columns_solved": n, "columns_total": Dg, "iterations_mean": float(np.mean(iters)),
            "iterations_max": int(np.max(iters)), "ms_per_solve": float(np.mean(ms)),
            "us_per_iteration": 1e3 * float(np.sum(ms)) / max(1, int(np.sum(iters))),
            "ms_total_all_columns": float(np.mean(ms)) * Dg, "extrapolated": n < Dg,
            "max_rel_diff_vs_schur": err,
            "note": "the point is the bench's (not an optimum): if H is not positive definite there CG reports "
                    "info != 0 and the run stops"}


def e2e_measure(ctx, res, steps, warmup):
    """The same metric through the public API with HOST buffers: numpy x in, scipy CSR + numpy gradient
    + float out, every step at a different point; wall clock, max over ranks."""
    torch, dist, vb = ctx.torch, ctx.dist, ctx.vb
    model, x_dev, D = res["model"], res["x_dev"], res["D"]
    sharded = res["mode"] != "single"
    obj = vb.Objective(model.glmm_par, model) if not sharded else None
    x0 = x_dev.cpu().numpy()
    x_host = [x0 + 1e-3 * np.random.default_rng(s).standard_normal(D) for s in range(min(steps + warmup, 8))]

    def step(i):
        xh = x_host[i % len(x_host)]
        if sharded:
            # sharded: every rank brings ITS part of the distributed Hessian / gradient to its host
            model.evaluate(xh, 2)
            H = model.local.hessian_scipy()      # one synchronisation: values + gradient + KL
            gr = model.local.grad_host()
            kl = model.local.kl_host()
            return H, gr, kl
        H = obj.fun_free_hessian(xh)     # scipy CSR on the host (order-2 evaluation, cached)
        gr = obj.fun_free_grad(xh)       # numpy (D,)
        kl = obj.fun_free(xh)            # float
        return H, gr, kl
    for i in range(warmup):
        H, gr, kl = step(i)                 # bound as in the timed loop: the previous result lives until the next is back
    gc.collect()
    gc.disable()                            # as in the device loop: no collector pauses inside the timed steps
    torch.cuda.synchronize()
    if sharded:
        dist.barrier()
    prof = None
    if os.environ.get("LRVB_BENCH_PROFILE"):
        import cProfile
        prof = cProfile.Profile()
        prof.enable()
    t0 = time.perf_counter()
    marks = []
    for i in range(steps):
        H, gr, kl = step(warmup + i)
        marks.append(time.perf_counter())
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    gc.enable()
    per = np.diff(np.asarray([t0] + marks)) * 1e3
    if ctx.rank == 0:
        print("e2e step ms (rank 0): min %.3f median %.3f max %.3f (step #%d) mean %.3f" % (
            per.min(), np.median(per), per.max(), int(per.argmax()), per.mean()), file=sys.stderr)
    if prof is not None:
        import pstats
        prof.disable()
        pstats.Stats(prof, stream=sys.stderr).sort_stats("tottime").print_stats(14)
    dt = float(_gather_floats(ctx, [dt])[:, 0].max()) if sharded else dt
    nnz = int(H.nnz)
    return {"value": res["n_total"] / (dt / steps), "unit": UNIT, "ms_per_step": 1e3 * dt / steps,
            "median_ms_rank0": float(np.median(per)), "steps": steps, "warmup": warmup,
            "h2d_bytes_per_step": 8 * D,
            "d2h_bytes_per_step": 8 + 8 * int(gr.size) + 12 * nnz + 4 * (int(H.shape[0]) + 1),
            "d2h_note": "bytes of the RESULT handed to the caller (data + indices + indptr + gradient + KL); "
                        "the static pattern (indices, indptr) is transferred again only when it changes",
            "api": "Objective.fun_free_hessian/fun_free_grad/fun_free with numpy x; "
                   "scipy CSR + numpy gradient + float returned to the host"}


def parity_single(ctx, res, wl):
    """Untimed check of the very model that was timed (N = 1): KL / gradient / CSR against the CPU oracle
    on the same data and point (tolerance of the north star: 1e-9 relative).  Workloads whose oracle pass
    would take minutes (N K > 4e7) are checked on their first 200k observations / 2000 groups, same K."""
    from oracle import glmm_oracle as go
    model, x_dev = res["model"], res["x_dev"]
    t0 = time.perf_counter()
    gh_x, gh_w = np.polynomial.hermite.hermgauss(wl["Q"])
    if wl["N"] * wl["K"] > 4e7:
        per = wl["N"] // wl["G"]
        Gs = max(1, 200_000 // per)
        Ns = Gs * per
        sub = ctx.vb.LogisticGLMM(model.X[:Ns], model.y[:Ns], model.g[:Ns], num_gh_points=wl["Q"], num_groups=Gs)
        Dg = 4 + 2 * wl["K"]
        idx = ctx.torch.cat([ctx.torch.arange(Dg, device=ctx.device),
                             Dg + ctx.torch.arange(Gs, device=ctx.device),
                             Dg + wl["G"] + ctx.torch.arange(Gs, device=ctx.device)])
        x_dev = x_dev[idx].contiguous()
        model = sub
        wl = dict(wl, N=Ns, G=Gs)
    o = go.GLMMOracle(model.X.cpu().numpy(), model.y.cpu().numpy(), model.g.cpu().numpy().astype(np.int64),
                      gh_x, gh_w, G=wl["G"])
    x = x_dev.cpu().numpy()
    model.evaluate(x_dev, 2, force=True)
    H = model.hessian_csr().to_scipy()
    kl = float(model.kl_tensor().item())
    gr = model.grad_tensor().cpu().numpy()
    klo, go_, _ = o.kl_blocks(x)
    He = o.kl_hessian_csr(x)
    same = bool(np.array_equal(H.indptr, He.indptr) and np.array_equal(H.indices, He.indices))
    out = {"against": "oracle.GLMMOracle on the timed data (N=%d, K=%d, G=%d) at the timed point" % (
               wl["N"], wl["K"], wl["G"]),
           "kl_rel": abs(kl - klo) / abs(klo),
           "grad_rel": float(np.abs(gr - go_).max() / np.abs(go_).max()),
           "hess_rel": float(np.abs(H.data - He.data).max() / np.abs(He.data).max()) if same else None,
           "pattern_equal": same, "nnz": int(H.nnz), "oracle_seconds": round(time.perf_counter() - t0, 2),
           "tolerance": 1e-9}
    out["ok"] = bool(same and out["kl_rel"] < 1e-9 and out["grad_rel"] < 1e-9 and out["hess_rel"] < 1e-9)
    return out


def parity_sharded(ctx, res):
    """Untimed checks at N > 1: (i) the replicated block [KL, grad_g, A] summed by the peer-memory kernel
    against NCCL's sum of the same per-rank buffers, and bitwise equality of the result across ranks;
    (ii) on one common 200k-observation data set: N shards == 1 GPU == oracle (SURVEY.md section 4)."""
    torch, dist, vb = ctx.torch, ctx.dist, ctx.vb
    from lrvb_b200 import distributed as vbd
    from oracle import glmm_oracle as go
    model, local, x_dev = res["model"], res["local"], res["x_dev"]
    out = {}
    # (i) same per-rank partial buffers through both collectives
    local.evaluate(x_dev, 2, force=True)                 # un-reduced partials of this rank
    part = local._out_global.clone()
    a = part.clone()
    dist.all_reduce(a)
    if model._peer is not None and model._peer.fits(part):
        b = part.clone()
        model._peer.all_reduce_(b)
        gathered = [torch.empty_like(b) for _ in range(ctx.world)]
        dist.all_gather(gathered, b)
        out["peer_vs_nccl_rel"] = float(((a - b).abs().max() / a.abs().max()).item())
        out["peer_bitwise_equal_across_ranks"] = bool(all(torch.equal(gathered[0], t) for t in gathered))
        out["peer_status"] = model._peer.status()
    else:
        out["peer_vs_nccl_rel"] = None
        out["peer_note"] = "peer windows unavailable or message too large: NCCL path in use"
    model.invalidate() if hasattr(model, "invalidate") else None
    model._cache = dict(x=None, order=-1, coords=None)
    # (ii) N-shard == 1-shard == oracle on a common data set
    N, K, G, Q = 200_000, 20, 2_000, 8
    X, y, g = go.make_glmm_data(N, K, G, seed=4242)
    rng = np.random.default_rng(4243)
    g = np.sort(rng.integers(0, G, size=N)).astype(np.int64)      # ragged groups
    x = go.make_free(4 + 2 * K + 2 * G, 4242)
    sh = vbd.ShardedLogisticGLMM.from_full(X, y, g, G, num_gh_points=Q)
    obj = vb.Objective(sh.glmm_par, sh)
    kl_s, gr_s, H_s = obj.fun_free(x), obj.fun_free_grad(x), obj.fun_free_hessian(x)
    cov_s = sh.global_covariance().cpu().numpy()
    if ctx.rank == 0:
        gh_x, gh_w = np.polynomial.hermite.hermgauss(Q)
        o = go.GLMMOracle(X, y, g, gh_x, gh_w, G=G)
        klo, gro, _ = o.kl_blocks(x)
        He = o.kl_hessian_csr(x)
        one = vb.LogisticGLMM(X, y, g, num_gh_points=Q, num_groups=G)
        o1 = vb.Objective(one.glmm_par, one)
        kl_1, gr_1, H_1 = o1.fun_free(x), o1.fun_free_grad(x), o1.fun_free_hessian(x)
        cov_1 = one.global_covariance().cpu().numpy()
        cov_o = o.schur_global_cov(x)[0]
        same = bool(np.array_equal(H_s.indptr, He.indptr) and np.array_equal(H_s.indices, He.indices)
                    and np.array_equal(H_1.indices, He.indices))
        rel = lambda p, q: float(np.abs(np.asarray(p) - np.asarray(q)).max() / np.abs(np.asarray(q)).max())  # noqa: E731
        out["shards_vs_oracle"] = {"case": "N=200k K=20 G=2000 ragged groups, %d shards" % ctx.world,
                                   "kl_rel": rel(kl_s, klo), "grad_rel": rel(gr_s, gro),
                                   "hess_rel": rel(H_s.data, He.data) if same else None,
                                   "cov_rel": rel(cov_s, cov_o), "pattern_equal": same}
        out["shards_vs_one_gpu"] = {"kl_rel": rel(kl_s, kl_1), "grad_rel": rel(gr_s, gr_1),
                                    "hess_rel": rel(H_s.data, H_1.data) if same else None,
                                    "cov_rel": rel(cov_s, cov_1)}
        so = out["shards_vs_oracle"]
        out["ok"] = bool(same and so["kl_rel"] < 1e-9 and so["grad_rel"] < 1e-9 and so["hess_rel"] < 1e-9
                         and so["cov_rel"] < 1e-8 and (out["peer_vs_nccl_rel"] is None or (
                             out["peer_vs_nccl_rel"] < 1e-13 and out["peer_bitwise_equal_across_ranks"]
                             and out["peer_status"] == 0)))
        del one
    dist.barrier()
    del sh
    return out


def _load_traffic(key):
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(tpath)).get(key, {})
    except Exception:
        return {}


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    ctx = Ctx()
    ctx.torch, ctx.dist = torch, dist
    ctx.rank = rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    ctx.world = world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    ctx.device = device = torch.device("cuda", local_rank)
    # stdout must carry the one JSON line only, but native libraries write there too (NCCL prints its
    # version banner with printf): point fd 1 at stderr for the whole run and keep the real stdout
    # for the result line
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    if args.gpus != world and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE %d" % (args.gpus, world), file=sys.stderr)

    import lrvb_b200 as vb
    from lrvb_b200 import _native as nat
    ctx.vb, ctx.nat = vb, nat
    ctx.lib = nat.load()
    ctx.flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=device)

    if args.workload == "c5":
        import bench_ef
        line, outputs = bench_ef.run_ours(ctx, args, dump=args.dump_outputs is not None and rank == 0)
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        if rank == 0:
            os.write(result_fd, (json.dumps(line) + "\n").encode())
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        os.dup2(result_fd, 1)
        os.close(result_fd)
        return

    K, G, Q = wl["K"], wl["G"], wl["Q"]
    mode = "single" if world == 1 else "weak"
    sampler = ClockSampler(local_rank) if rank == 0 else None
    res = time_workload(ctx, wl, mode, args.steps, args.warmup, sampler=sampler,
                        dump=args.dump_outputs is not None and rank == 0)
    if res["outputs"] is not None:
        write_outputs(args.dump_outputs, res.pop("outputs"))
    peak_tf = measure_dgemm_tflops(torch) if rank == 0 else 1.0
    cov = cov_entry(ctx, res["model"], K, G, peak_tf, ncov=20 if K <= 64 else 3)
    if args.workload == "c4" and world == 1:
        cov["cg"] = cov_cg_entry(ctx, res)
    # warm-up of the host path: the pinned staging blocks of torch's caching host allocator (three 14 MB
    # blocks rotate at C2) are created by cudaHostAlloc calls of several milliseconds each the first time
    # wide models move GBs per step: fewer steps, but enough warm-up that the rotating pinned result blocks
    # (one is created while the previous result is still alive) exist before the timed steps
    e2e = e2e_measure(ctx, res, min(args.steps, 50 if K <= 64 else 3), max(args.warmup, 10) if K <= 64 else 3)
    parity = parity_single(ctx, res, wl) if world == 1 else parity_sharded(ctx, res)

    line = None
    if rank == 0:
        ns = min(CPU_SAMPLE["N"], wl["N"])
        sample_cfg = dict(N=ns, G=max(1, G * ns // wl["N"]))
        stepf = cpu_oracle_step(sample_cfg, K, Q)
        stepf()
        ts = [stepf()[0] for _ in range(3)]
        cores = blas_threads()
        cpu = {"value": sample_cfg["N"] / float(np.median(ts)), "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "N=%d obs, K=%d, G=%d, Q=%d (1/%d of the per-GPU workload; obs/s is rate-normalised), "
                         "median of 3" % (sample_cfg["N"], K, sample_cfg["G"], Q, max(1, wl["N"] // sample_cfg["N"]))}
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["name"], "obs_per_gpu": wl["N"], "K": K, "groups_per_gpu": G,
                       "gh_points": Q, "free_dim": res["D"], "hessian_nnz": res["nnz"],
                       "parallelism": ("obs-sharded x%d (group-aligned shards, groups rank-private); one sum of "
                                       "[KL, grad_g, H_gg] per step by lrvb::k_p2p_allreduce over NVLink peer "
                                       "memory (csrc/p2p.cu); NCCL only for init / barriers" % world)
                       if world > 1 else "single GPU",
                       "l2": "flushed between timed steps (256 MiB write); X alone is %d MB"
                             % (wl["N"] * K * 8 // 10 ** 6),
                       "timing": "CUDA events per step on the launching stream, mean over steps, max over ranks; "
                                 "GC off and ranks synchronised before the last barrier, one untimed step after it"},
            "e2e": e2e, "lrvb_covariance": cov, "gpu_launches": res["launches"],
            "roofline": rooflines(res, wl, peak_tf, _load_traffic(args.workload)),
            "parity": parity, "cpu_baseline": cpu, "clocks": res["clocks"],
            "median_ms_max_over_ranks": res["median_ms_max_over_ranks"], "per_rank_ms": res["per_rank_ms"],
        }
        if "collective_wait_us" in res:
            line["collective_wait_us"] = res["collective_wait_us"]
    # free the headline workload before the target configuration
    for k in ("model", "local", "x_dev"):
        res.pop(k, None)
    del cov, e2e
    gc.collect()
    torch.cuda.empty_cache()

    # ---------------- target configuration: C3 (BASELINE configs[2]) ----------------
    if not args.no_target and args.workload == "c2":
        wt = WORKLOADS["c3"]
        tsteps, twarm = max(5, min(args.steps, 20)), 3
        tmode = "single" if world == 1 else "strong"
        rt = time_workload(ctx, wt, tmode, tsteps, twarm, kernel_steps=5)
        tcov = cov_entry(ctx, rt["model"], wt["K"], rt["local"].G, peak_tf, ncov=5)
        te2e = e2e_measure(ctx, rt, 5, 3) if world == 1 else None
        tline = None
        if rank == 0:
            tline = {"workload": wt["name"], "n_gpus": world,
                     "scaling": "strong" if world > 1 else "single GPU",
                     "value": rt["value"], "unit": UNIT, "ms_per_step": rt["ms_per_step"], "steps": tsteps,
                     "obs_total": rt["n_total"], "obs_this_rank": rt["n_local"], "hessian_nnz_this_rank": rt["nnz"],
                     "gpu_launches": rt["launches"], "lrvb_covariance": tcov,
                     "roofline": rooflines(rt, wt, peak_tf, _load_traffic("c3")),
                     "per_rank_ms": rt["per_rank_ms"],
                     "median_ms_max_over_ranks": rt["median_ms_max_over_ranks"]}
            if te2e is not None:
                tline["e2e"] = te2e
            if "collective_wait_us" in rt:
                tline["collective_wait_us"] = rt["collective_wait_us"]
                tline["partition"] = "distributed.partition_groups over the 100k balanced groups: %d obs on rank 0" \
                                     % rt["n_local"]
        for k in ("model", "local", "x_dev"):
            rt.pop(k, None)
        gc.collect()
        torch.cuda.empty_cache()
        if world > 1:
            # the same 10M problem on ONE GPU (rank 0) in the same process: the strong-scaling denominator
            dist.barrier()
            if rank == 0:
                r1 = time_workload(ctx_single(ctx), wt, "single", max(5, tsteps // 2), 3, kernel_steps=3)
                tline["one_gpu_same_run"] = {"value": r1["value"], "ms_per_step": r1["ms_per_step"],
                                             "steps": max(5, tsteps // 2)}
                tline["speedup_vs_one_gpu"] = rt["value"] / r1["value"]
                for k in ("model", "local", "x_dev"):
                    r1.pop(k, None)
                gc.collect()
                torch.cuda.empty_cache()
            dist.barrier()
        if rank == 0:
            line["target_config"] = tline

    if rank == 0:
        sys.stdout.flush()
        os.write(result_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(result_fd, 1)
    os.close(result_fd)


def ctx_single(ctx):
    c = Ctx()
    c.__dict__.update(ctx.__dict__)
    c.world = 1
    return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps of the headline measurement (c5: launches per family); the e2e, "
                         "kernel-time and target_config loops keep their own bounded counts, reported beside them")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS) + ["c5"])
    ap.add_argument("--no-target", action="store_true",
                    help="skip the target_config (C3) section of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy, float64, 64 MB at most: "
                         "KL, gradient and Hessian (COO; a seeded sample of its entries where they do not fit), "
                         "or for c5 each family's terms on a seeded sample of the factors; rank 0's at N > 1")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3   # timing rules: W >= 3
    wl = WORKLOADS.get(args.workload)
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
