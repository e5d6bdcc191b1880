"""bench.py --workload c5: BASELINE.json configs[4] -- mean-field Gamma / Dirichlet / Beta / Wishart / UVN
exponential-family entropy and E-log terms (ExponentialFamilies.py:5-120) batched over 1M local factors.

A step = one launch per family over 1M factors resident in HBM.  The launches are a few microseconds of
HBM traffic each (16 - 80 B per factor), so the device numbers are taken from a CUDA-graph replay of the
C-ABI calls (the Python / ctypes call overhead of ~20 us per launch would otherwise be the measurement);
`e2e` goes through the public Python functions with host buffers.  Roofline: HBM (SURVEY.md 8(d): algorithmic
bytes per factor = 8 x (inputs + outputs))."""
import ctypes
import json
import os
import time

import numpy as np

METRIC = "exponential-family factors/sec for entropy + E-log terms (BASELINE configs[4], 1M local factors)"
UNIT = "factors/s"
M = 1_000_000


def _hbm():
    import bench
    return bench._hbm_peak(), bench._hbm_peak_source()


def make_inputs(torch, device, seed=5):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    f64 = dict(dtype=torch.float64, device=device, generator=g)
    shape = torch.exp(0.5 * torch.randn(M, **f64))
    rate = torch.exp(0.5 * torch.randn(M, **f64))
    alpha = 10 * torch.rand(5, M, **f64) + 0.1
    tau = 5 * torch.rand(M, 2, **f64) + 0.1
    A = torch.randn(M, 2, 2, **f64)
    v = (A @ A.transpose(1, 2) + torch.eye(2, dtype=torch.float64, device=device)).contiguous()
    df = 3 + 5 * torch.rand(M, **f64)
    info = torch.exp(0.5 * torch.randn(M, **f64))
    return dict(shape=shape, rate=rate, alpha=alpha, tau=tau, v=v, df=df, info=info)


def cpu_terms(inp):
    """The reference's formulas with numpy / scipy (ExponentialFamilies.py:23-25, 33-35, 43-52, 54-69, 111-112,
    118-120) on host copies -- the CPU arm and the parity check."""
    import scipy.special as sp
    a, b, al, tau, info = inp["shape"], inp["rate"], inp["alpha"], inp["tau"], inp["info"]
    out = {}
    out["gamma_entropy"] = a - np.log(b) + sp.gammaln(a) + (1 - a) * sp.digamma(a)
    out["gamma_e_log"] = sp.digamma(a) - np.log(b)
    sa = al.sum(0)
    logb = sp.gammaln(al).sum(0) - sp.gammaln(sa)
    out["dirichlet_entropy"] = logb - (al.shape[0] - sa) * sp.digamma(sa) - ((al - 1) * sp.digamma(al)).sum(0)
    out["dirichlet_e_log"] = sp.digamma(al) - sp.digamma(sa)[None, :]
    s = tau.sum(1)
    lbeta = sp.gammaln(tau[:, 0]) + sp.gammaln(tau[:, 1]) - sp.gammaln(s)
    out["beta_entropy"] = (lbeta - (tau[:, 0] - 1) * sp.digamma(tau[:, 0]) - (tau[:, 1] - 1) * sp.digamma(tau[:, 1])
                           + (s - 2) * sp.digamma(s))
    out["uvn_entropy"] = 0.5 * (-np.log(info) + 1 + np.log(2 * np.pi))
    return out


def run_reference(args):
    import torch
    inp = {k: v.numpy() for k, v in make_inputs(torch, torch.device("cpu")).items()}
    sub = {k: (v[..., :M // 4] if k == "alpha" else v[:M // 4]) for k, v in inp.items()}
    n = M // 4
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_terms(sub)
    ts = []
    for _ in range(args.steps):
        t = time.perf_counter()
        cpu_terms(sub)
        ts.append(time.perf_counter() - t)
    ms = 1e3 * float(np.mean(ts))
    value = n / (ms * 1e-3)
    sample = "%d of the 1M factors per step, every family once (numpy / scipy.special, 1 thread)" % n
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "mean-field EF entropy / E-log terms over 1M local factors (BASELINE configs[4])",
                       "cpu_sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def sample_factors(n_values):
    """Sorted factor indices drawn with a fixed seed: the factors whose results --dump-outputs writes when
    ``n_values`` float64 values per factor would take all 1M factors past bench.DUMP_BYTES."""
    import bench
    n = min(M, (bench.DUMP_BYTES - 4096) // (8 * n_values))      # 4096: the .npy headers
    return np.sort(np.random.default_rng(0).choice(M, size=n, replace=False))


def run_ours(ctx, args, dump=False):
    """Returns (JSON line, outputs): with ``dump``, outputs holds the results of the last timed launch of
    each family of the step, on the host for the factors of sample_factors; otherwise None."""
    torch, nat, lib, vb = ctx.torch, ctx.nat, ctx.lib, ctx.vb
    ef = vb.ExponentialFamilies
    dev = ctx.device
    inp = make_inputs(torch, dev, seed=5 + ctx.rank)
    hbm, hbm_src = _hbm()
    out1 = torch.empty(M, dtype=torch.float64, device=dev)
    out2 = torch.empty(M, dtype=torch.float64, device=dev)
    outd = torch.empty(5, M, dtype=torch.float64, device=dev)
    st = torch.cuda.Stream()
    sp = ctypes.c_void_p(st.cuda_stream)
    P = nat.ptr
    cases = [
        # name, launch, algorithmic bytes per factor (8 x (inputs + outputs)), results kept by --dump-outputs
        ("gamma entropy + E log (fused)", lambda: lib.lrvb_ef_gamma_terms(P(inp["shape"]), P(inp["rate"]), M, P(out1), P(out2), sp), 32,
         (("gamma_entropy", out1), ("gamma_e_log", out2))),
        ("gamma entropy", lambda: lib.lrvb_ef_gamma_terms(P(inp["shape"]), P(inp["rate"]), M, P(out1), None, sp), 24, ()),
        ("E log gamma", lambda: lib.lrvb_ef_gamma_terms(P(inp["shape"]), P(inp["rate"]), M, None, P(out2), sp), 24, ()),
        ("dirichlet (d=5) entropy + E log (fused)", lambda: lib.lrvb_ef_dirichlet_terms(P(inp["alpha"]), 5, M, P(out1), P(outd), sp), 88,
         (("dirichlet_entropy", out1), ("dirichlet_e_log", outd))),
        ("dirichlet (d=5) entropy", lambda: lib.lrvb_ef_dirichlet_terms(P(inp["alpha"]), 5, M, P(out1), None, sp), 48, ()),
        ("beta entropy", lambda: lib.lrvb_ef_beta_entropy(P(inp["tau"]), M, P(out1), sp), 24, (("beta_entropy", out1),)),
        ("uvn entropy", lambda: lib.lrvb_ef_uvn_entropy(P(inp["info"]), M, P(out1), sp), 16, (("uvn_entropy", out1),)),
    ]
    rows = []
    total_ms = 0.0
    outputs, pick = None, None
    if dump:
        outputs = {}
        pick = torch.from_numpy(sample_factors(10)).to(dev)   # 10 values per factor: 2 gamma, 6 dirichlet, beta, uvn
    launches0 = lib.lrvb_launch_count()
    for name, fn, bpf, keep in cases:
        with torch.cuda.stream(st):
            for _ in range(args.warmup):
                nat.check(fn())
            st.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=st):
                for _ in range(args.steps):
                    nat.check(fn())
            graph.replay()                  # untimed: the first replay uploads the graph
            st.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            graph.replay()
            e1.record(st)
            e1.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
        if outputs is not None:
            for oname, buf in keep:
                outputs[oname] = buf[..., pick].cpu().numpy()
        gbs = M * bpf / (ms * 1e-3) / 1e9
        rows.append({"family": name, "us": 1e3 * ms, "factors_per_s": M / (ms * 1e-3), "bytes_per_factor": bpf,
                     "achieved_gbs": gbs, "frac_of_hbm": gbs / hbm})
        if "fused" in name or name in ("beta entropy", "uvn entropy"):
            total_ms += ms
    launches = lib.lrvb_launch_count() - launches0
    # Wishart (k = 2) through the Python function (its C entry point synchronises for the PD status)
    for _ in range(args.warmup):
        ef.wishart_entropy(inp["df"], inp["v"])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        ef.wishart_entropy(inp["df"], inp["v"])
    e1.record()
    e1.synchronize()
    wms = e0.elapsed_time(e1) / args.steps
    rows.append({"family": "wishart (k=2) entropy, Python call incl. status sync", "us": 1e3 * wms,
                 "factors_per_s": M / (wms * 1e-3), "bytes_per_factor": 48,
                 "achieved_gbs": M * 48 / (wms * 1e-3) / 1e9, "frac_of_hbm": M * 48 / (wms * 1e-3) / 1e9 / hbm})
    # parity of every family against the numpy / scipy restatement of the reference formulas
    host = {k: v.cpu().numpy() for k, v in inp.items()}
    ref = cpu_terms(host)
    ge, gl = ef.gamma_entropy_and_e_log(inp["shape"], inp["rate"])
    de, dl = ef.dirichlet_entropy_and_e_log(inp["alpha"])
    got = {"gamma_entropy": ge, "gamma_e_log": gl, "dirichlet_entropy": de, "dirichlet_e_log": dl,
           "beta_entropy": ef.beta_entropy_batched(inp["tau"]),
           "uvn_entropy": ef.univariate_normal_entropy_batched(inp["info"])}
    parity = {}
    for k, r in ref.items():
        g = got[k].cpu().numpy()
        parity[k] = float(np.max(np.abs(g - r) / np.maximum(1.0, np.abs(r))))
    parity["ok"] = bool(max(parity.values()) < 1e-9)
    parity["against"] = "numpy / scipy.special restatement of ExponentialFamilies.py on the same 1M factors"
    # end to end: host arrays in, host arrays out, through the public functions
    t0 = time.perf_counter()
    for _ in range(3):
        a, b = ef.gamma_entropy_and_e_log(host["shape"], host["rate"])
        c, d = ef.dirichlet_entropy_and_e_log(host["alpha"])
        e = ef.beta_entropy_batched(host["tau"])
        f = ef.univariate_normal_entropy_batched(host["info"])
    e2e_s = (time.perf_counter() - t0) / 3
    # CPU arm
    sub = {k: (v[..., :M // 4] if k == "alpha" else v[:M // 4]) for k, v in host.items()}
    cpu_terms(sub)
    ts = []
    for _ in range(3):
        t = time.perf_counter()
        cpu_terms(sub)
        ts.append(time.perf_counter() - t)
    dom = max(rows[:7], key=lambda r: r["us"])
    line = {
        "metric": METRIC, "value": M / (total_ms * 1e-3), "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "mean-field EF entropy / E-log terms over 1M local factors (BASELINE configs[4]): "
                               "a step = Gamma (entropy + E log) + Dirichlet d=5 (entropy + E log) + Beta entropy "
                               "+ UVN entropy, one launch per family",
                   "timing": "per family, --steps C-ABI launches captured in one CUDA graph and replayed once, CUDA "
                             "events on the launching stream.  A family's inputs (8 - 40 MB) are smaller than the 126 MB L2 and are "
                             "re-read by consecutive launches, so they may be L2-resident: frac_of_hbm measures "
                             "the kernels' rate against the HBM roofline figure, not DRAM efficiency (these "
                             "kernels are bound by fp64 special-function throughput)",
                   "families": rows},
        "e2e": {"value": M / e2e_s, "unit": UNIT, "ms_per_step": 1e3 * e2e_s,
                "h2d_bytes_per_step": 8 * M * (2 + 5 + 2 + 1), "d2h_bytes_per_step": 8 * M * (2 + 6 + 1 + 1),
                "api": "ExponentialFamilies.gamma_entropy_and_e_log / dirichlet_entropy_and_e_log / "
                       "beta_entropy_batched / univariate_normal_entropy_batched with numpy arrays"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "lrvb::" + ("k_dirichlet_terms" if "dirichlet" in dom["family"] else
                                                           "k_gamma_terms") + " (" + dom["family"] + ")",
                     "achieved": dom["achieved_gbs"], "peak": hbm, "unit": "GB/s", "frac": dom["frac_of_hbm"],
                     "traffic": None, "peak_source": hbm_src, "bytes_per_factor": dom["bytes_per_factor"]},
        "parity": parity,
        "cpu_baseline": {"value": (M // 4) / float(np.median(ts)), "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": "%d of the 1M factors, every family once, numpy / scipy.special; median of 3" % (M // 4)},
        "clocks": None,
    }
    return line, outputs
