"""Quick device-step timing of one workload (A/B of library builds): prints ms per step,
per-kernel times, and checks the result against a reference build if LRVB_AB_REF is set."""
import os, sys, ctypes
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import lrvb_b200 as vb
from lrvb_b200 import _native as nat
import bench

wl = bench.WORKLOADS[sys.argv[1] if len(sys.argv) > 1 else "c2"]
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 30
dev = torch.device("cuda", 0)
X, y, g = bench.synth_shard(torch, wl["N"], wl["K"], wl["G"], 2000, dev)
model = vb.LogisticGLMM(X, y, g, num_gh_points=wl["Q"], num_groups=wl["G"])
gen = torch.Generator(device=dev); gen.manual_seed(7)
x = 0.1 * torch.randn(model.D, dtype=torch.float64, device=dev, generator=gen)
flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
lib = nat.load()
def step():
    model.evaluate(x, 2, force=True)
    return model.hessian_csr()
for _ in range(5):
    flush.zero_(); csr = step()
torch.cuda.synchronize()
ts = []
for _ in range(steps):
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); csr = step(); e1.record(); e1.synchronize()
    ts.append(e0.elapsed_time(e1))
ms3 = (ctypes.c_float * 3)()
nat.check(lib.lrvb_glmm_set_timing(model._h, 1))
ev, ob, gr = [], [], []
for i in range(8):
    flush.zero_(); csr = step(); torch.cuda.synchronize()
    nat.check(lib.lrvb_glmm_last_timing(model._h, ms3))
    if i >= 3:
        ev.append(ms3[0]); ob.append(ms3[1]); gr.append(ms3[2])
A, B, L = model.blocks()
chk = float(A.abs().sum() + B.abs().sum() + L.abs().sum() + model.kl_tensor().abs() + model.grad_tensor().abs().sum())
print("%s lib=%s: step %.4f ms (min %.4f) eval %.4f obs/onepass %.4f gram %.4f  checksum %.15e" % (
    sys.argv[1] if len(sys.argv) > 1 else "c2", os.path.basename(nat.LIB_PATH), np.mean(ts), np.min(ts), np.mean(ev),
    np.mean(ob), np.mean(gr), chk))
