"""Builds liblrvb_b200.so (the C-ABI CUDA library, sm_100a) in-tree with nvcc.

Usage: ``python linearresponsevariationalbayes.py_b200/build.py [--force] [--verbose]``
Called by ``__graft_entry__.build()``.  The .so is git-ignored but travels to the GPU box.
"""
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "lib", "liblrvb_b200.so")
SOURCES = ["api.cu", "glmm_eval.cu", "solve.cu", "csr.cu", "ef.cu", "sensitivity.cu", "p2p.cu", "packing.cu",
           "predict.cu", "logo.cu", "amip.cu", "ij.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xptxas", "-v",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the lrvb_b200 CUDA library cannot be built")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = _nvcc()
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(HERE, "..", "include", "lrvb_b200.h"))

    def compile_one(src):
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            cmd = [nvcc] + NVCC_FLAGS + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            log = r.stdout + r.stderr
            with open(o + ".log", "w") as f:
                f.write(log)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed for %s:\n%s" % (src, log))
            if verbose:
                print(log)
        return o

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    if force or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + \
              ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
