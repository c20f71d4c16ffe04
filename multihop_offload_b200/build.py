"""Build libmho.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmho.so")
SOURCES = ["mho_api.cu", "cheb_forward.cu", "cheb_forward_dense.cu", "cheb_forward_f16.cu", "cheb_mlp_f16.cu", "cheb_backward.cu", "cheb_backward_f16.cu", "cheb_mlp_backward_f16.cu", "optimizer.cu", "queue_head.cu", "apsp.cu", "env_step.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xptxas=-v", "-Xcompiler", "-fPIC", "-shared"]


def nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "mho.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    probe = bool(os.environ.get("MHO_PROBE"))   # instrumented build (clock marks printed by the forward kernels): libmho_probe.so
    extra = ["-DMHO_PROBE"] if probe else []
    out = LIB.replace("libmho.so", "libmho_probe.so") if probe else LIB
    if os.environ.get("MHO_EXTRA_FLAGS"):   # experiment builds: MHO_EXTRA_FLAGS="-DFOO" MHO_OUT=libmho_foo.so
        extra += os.environ["MHO_EXTRA_FLAGS"].split()
        out = os.path.join(HERE, os.environ.get("MHO_OUT", "libmho_exp.so"))
    cmd = [nvcc()] + NVCC_FLAGS + extra + ["-o", out] + srcs + ["-lcudart"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libmho.so")
    return out


if __name__ == "__main__":
    build(force=True, verbose=True)
    print(LIB)
