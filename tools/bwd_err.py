"""Worst per-block relative error of the VJP (vs the fp64 numpy oracle) per order K, for the kernel the library picks.
Debug aid for tests/test_backward_f16_gpu.py; run from the repo root."""
import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, torch
import chebnet_oracle as O
from helpers import random_weights
import test_backward_f16_gpu as T
from multihop_offload_b200 import LayerSpec
for K in (2, 4, 5, 6, 8, 10):
    rng = np.random.default_rng(300 + K)
    sizes = rng.integers(3, 129, size=90)
    mats = O.make_batch(sizes, seed0=7000 + K)
    n = int(sizes.sum())
    worst = []
    for act in (O.ACT_LEAKY, O.ACT_NONE):
        ws = random_weights([LayerSpec(K, 32, 32, act, 0.2)], rng, bias=0.2)
        X = rng.normal(size=(n, 32)); dY = rng.normal(size=(n, 32))
        gpg, gsum = T._run(torch, K, act, ws, mats, X, dY)
        ref = T._oracle(mats, X, ws, act, dY)
        errs = np.array([[T._block_err(gpg[g][k*1024:(k+1)*1024], ref[g][k*1024:(k+1)*1024], 0)[0] if False else
                          np.abs(gpg[g][k*1024:(k+1)*1024] - ref[g][k*1024:(k+1)*1024]).max() / max(np.abs(ref[g][k*1024:(k+1)*1024]).max(), 1e-300)
                          for k in range(K)] for g in range(len(mats))])
        worst.append(errs.max(0))
    w = np.maximum(*worst)
    print("K=%2d worst block errors:" % K, " ".join("%.1e" % e for e in w))
