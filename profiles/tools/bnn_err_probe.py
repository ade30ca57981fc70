#!/usr/bin/env python
"""Error of the K3 CUDA path against the fp64 oracle, relative to each tensor's own scale (max |g|), for one shape.
Run on a B200:  python profiles/tools/bnn_err_probe.py [B P H C S tied]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from brancher_b200 import _cuda as cu
from oracle import elbo_oracle as O
import test_cuda_kernels as T

args = [int(a) for a in sys.argv[1:6]] or [1024, 784, 100, 10, 4]
tied = (sys.argv[6] == "1") if len(sys.argv) > 6 else False
B, P, H, C, S = args
os.environ.setdefault("BRN_BNN_VARIANT", "tcgen05")
X, y, params, eps, shapes = T.random_bnn(B * 3 + H, B, P, H, C, S)
prior = None if tied else {n: (0.0, 10.0) for n in shapes}
l64, g64 = O.bnn_elbo(X, y, params, eps, prior, dtype=torch.float64, sample_chunk=4)
l32, g32 = O.bnn_elbo(X, y, params, eps, prior, sample_chunk=4)
loss, grads, _ = T.run_bnn(cu, X, y, params, eps, prior)
print("variant=%s  loss rel err %.2e (fp32 oracle %.2e)" % (
    cu.last_variant(),
    abs(loss - l64) / abs(l64), abs(l32 - l64) / abs(l64)))
for k in sorted(g64):
    sc = np.abs(g64[k]).max()
    e = np.abs(np.asarray(grads[k], dtype=np.float64).reshape(g64[k].shape) - g64[k])
    e32 = np.abs(np.asarray(g32[k], dtype=np.float64) - g64[k])
    lit = e > 1e-6 + 1e-5 * np.abs(g64[k])
    print("  %-16s scale %.3e  max err/scale: cuda %.2e  fp32-oracle %.2e   outside literal rtol1e-5/atol1e-6: %d/%d" % (
        k, sc, e.max() / sc, e32.max() / sc, lit.sum(), lit.size))
