#!/usr/bin/env python
"""Tile-shape sweep of the tcgen05 3xTF32 GEMM at the K3 forward shape (M = 1024 rows, K = 784, N = 256 samples x 104):
time per launch and per useful MAC for N tiles of 208 / 224 / 256 columns.  Run on a B200:
    for bn in 208 224 256; do BRN_GEMM_BN=$bn python profiles/gemm_bn_sweep.py; done"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from brancher_b200 import _cuda as cu

M, K, N = 1024, 784, 256 * 104
g = torch.Generator(device="cuda").manual_seed(0)
A = torch.randn(M, K, device="cuda", generator=g)
B = torch.randn(N, K, device="cuda", generator=g)
for _ in range(3):
    D = cu.gemm_nt_3xtf32(A, B)
torch.cuda.synchronize()
cu.profile_reset(); cu.profile_enable(True)
for _ in range(20):
    D = cu.gemm_nt_3xtf32(A, B)
torch.cuda.synchronize()
st = cu.profile_collect(); cu.profile_enable(False)
ms, calls = st["gemm.umma"]
ref = (A[:64].double() @ B[:512].double().T)
err = (D[:64, :512].double() - ref).abs().max().item()
print("BN=%s: %.1f us per launch, %.1f TFLOP/s fp32-equivalent, max err %.2e" % (
    os.environ.get("BRN_GEMM_BN", "224"), 1e3 * ms / calls,
    2.0 * M * N * K / (ms / calls * 1e-3) / 1e12, err))
