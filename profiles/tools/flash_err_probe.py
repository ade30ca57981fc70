"""Probe: signed loss / gradient error of the K2 variants (staged GEMM pair, one-pass kernel, the latter also with y at a 4-byte
offset, which loads the targets per lane) against the fp64 oracle at a C2-shaped problem.  Usage: python profiles/tools/flash_err_probe.py [N] [S]
(This probe found the loss error that grew linearly with N: a per-thread fp32 running sum of the log-likelihood.)"""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from brancher_b200 import _cuda as cu
from oracle import elbo_oracle as O

N = int(sys.argv[1]) if len(sys.argv) > 1 else 262144
S = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
F = 128
DEV = torch.device("cuda:0")
g = torch.Generator().manual_seed(0)
X = torch.randn(N, F, generator=g)
wstar = torch.randn(F, generator=g) / F ** 0.5
y = (torch.rand(N, generator=g) < torch.sigmoid(X @ wstar)).float()
params = {"weights": (np.zeros((1, F), "f4"), O.softplus_inverse(np.ones((1, F))).astype("f4"))}
prior = {"weights": (0.0, 0.5)}
r = cu.sample_range(S, seed=3, offset=5)
eps = {"weights": cu.philox_normal(F, 0, r, DEV).cpu().numpy().reshape(S, 1, F)}
l64, g64 = O.logreg_elbo_streamed(X.numpy(), y.numpy(), params, eps, prior)
Xd, yd = X.to(DEV), y.to(DEV)
y_off = torch.empty(N + 1, device=DEV)[1:]
y_off.copy_(yd)
for env, yt in (({"BRN_LINEAR_FLASH": "0"}, yd), ({}, yd), ({}, y_off)):
    os.environ.pop("BRN_LINEAR_FLASH", None)
    os.environ.update(env)
    w = cu.MeanFieldVar(torch.tensor(params["weights"][0], device=DEV), torch.tensor(params["weights"][1], device=DEV), var_id=0,
                        prior_loc=torch.zeros(1, F, device=DEV), prior_scale=torch.full((1, F), 0.5, device=DEV))
    loss = cu.linear_elbo_fwd_bwd(Xd, yt, cu.BERNOULLI, w, 1, r).item()
    gm = w.dmu.cpu().numpy().reshape(1, F); gs = w.drho.cpu().numpy().reshape(1, F)
    print(env, "y offset %d" % (yt.data_ptr() % 16), cu.last_variant(), "loss rel err %+.3e" % ((loss - l64) / abs(l64)),
          "dmu %.3e drho %.3e" % (np.abs(gm - g64["weights_loc"]).max() / np.abs(g64["weights_loc"]).max(),
                                  np.abs(gs - g64["weights_scale"]).max() / np.abs(g64["weights_scale"]).max()))
