"""Time one K2 evaluation (CUDA events around linear_elbo_fwd_bwd at the C2 shape, X re-prepared in every call) for each setting of
an environment switch: python profiles/tools/flash_time.py [VAR=value ...], e.g. default=1 BRN_LINEAR_FLASH=0.
(During development the kernel had a BRN_LF_DBG mask that skipped MMAs / epilogue math / loads / barriers to find the critical path:
profiles/r2f_flash_history.txt.)"""
import os, sys, torch
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from brancher_b200 import _cuda as cu
N, F, S = 1_000_000, 128, 1024
DEV = torch.device("cuda:0")
X = torch.randn(N, F, device=DEV); y = (torch.rand(N, device=DEV) < 0.5).float()
w = cu.MeanFieldVar(torch.zeros(1, F, device=DEV), torch.full((1, F), 0.5413, device=DEV), var_id=0,
                    prior_loc=torch.zeros(1, F, device=DEV), prior_scale=torch.full((1, F), 0.5, device=DEV))
r = cu.sample_range(S, seed=3, offset=5)
for setting in sys.argv[1:] or ["default=1"]:
    dbg = setting
    name, _, val = setting.partition("=")
    if name != "default":
        os.environ[name] = val
    for _ in range(3): cu.linear_elbo_fwd_bwd(X, y, cu.BERNOULLI, w, 1, r)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): cu.linear_elbo_fwd_bwd(X, y, cu.BERNOULLI, w, 1, r)
    e1.record(); torch.cuda.synchronize()
    print(dbg, "%.3f ms per call" % (e0.elapsed_time(e1) / 10))
    if name != "default":
        os.environ.pop(name, None)
