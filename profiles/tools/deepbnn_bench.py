#!/usr/bin/env python
"""Cost of the extra hidden layers of the K3 BNN: one ELBO evaluation (forward + backward + statistics) of the 784-100-10 network
(brn_bnn_elbo_fwd_bwd_act) and of the 784-100-100-10 and 784-100-100-100-10 networks (brn_bnn_deep_elbo_fwd_bwd), tanh and relu,
B = 1024, S = 256, Philox noise.  The six configurations alternate in one process and are timed with CUDA events; a separate
pass with the stage profiler gives the per-stage times.  For the new stages (bnn.deep_fwd, bnn.deep_bwd) it prints the FLOPs
and the minimum HBM bytes they need, computed from the shapes, and the rates achieved.  Prints JSON lines; the first holds the
GPU name and power limit (read-only nvidia-smi query).  Needs a GPU:  python profiles/tools/deepbnn_bench.py [reps]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from brancher_b200 import _cuda as cu  # noqa: E402
import deepbnn_models as dm  # noqa: E402

B, P, C, S = 1024, 784, 10, 256
NETS = {"784-100-10": (100,), "784-100-100-10": (100, 100), "784-100-100-100-10": (100, 100, 100)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def setup(H, act):
    X, y, params, _, shapes, layers = dm.random_net(5, B, P, H, C, 1, sigma=0.01, mu_scale=0.5)
    names = [n for pair in layers for n in pair]
    dev = torch.device("cuda:0")
    vs = [cu.MeanFieldVar(torch.tensor(params[n][0], device=dev), torch.tensor(params[n][1], device=dev), var_id=i)
          for i, n in enumerate(names)]
    Xd, yd = torch.tensor(X, device=dev), torch.tensor(y, dtype=torch.int32, device=dev)
    r = cu.sample_range(S, seed=1, offset=2)
    loss = torch.zeros(1, dtype=torch.float64, device=dev)
    if len(H) == 1:
        return lambda: cu.bnn_elbo_fwd_bwd(Xd, yd, vs, r, loss=loss, activation=act)
    return lambda: cu.bnn_deep_elbo_fwd_bwd(Xd, yd, vs, r, [act] * len(H), loss=loss)


def stage_needs(H):
    """FLOPs (useful multiply-adds x 2, not counting the 3-product split) and minimum HBM bytes of the new stages, per evaluation"""
    fwd_f = fwd_b = bwd_f = bwd_b = 0
    for l in range(1, len(H)):
        hin, hout = H[l - 1], H[l]
        fwd_f += 2 * S * B * hin * hout
        fwd_b += 4 * S * (B * hin * 2 + B * hout + hin * hout + hin)                 # pre in, h out, pre out, W, b
        bwd_f += 2 * 2 * S * B * hin * hout                                           # dh and dW
        bwd_b += 4 * S * (B * hout + B * hin * 2 + 2 * hin * hout + hin)              # dpre in, h in, dpre out, W, dW, db
    return {"bnn.deep_fwd": (fwd_f, fwd_b), "bnn.deep_bwd": (bwd_f, bwd_b)}


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    print(json.dumps(gpu_info()), flush=True)
    cfgs = [(net, act) for net in NETS for act in ("tanh", "relu")]
    runs = {c: setup(NETS[c[0]], c[1]) for c in cfgs}
    for c in cfgs:                       # warm-up: module load, workspace growth
        for _ in range(3):
            runs[c]()
    torch.cuda.synchronize()
    times = {c: [] for c in cfgs}
    for _ in range(reps):                # alternate the configurations; 5 evaluations per event pair
        for c in cfgs:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                runs[c]()
            e1.record()
            e1.synchronize()
            times[c].append(e0.elapsed_time(e1) / 5)
    variants = {}
    stages = {}
    for c in cfgs:                       # per-stage pass, profiler on
        cu.profile_reset()
        cu.profile_enable(True)
        for _ in range(10):
            runs[c]()
        st = cu.profile_collect()
        cu.profile_enable(False)
        variants[c] = cu.last_variant()
        stages[c] = {k: v[0] / v[1] for k, v in st.items() if v[1]}
    for c in cfgs:
        t = np.array(times[c])
        rec = {"net": c[0], "act": c[1], "B": B, "S": S, "variant": variants[c], "ms_mean": float(t.mean()),
               "ms_p10": float(np.percentile(t, 10)), "ms_p50": float(np.median(t)), "ms_p90": float(np.percentile(t, 90)),
               "stages_ms": {k: round(v, 4) for k, v in sorted(stages[c].items())}}
        H = NETS[c[0]]
        if len(H) > 1:
            rec["new_stages"] = {}
            for k, (f, b) in stage_needs(H).items():
                ms = stages[c].get(k)
                rec["new_stages"][k] = {"gflop": f / 1e9, "gbyte": b / 1e9, "ms": ms,
                                        "tflops": f / (ms * 1e-3) / 1e12 if ms else None,
                                        "tbps": b / (ms * 1e-3) / 1e12 if ms else None}
        print(json.dumps(rec), flush=True)
    # what one extra 100-wide layer costs, next to the layer-1 forward GEMM of the same run
    for act in ("tanh", "relu"):
        m = [float(np.median(times[(net, act)])) for net in NETS]
        g = stages[("784-100-100-10", act)].get("bnn.gemm_fwd")
        print(json.dumps({"act": act, "extra_layer_ms": [m[1] - m[0], m[2] - m[1]], "gemm_fwd_ms": g,
                          "extra_layer_over_gemm_fwd": [(m[1] - m[0]) / g, (m[2] - m[1]) / g] if g else None}), flush=True)


if __name__ == "__main__":
    main()
