"""Regression particles (K4a: brn_linreg_particles_loss_grad, Normal / Cauchy / Laplace likelihoods) against the Bernoulli particle
loss (brn_linear_particles_loss_grad) on the same data matrix, and one whole SVGD step (K4a + K4b) for each.

    python profiles/tools/regparticles_bench.py [--n 4096 --N 65536 --F 128 --steps 40 --warmup 5 --out FILE]

The C4 shape of bench.py's svgd workload: n = 4096 particles, N = 65536 rows, F = 128 features.  The regression calls share one
prepared X.  Each timed call is preceded by overwriting a 256 MiB buffer to flush the L2 (X alone is 32 MB and would otherwise
stay resident), and is timed with CUDA events around the eager call; the four likelihoods alternate call by call in one process,
so clock and neighbour effects fall on all of them alike.  Targets: y = X w* + 0.3 noise (Bernoulli: y ~ Bernoulli(sigmoid(X w*)),
Cauchy / Laplace: standard-Cauchy noise); particles w* + 0.3 N(0, 1).  Prints one JSON line with the GPU name and power limit
(read-only nvidia-smi query), ms per call (mean and p10 / p50 / p90), ratios to Bernoulli and the variants taken.  Needs a GPU:
there is no CPU path.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--N", type=int, default=65536)
    ap.add_argument("--F", type=int, default=128)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("regparticles_bench.py needs a CUDA device")
    from brancher_b200 import _cuda as cu
    dev = torch.device("cuda:0")
    n, N, F = a.n, a.N, a.F
    g = torch.Generator().manual_seed(0)
    X = torch.randn(N, F, generator=g)
    wstar = torch.randn(F, generator=g) / F ** 0.5
    y_gauss = (X @ wstar + 0.3 * torch.randn(N, generator=g)).to(dev)
    y_bern = (torch.rand(N, generator=g) < torch.sigmoid(X @ wstar)).float().to(dev)
    y_heavy = (X @ wstar + 0.3 * torch.tan(np.pi * (torch.rand(N, generator=g, dtype=torch.float64) - 0.5)).float()).to(dev)
    theta = (wstar[None, :] + 0.3 * torch.randn(n, F, generator=g)).to(dev).contiguous()
    X = X.to(dev).contiguous()
    prior_loc, prior_scale = torch.zeros(F, device=dev), torch.full((F,), 2.0, device=dev)
    scale = torch.full((1,), 0.3, device=dev)
    px = cu.PreparedX()
    ys = {"normal": y_gauss, "cauchy": y_heavy, "laplace": y_heavy}
    codes = {"normal": cu.GAUSSIAN, "cauchy": cu.CAUCHY, "laplace": cu.LAPLACE}

    def k4a(name):
        if name == "bernoulli":
            return cu.linear_particles_loss_grad(X, y_bern, cu.BERNOULLI, theta, 1, prior_loc, prior_scale)
        return cu.linreg_particles_loss_grad(X, ys[name], codes[name], theta, scale, prior_loc, prior_scale, prepared=px)

    def svgd_step(name):
        _, G = k4a(name)
        return cu.svgd_direction(theta, G)

    names = ["bernoulli", "normal", "cauchy", "laplace"]
    variants = {}
    for nm in names:                       # every workspace is grown (and X prepared) before timing
        k4a(nm)
        variants[nm] = cu.last_variant()
        svgd_step(nm)
    torch.cuda.synchronize()
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    times = {"k4a": {nm: [] for nm in names}, "svgd_step": {nm: [] for nm in names}}
    for i in range(a.warmup + a.steps):
        for kind, fn in (("k4a", k4a), ("svgd_step", svgd_step)):
            for nm in names:
                flush.fill_(float(i))
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                fn(nm)
                e.record()
                if i >= a.warmup:
                    times[kind][nm].append((s, e))
    torch.cuda.synchronize()
    ms = {k: {nm: [s.elapsed_time(e) for s, e in v] for nm, v in d.items()} for k, d in times.items()}
    mean = {k: {nm: float(np.mean(v)) for nm, v in d.items()} for k, d in ms.items()}
    out = dict(gpu_info(), n=n, N=N, F=F, steps=a.steps, warmup=a.warmup,
               method="eager calls, 256 MiB L2 flush before each, CUDA events, the likelihoods alternating call by call",
               variants=variants, ms_mean=mean,
               ms_p10_p50_p90={k: {nm: [float(np.percentile(v, q)) for q in (10, 50, 90)] for nm, v in d.items()} for k, d in ms.items()},
               ratio_to_bernoulli={k: {nm: d[nm] / d["bernoulli"] for nm in d} for k, d in mean.items()})
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
