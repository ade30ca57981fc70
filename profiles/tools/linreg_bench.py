"""Bayesian linear regression (K2g, brn_linreg_elbo_fwd_bwd_lik: Normal, Cauchy and Laplace likelihoods) against the Bernoulli K2
evaluation on the same data matrix.

    python profiles/tools/linreg_bench.py [--N 1000000 --F 128 --S 1024 --steps 60 --warmup 10]

N = 10^6 rows, F = 128 features, S = 1024 samples, one prepared X shared by every evaluation.  Method of bench.py (DESIGN.md
section 6): each evaluation (loss and gradient buffers zeroed, then one fused call) is captured once in a CUDA graph and
replayed; a 256 MiB buffer is overwritten between timed replays to flush the L2; CUDA events time each replay.  The seven
evaluations -- Bernoulli, then Gaussian, Cauchy and Laplace each with a fixed noise scale and with a LogNormal noise latent --
alternate replay by replay in one process, so clock and neighbour effects fall on all of them alike.  The Cauchy and Laplace
targets are y = X w* + 0.3 standard-Cauchy noise.  Prints one JSON line: GPU name and power limit
(read-only nvidia-smi query), ms per evaluation, the ratio to Bernoulli and the fraction of the 3xFP16 roofline (4 S N F flop
at a third of the bf16 dense rate).  Needs a GPU: there is no CPU path.
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


def bf16_burst_tflops():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["bf16_tflops"]), "measured (MEASURED_PEAKS.json)"
    return 1590.0, "fallback (bench.py)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=1_000_000)
    ap.add_argument("--F", type=int, default=128)
    ap.add_argument("--S", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("linreg_bench.py needs a CUDA device")
    from brancher_b200 import _cuda as cu
    from oracle.elbo_oracle import softplus_inverse
    dev = torch.device("cuda:0")
    N, F, S = a.N, a.F, a.S
    g = torch.Generator().manual_seed(0)
    X = torch.randn(N, F, generator=g)
    wstar = torch.randn(F, generator=g) / F ** 0.5
    y_gauss = (X @ wstar + 0.3 * torch.randn(N, generator=g)).to(dev)
    y_bern = (torch.rand(N, generator=g) < torch.sigmoid(X @ wstar)).float().to(dev)
    y_heavy = (X @ wstar + 0.3 * torch.tan(np.pi * (torch.rand(N, generator=g, dtype=torch.float64) - 0.5)).float()).to(dev)
    X = X.to(dev).contiguous()
    px = cu.PreparedX()
    mu = torch.zeros(1, F, device=dev)
    rho = torch.full((1, F), float(softplus_inverse(0.05)), device=dev)
    w = cu.MeanFieldVar(mu, rho, var_id=0)
    nu = cu.MeanFieldVar(torch.full((1,), float(np.log(0.3)), device=dev), torch.full((1,), -2.0, device=dev), var_id=1)
    scale = torch.full((1,), 0.3, device=dev)
    r = cu.sample_range(S, seed=1, offset=0)
    loss = torch.zeros(1, dtype=torch.float64, device=dev)

    def zero():
        loss.zero_(); w.dmu.zero_(); w.drho.zero_(); nu.dmu.zero_(); nu.drho.zero_()

    evals = {
        "bernoulli": lambda: cu.linear_elbo_fwd_bwd(X, y_bern, cu.BERNOULLI, w, 1, r, loss=loss, prepared=px),
        "gaussian_fixed": lambda: cu.linreg_elbo_fwd_bwd(X, y_gauss, w, r, noise_scale=scale, loss=loss, prepared=px),
        "gaussian_lognormal": lambda: cu.linreg_elbo_fwd_bwd(X, y_gauss, w, r, nu=nu, loss=loss, prepared=px),
    }
    for lik, name in ((cu.CAUCHY, "cauchy"), (cu.LAPLACE, "laplace")):
        evals[name + "_fixed"] = (lambda lik=lik: cu.linreg_elbo_fwd_bwd(X, y_heavy, w, r, noise_scale=scale, loss=loss, prepared=px,
                                                                          likelihood=lik))
        evals[name + "_lognormal"] = (lambda lik=lik: cu.linreg_elbo_fwd_bwd(X, y_heavy, w, r, nu=nu, loss=loss, prepared=px,
                                                                              likelihood=lik))
    variants = {}
    for name, fn in evals.items():          # every workspace is grown (and X prepared) before the first capture
        zero(); fn()
        variants[name] = cu.last_variant()
    torch.cuda.synchronize()
    graphs = {}
    for name, fn in evals.items():
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            zero(); fn()
        graphs[name] = gr
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    for i in range(a.warmup):
        for gr in graphs.values():
            flush.fill_(float(i)); gr.replay()
    torch.cuda.synchronize()
    evs = {n: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)] for n in graphs}
    for i in range(a.steps):
        for n, gr in graphs.items():
            flush.fill_(float(i))
            evs[n][i][0].record()
            gr.replay()
            evs[n][i][1].record()
    torch.cuda.synchronize()
    ms = {n: float(np.mean([s.elapsed_time(e) for s, e in evs[n]])) for n in graphs}
    spread = {n: [float(np.percentile([s.elapsed_time(e) for s, e in evs[n]], q)) for q in (10, 50, 90)] for n in graphs}
    # per-stage split (StageTimer events), in a separate eager pass after the timed replays: the events are not in the graphs
    stages = {}
    for name, fn in evals.items():
        cu.profile_reset(); cu.profile_enable(True)
        for _ in range(10):
            flush.fill_(0.0); zero(); fn()
        st = cu.profile_collect()
        cu.profile_enable(False)
        stages[name] = {k: v[0] / v[1] for k, v in st.items() if v[1] > 0}
    bf16, peak_src = bf16_burst_tflops()
    roof_ms = 4.0 * S * N * F / (bf16 / 3 * 1e12) * 1e3
    out = dict(gpu_info(), N=N, F=F, S=S, steps=a.steps, warmup=a.warmup, method="CUDA graph replay, 256 MiB L2 flush between "
               "replays, CUDA events, the evaluations alternating", variants=variants,
               ms_per_eval=ms, ms_p10_p50_p90=spread, ratio_to_bernoulli={n: ms[n] / ms["bernoulli"] for n in ms},
               frac_3xfp16_roofline={n: roof_ms / ms[n] for n in ms}, roofline_ms=roof_ms,
               stage_ms_eager=stages,
               roofline="4 S N F flop at bf16 burst / 3 = %.0f TFLOP/s, peak %s" % (bf16 / 3, peak_src))
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
