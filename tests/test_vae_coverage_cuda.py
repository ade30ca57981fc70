"""K5 (brn_vae_elbo_fwd_bwd) on every tile width, latent size, depth, K-split regime and operand layout its host code can
select, against the fp32 / fp64 oracle.

`CASES` is a plain list: tests/test_vae_coverage.py walks it through a mirror of the host-side selections of vae.cu and
umma_gemm.cuh and fails (on the CPU) when an edit of the table leaves a branch unreached.

ReLU kinks: a unit whose pre-activation lies within rounding error of zero is switched on by one correct fp32 evaluation and
off by another (see test_c5_vae_full_config).  Each case therefore draws more data rows than it runs, and keeps the first B
rows whose every ReLU pre-activation is at least 4e-6 (relative to its own terms) away from the kink in the fp64 forward pass.

Run as a script (`python test_vae_coverage_cuda.py IN.npz... -- OUT_DIR`), the file evaluates saved inputs in a fresh process,
so that the selections vae.cu fixes at its first call in a process (BRN_VAE_EW16, BRN_VAE_CW, BRN_VAE_WGRAD_TILE) can be
tested."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MARGIN = 4e-6          # relative ReLU margin below which a data row is left out (test_c5_vae_full_config)


def tail_split_case(sms, S=8, B=50):
    """The case whose output-layer weight gradient takes umma_plan's "tail units split" regime on `sms` SMs.

    That GEMM is M = D (output width) by N = 1200 (last decoder width: the 128-wide MN-major tile, 10 n-tiles) over
    K = S * B rows.  D = 128 m - 48 for the smallest m with U = 10 m > sms units, T = U % sms tail units, 2 T <= sms and
    ceil(K / 16) >= 2 (sms // T) K chunks (umma_gemm.cuh:486).  148 SMs: D = 2000, U = 160, T = 12."""
    k_chunks = (S * B + 15) // 16
    m = sms // 10 + 1
    while True:
        U = 10 * m
        T = U % sms
        if U > sms and T > 0 and 2 * T <= sms and k_chunks >= 2 * (sms // T):
            break
        m += 1
    return dict(name="tail_split", B=B, D=128 * m - 48, L=16, h_enc=(512,), h_dec=(1024, 1200), S=S, seed=105, row_chunk=25)


# name, shape and seed of each case; the branches each one reaches are listed by tests/test_vae_coverage.py
CASES = [
    dict(name="w176_B1", B=1, D=150, L=1, h_enc=(300,), h_dec=(512, 500), S=8, seed=101),
    dict(name="deep6", B=31, D=5, L=4, h_enc=(40, 64, 33, 250, 48, 20), h_dec=(20, 250, 300, 30, 1000, 16), S=3, seed=102),
    dict(name="h513_L8", B=33, D=50, L=8, h_enc=(256,), h_dec=(513, 256), S=5, seed=103),
    dict(name="h1024_L9", B=77, D=784, L=9, h_enc=(200,), h_dec=(1024,), S=4, seed=104),
    tail_split_case(148),
    dict(name="out256", B=40, D=256, L=2, h_enc=(150, 500), h_dec=(200, 300), S=6, seed=106),
    dict(name="D1_L16", B=33, D=1, L=16, h_enc=(250,), h_dec=(64, 250), S=2, seed=107),
    dict(name="out512_split300", B=64, D=512, L=3, h_enc=(1000, 64), h_dec=(300,), S=8, seed=108),
    dict(name="out1000_L5", B=20, D=1000, L=5, h_enc=(500,), h_dec=(250, 150), S=6, seed=109),
    dict(name="D300_h1024enc", B=9, D=300, L=2, h_enc=(1024, 150), h_dec=(64,), S=7, seed=110),
]
CASE = {c["name"]: c for c in CASES}

# BRN_VAE_WGRAD_MN=0 (transposed K-major operands, read on every call): the 176, 208 and -128 tiles and L = 16
TRANSPOSED = ["w176_B1", "deep6", "h1024_L9", "out256", "D1_L16", "D300_h1024enc"]
# selections fixed at the first call in a process: one child process per setting, each on CHILD_CASES
CHILD_SETTINGS = [("BRN_VAE_EW16", "0"), ("BRN_VAE_CW", "4"), ("BRN_VAE_WGRAD_TILE", "0"), ("BRN_VAE_WGRAD_TILE", "1")]
CHILD_CASES = ["h513_L8", "h1024_L9", "D300_h1024enc"]


@pytest.fixture(scope="module")
def cu():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from brancher_b200 import _cuda
    _cuda.lib()
    return _cuda


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def case_inputs(c, sd_offset=0.1, saturate=False):
    """(X, enc, dec, eps, kept fraction): the first B of the drawn rows that keep every ReLU pre-activation MARGIN away
    from its kink.  saturate: output biases of magnitude 35..85 and W_out scaled by 4, so that most logits lie far in the
    flat tails of the sigmoid (the output layer has no kink to move)."""
    from oracle import elbo_oracle as O
    import test_vae_cuda as V
    B = c["B"]
    B_draw = 2 * B + 8
    X, enc, dec, eps = V.random_vae(c["seed"], B_draw, c["D"], c["L"], c["h_enc"], c["h_dec"], c["S"])
    if saturate:
        rng = np.random.RandomState(c["seed"] + 1)
        D = c["D"]
        dec["b_out"] = (np.where(rng.rand(D) < 0.5, -1.0, 1.0) * rng.uniform(35.0, 85.0, D)).astype("f4")
        dec["W_out"] = (4.0 * dec["W_out"]).astype("f4")
    clean = O.vae_relu_margins(X, enc, dec, eps, sd_offset=sd_offset) >= MARGIN
    assert clean.mean() > 0.5 and clean.sum() >= B, "%s: %d of %d rows away from ReLU kinks" % (c["name"], clean.sum(), B_draw)
    idx = np.flatnonzero(clean)[:B]
    return np.ascontiguousarray(X[idx]), enc, dec, np.ascontiguousarray(eps[:, idx]), float(clean.mean())


def oracles(X, enc, dec, eps, sd_offset=0.1, row_chunk=None):
    from oracle import elbo_oracle as O
    o32 = O.vae_elbo(X, enc, dec, eps, sd_offset=sd_offset, row_chunk=row_chunk)
    o64 = O.vae_elbo(X, enc, dec, eps, sd_offset=sd_offset, dtype=torch.float64, row_chunk=row_chunk)
    return o32, o64


_prepared = {}


def prepared(name):
    """inputs and oracle results of a table case, computed once per process"""
    if name not in _prepared:
        c = CASE[name]
        X, enc, dec, eps, kept = case_inputs(c)
        _prepared[name] = (X, enc, dec, eps, kept) + oracles(X, enc, dec, eps, row_chunk=c.get("row_chunk"))
    return _prepared[name]


def run_cuda(cu, X, enc, dec, eps, sd_offset=0.1):
    import test_vae_cuda as V
    net = V.make_net(cu, enc, dec, sd_offset=sd_offset)
    loss = cu.vae_elbo_fwd_bwd(V.dev(X), net, cu.sample_range(eps.shape[0]), eps=V.dev(eps)).item()
    assert cu.last_variant() == "tcgen05"
    return loss, V.grads_of(net)


def check(what, loss, grads, o32, o64):
    """the repository's parity rule, and one line with the largest error over tensor scale against fp64"""
    from helpers import check_against_oracle
    worst = max(abs(loss - o64[0]) / max(abs(o64[0]), 1.0),
                max(np.abs(np.asarray(grads[k], np.float64).reshape(g.shape) - g).max() / max(np.abs(g).max(), 1e-8)
                    for k, g in o64[1].items()))
    print("vae coverage %-40s max |cuda - fp64| / scale = %.2e" % (what, worst))
    check_against_oracle(loss, grads, o32, o64, what)


@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_vae_coverage_case(cu, name):
    X, enc, dec, eps, kept, o32, o64 = prepared(name)
    loss, grads = run_cuda(cu, X, enc, dec, eps)
    check("%s (%.0f %% rows kept)" % (name, 100 * kept), loss, grads, o32, o64)


def test_vae_tail_split_regime_on_this_device(cu):
    """The tail-split case is built for the device's SM count, and umma_plan's mirror puts its output-layer weight gradient
    in the "tail units split" regime there; on a device other than the 148-SM B200 the case is rebuilt and run."""
    import test_vae_coverage as M
    sms = sm_count()
    c = tail_split_case(sms)
    assert M.umma_regime(128, c["D"], c["h_dec"][-1], c["S"] * c["B"], sms) == "tail"
    if c == CASE["tail_split"]:
        return          # run by test_vae_coverage_case
    X, enc, dec, eps, kept = case_inputs(c)
    loss, grads = run_cuda(cu, X, enc, dec, eps)
    check("tail_split for %d SMs" % sms, loss, grads, *oracles(X, enc, dec, eps, row_chunk=c["row_chunk"]))


@pytest.mark.parametrize("name", TRANSPOSED)
def test_vae_coverage_transposed_layouts(cu, monkeypatch, name):
    """BRN_VAE_WGRAD_MN=0: transposed K-major copies of every activation and gradient, the K-major weight-gradient GEMM on
    pick_bn's tiles, the transposed stores of store_split4 / vae_sample_dec0_kernel / vae_heads_bwd_kernel and the transposed
    TF32 split of X"""
    monkeypatch.setenv("BRN_VAE_WGRAD_MN", "0")
    X, enc, dec, eps, kept, o32, o64 = prepared(name)
    loss, grads = run_cuda(cu, X, enc, dec, eps)
    check("%s WGRAD_MN=0" % name, loss, grads, o32, o64)


@pytest.mark.parametrize("sd_offset", [1e-3, 1.0])
def test_vae_sd_offset(cu, sd_offset):
    """the encoder's sd = softplus(W_sd h + b_sd) + sd_offset with the model's offset, not the example's 0.1"""
    c = dict(name="sd_offset", B=33, D=50, L=8, h_enc=(64,), h_dec=(64,), S=4, seed=120)
    X, enc, dec, eps, kept = case_inputs(c, sd_offset=sd_offset)
    loss, grads = run_cuda(cu, X, enc, dec, eps, sd_offset=sd_offset)
    check("sd_offset=%g" % sd_offset, loss, grads, *oracles(X, enc, dec, eps, sd_offset=sd_offset))


def test_vae_saturated_logits(cu):
    """decoder logits of magnitude 30..90 on a sizeable fraction of the elements: EpiBern's ex2 / rcp / lg2 at saturation"""
    import test_vae_coverage as M
    c = dict(name="saturated", B=40, D=300, L=2, h_enc=(64,), h_dec=(150,), S=4, seed=121)
    X, enc, dec, eps, kept = case_inputs(c, saturate=True)
    frac, top = M.saturated_fraction(X, enc, dec, eps)
    assert frac > 0.5 and 60 < top < 120, (frac, top)
    loss, grads = run_cuda(cu, X, enc, dec, eps)
    check("saturated logits (%.0f %% with |l| > 30)" % (100 * frac), loss, grads, *oracles(X, enc, dec, eps))


def pack(X, enc, dec, eps):
    d = {"X": X, "eps": eps}
    for side, net in (("enc", enc), ("dec", dec)):
        for k, v in net.items():
            if isinstance(v, list):
                for i, a in enumerate(v):
                    d["%s.%s.%d" % (side, k, i)] = a
            else:
                d["%s.%s" % (side, k)] = v
    return d


def unpack(z):
    nets = {"enc": {"W": [], "b": []}, "dec": {"W": [], "b": []}}
    for k in z.files:
        if k in ("X", "eps"):
            continue
        side, rest = k.split(".", 1)
        if rest[:2] in ("W.", "b."):
            nets[side][rest[0]].append((int(rest[2:]), z[k]))
        else:
            nets[side][rest] = z[k]
    for net in nets.values():
        for wb in ("W", "b"):
            net[wb] = [a for _, a in sorted(net[wb], key=lambda t: t[0])]
    return z["X"], nets["enc"], nets["dec"], z["eps"]


def child_main(inputs, out_dir):
    """evaluate each saved case once on cuda:0; write loss and gradients to OUT_DIR/<basename of the input>"""
    sys.path[:0] = [ROOT, HERE]
    from brancher_b200 import _cuda as cu
    cu.lib()
    for path in inputs:
        with np.load(path) as z:
            X, enc, dec, eps = unpack(z)
        loss, grads = run_cuda(cu, X, enc, dec, eps)
        np.savez(os.path.join(out_dir, os.path.basename(path)), loss=np.float64(loss), **grads)
    torch.cuda.synchronize()


@pytest.mark.parametrize("var,value", CHILD_SETTINGS)
def test_vae_function_static_selection(tmp_path, var, value):
    """BRN_VAE_EW16=0 (no 16-epilogue-warp tile), BRN_VAE_CW=4 (four converter warps) and BRN_VAE_WGRAD_TILE=0|1 (the
    128-wide weight-gradient tiles) are read once per process: a child process evaluates CHILD_CASES under each"""
    inputs = []
    for name in CHILD_CASES:
        X, enc, dec, eps = prepared(name)[:4]
        p = str(tmp_path / ("%s.npz" % name))
        np.savez(p, **pack(X, enc, dec, eps))
        inputs.append(p)
    out_dir = tmp_path / "out"
    out_dir.mkdir()
    env = dict(os.environ, **{var: value})
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__)] + inputs + ["--", str(out_dir)]
    res = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, "child (%s=%s) exited with %d:\n%s\n%s" % (var, value, res.returncode, res.stdout[-4000:],
                                                                         res.stderr[-4000:])
    for name in CHILD_CASES:
        o32, o64 = prepared(name)[5:]
        with np.load(str(out_dir / ("%s.npz" % name))) as z:
            grads = {k: z[k] for k in z.files if k != "loss"}
            loss = float(z["loss"])
        check("%s %s=%s" % (name, var, value), loss, grads, o32, o64)


def test_vae_zero_local_samples_leave_outputs_untouched(cu):
    """s_local = 0 (a rank without samples) adds nothing to the loss or to any gradient"""
    import test_vae_cuda as V
    X, enc, dec, eps = V.random_vae(122, 33, 50, 4, (64,), (64,), 1)
    net = V.make_net(cu, enc, dec)
    net.zero_grads()
    net.flat.copy_(torch.randn(net.flat.shape, generator=torch.Generator().manual_seed(0)).to(DEV))
    before = net.flat.clone()
    loss = torch.full((1,), 3.25, dtype=torch.float64, device=DEV)
    for eps_arg in (None, V.dev(np.zeros((0, 33, 4), "f4"))):
        cu.vae_elbo_fwd_bwd(V.dev(X), net, cu.sample_range(4, s0=4, s_local=0), eps=eps_arg, loss=loss)
        torch.cuda.synchronize()
        assert loss.item() == 3.25
        assert torch.equal(net.flat, before)


def _bad_nets():
    """(what, enc, dec) of models the library must refuse"""
    import test_vae_cuda as V
    out = []
    for L in (0, 17):
        _, enc, dec, _ = V.random_vae(123, 8, 10, 2, (6,), (6,), 1)
        rng = np.random.RandomState(L)
        enc["W_mean"], enc["W_sd"] = rng.randn(L, 6).astype("f4"), rng.randn(L, 6).astype("f4")
        enc["b_mean"], enc["b_sd"] = np.zeros(L, "f4"), np.zeros(L, "f4")
        dec["W"][0] = rng.randn(6, L).astype("f4")
        out.append(("L=%d" % L, enc, dec))
    _, enc, dec, _ = V.random_vae(124, 8, 10, 2, (6,), (1025, 6), 1)
    out.append(("h0=1025", enc, dec))
    _, enc, dec, _ = V.random_vae(125, 8, 10, 2, (6,), (12, 6), 1)
    dec["W"][1] = np.ones((6, 13), "f4")
    out.append(("decoder layer 1 is 13 -> 6 after a 12-wide layer", enc, dec))
    return out


@pytest.mark.parametrize("i", range(4))
def test_vae_rejects_invalid_models(cu, i):
    """each invalid model raises before anything runs: brn_vae_workspace_bytes returns 0, brn_vae_elbo_fwd_bwd refuses it, and
    neither the loss nor a gradient is written"""
    import ctypes
    import test_vae_cuda as V
    what, enc, dec = _bad_nets()[i]
    X = V.dev((np.random.RandomState(i).rand(8, 10) < 0.5).astype("f4"))
    net = V.make_net(cu, enc, dec)
    loss = torch.zeros(1, dtype=torch.float64, device=DEV)
    with pytest.raises(cu.BrancherCudaError):
        cu.vae_elbo_fwd_bwd(X, net, cu.sample_range(2), loss=loss)
    m = net.struct()
    assert cu.lib().brn_vae_workspace_bytes(ctypes.byref(m), 8, 2) == 0, what
    r = cu.sample_range(2)
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    status = cu.lib().brn_vae_elbo_fwd_bwd(X.data_ptr(), 8, 0, 8, ctypes.byref(m), None, 0, ctypes.byref(r), ws.data_ptr(),
                                           ws.numel(), 1, loss.data_ptr(), cu._stream(X.device))
    assert status != 0, what
    torch.cuda.synchronize()
    assert loss.item() == 0.0 and not net.flat.any().item(), what


def test_vae_rejects_seven_hidden_layers(cu):
    import test_vae_cuda as V
    _, enc, dec, _ = V.random_vae(126, 8, 10, 2, (6,) * 7, (6,), 1)
    with pytest.raises(cu.BrancherCudaError):
        V.make_net(cu, enc, dec)


if __name__ == "__main__":
    sep = sys.argv.index("--")
    child_main(sys.argv[1:sep], sys.argv[sep + 1])
