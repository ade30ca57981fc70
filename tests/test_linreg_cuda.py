"""GPU: Bayesian linear regression (K2g, brn_linreg_elbo_fwd_bwd) against the oracle -- the one-pass tcgen05 kernel and the
SIMT kernel, both noise modes (a fixed scale, a LogNormal latent tied or declared), Philox noise, sample sharding, the prepared
X, the API path, the scalar-written K1 twin, the graph-captured loop and training."""
import os

import numpy as np
import pytest
import torch

import linreg_models as lm
import model_zoo as zoo
from helpers import check_against_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NOISES = [0.3, "tied", "declared"]


@pytest.fixture(scope="module")
def cu():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from brancher_b200 import _cuda
    _cuda.lib()
    return _cuda


@pytest.fixture(scope="module")
def ns():
    assert torch.cuda.is_available()
    from brancher_b200 import config
    config.set_device("cuda:0")
    return zoo.namespace("brancher_b200")


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.asarray(a), dtype=dtype).to(DEV).contiguous()


def problem(N, F, S, noise, seed=0):
    X, y, _, rng = lm.data(seed, N, F)
    params = {"weights": ((0.3 * rng.randn(1, F)).astype("f4"), (rng.randn(1, F) - 1.5).astype("f4")),
              "nu": (np.array(-1.0, "f4"), np.array(-0.5, "f4"))}
    eps = {"weights": rng.randn(S, 1, F).astype("f4"), "nu": rng.randn(S).astype("f4")}
    prior = {"weights": None, "nu": (-1.2, 0.7)} if noise == "declared" else None
    return X, y, params, eps, prior


def run(cu, X, y, params, noise, r, eps=None, prior=None, with_prior=True, prepared=None, Xd=None):
    F = X.shape[1]
    w = cu.MeanFieldVar(dev(params["weights"][0]), dev(params["weights"][1]), var_id=0,
                        eps=None if eps is None else dev(eps["weights"]).reshape(-1, F))
    nu = None
    if noise != 0.3 and not isinstance(noise, float):
        pl = None if prior is None else dev(np.array([prior["nu"][0]], "f4"))
        ps = None if prior is None else dev(np.array([prior["nu"][1]], "f4"))
        nu = cu.MeanFieldVar(dev(params["nu"][0]).reshape(1), dev(params["nu"][1]).reshape(1), var_id=1, prior_loc=pl, prior_scale=ps,
                             eps=None if eps is None else dev(eps["nu"]).reshape(-1, 1))
    Xd = dev(X) if Xd is None else Xd
    loss = cu.linreg_elbo_fwd_bwd(Xd, dev(y), w, r, nu=nu, noise_scale=None if nu is not None else dev(np.array([noise], "f4")),
                                  with_prior=with_prior, prepared=prepared)
    torch.cuda.synchronize()
    g = {"weights_loc": w.dmu.cpu().numpy().reshape(1, F), "weights_scale": w.drho.cpu().numpy().reshape(1, F)}
    if nu is not None:
        g["nu_loc"] = nu.dmu.cpu().numpy().reshape(()); g["nu_scale"] = nu.drho.cpu().numpy().reshape(())
    return loss.item(), g


def oracles(X, y, params, eps, prior, noise, with_prior=True):
    import linreg_oracle as LO
    kind = noise if isinstance(noise, float) else "lognormal"
    return (LO.linreg_elbo(X, y, params, eps, prior, kind, torch.float32, with_prior=with_prior),
            LO.linreg_elbo(X, y, params, eps, prior, kind, torch.float64, with_prior=with_prior))


# (N, F, S): every N, F and S of the sweep at least once; flash-eligible F (multiple of 16) with N >= 4096 and S >= 64
CASES = [(1, 16, 7, "simt"), (63, 3, 1, "simt"), (64, 17, 128, "simt"), (1000, 100, 300, "simt"), (4097, 16, 128, "tcgen05-flash"),
         (4097, 48, 300, "tcgen05-flash"), (20000, 128, 128, "tcgen05-flash"), (20000, 100, 128, "simt"), (4097, 3, 7, "simt"),
         (20000, 48, 7, "simt")]


@pytest.mark.parametrize("N,F,S,variant", CASES)
@pytest.mark.parametrize("noise", NOISES)
def test_kernel_vs_oracle_injected(cu, monkeypatch, N, F, S, variant, noise):
    X, y, params, eps, prior = problem(N, F, S, noise, seed=N + F + S)
    o32, o64 = oracles(X, y, params, eps, prior, noise)
    r = cu.sample_range(S)
    loss, g = run(cu, X, y, params, noise, r, eps, prior)
    assert cu.last_variant() == variant
    check_against_oracle(loss, g, o32, o64, "linreg N=%d F=%d S=%d %s %s" % (N, F, S, noise, variant))
    # each variant forced on the same inputs
    for forced, want in (("simt", "simt"), ("tcgen05", "tcgen05-flash" if F % 16 == 0 else "simt")):
        monkeypatch.setenv("BRN_LINEAR_VARIANT", forced)
        loss2, g2 = run(cu, X, y, params, noise, r, eps, prior)
        assert cu.last_variant() == want
        check_against_oracle(loss2, g2, o32, o64, "linreg forced %s N=%d F=%d S=%d %s" % (forced, N, F, S, noise))
    monkeypatch.delenv("BRN_LINEAR_VARIANT")


@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("N,F,S", [(5000, 64, 96), (300, 5, 9)])
def test_philox_noise(cu, noise, N, F, S):
    X, y, params, _, prior = problem(N, F, S, noise, seed=3)
    r = cu.sample_range(S, seed=11, offset=4)
    loss, g = run(cu, X, y, params, noise, r, None, prior)
    eps = {"weights": cu.philox_normal(F, 0, r, DEV).cpu().numpy().reshape(S, 1, F),
           "nu": cu.philox_normal(1, 1, r, DEV).cpu().numpy().reshape(S)}
    o32, o64 = oracles(X, y, params, eps, prior, noise)
    check_against_oracle(loss, g, o32, o64, "linreg philox %s" % noise)


@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("N,F,S", [(6000, 32, 256), (500, 7, 40)])
def test_shard_invariance(cu, noise, N, F, S):
    X, y, params, _, prior = problem(N, F, S, noise, seed=4)
    full = run(cu, X, y, params, noise, cu.sample_range(S, seed=2, offset=1), None, prior)
    parts = [run(cu, X, y, params, noise, cu.sample_range(S, s0=s0, s_local=sl, seed=2, offset=1), None, prior)
             for s0, sl in ((0, S // 4), (S // 4, S // 2), (S // 4 + S // 2, S - S // 4 - S // 2))]
    np.testing.assert_allclose(sum(p[0] for p in parts), full[0], rtol=2e-6)
    for k in full[1]:
        tot = sum(p[1][k] for p in parts)
        np.testing.assert_allclose(tot, full[1][k], rtol=1e-5, atol=1e-6 * max(np.abs(full[1][k]).max(), 1e-6), err_msg=k)


@pytest.mark.parametrize("noise", [0.3, "tied"])
def test_prepared_x(cu, noise):
    N, F, S = 8192, 64, 128
    X, y, params, eps, prior = problem(N, F, S, noise, seed=5)
    r = cu.sample_range(S)
    Xd = dev(X)
    plain = run(cu, X, y, params, noise, r, eps, prior, Xd=Xd)
    px = cu.PreparedX()
    prep = run(cu, X, y, params, noise, r, eps, prior, prepared=px, Xd=Xd)
    assert cu.last_variant() == "tcgen05-flash"
    # the same kernel on the same operands; only the order of the per-sample fp64 / noise-gradient atomics differs
    np.testing.assert_allclose(prep[0], plain[0], rtol=1e-12)
    for k in plain[1]:
        np.testing.assert_allclose(prep[1][k], plain[1][k], rtol=1e-6, err_msg=k)
    # X changes in place: the prepared form is rebuilt
    X2 = X * 1.5
    Xd.copy_(dev(X2))
    again = run(cu, X2, y, params, noise, r, eps, prior, prepared=px, Xd=Xd)
    o32, o64 = oracles(X2, y, params, eps, prior, noise)
    check_against_oracle(again[0], again[1], o32, o64, "linreg prepared X after a change")


@pytest.mark.parametrize("noise", NOISES)
def test_zero_rows_and_without_prior(cu, noise):
    F, S = 16, 70
    X, y, params, eps, prior = problem(0, F, S, noise)
    loss, g = run(cu, X, y, params, noise, cu.sample_range(S), eps, prior)
    o32, o64 = oracles(X, y, params, eps, prior, noise)
    check_against_oracle(loss, g, o32, o64, "linreg N=0")
    X, y, params, eps, prior = problem(5000, 32, 80, noise)
    loss, g = run(cu, X, y, params, noise, cu.sample_range(80), eps, prior, with_prior=False)
    o32, o64 = oracles(X, y, params, eps, prior, noise, with_prior=False)
    check_against_oracle(loss, g, o32, o64, "linreg with_prior=0")


def test_bad_arguments(cu):
    X, y, params, eps, prior = problem(10, 4, 2, 0.3)
    w = cu.MeanFieldVar(dev(params["weights"][0]), dev(params["weights"][1]), var_id=0)
    with pytest.raises(cu.BrancherCudaError, match="exactly one"):
        cu.linreg_elbo_fwd_bwd(dev(X), dev(y), w, cu.sample_range(2))
    lib = cu.lib()
    st = w.struct()
    import ctypes
    rc = lib.brn_linreg_elbo_fwd_bwd(None, None, None, 10, 4, ctypes.byref(st), None, None, ctypes.byref(cu.sample_range(2)), None, 0, 1,
                                     None, None)
    assert rc < 0 and lib.brn_last_error()


def literal_report(config, got, g64, g32):
    import test_full_config_parity as T
    return T.literal_report(config, got, g64, g32)


@pytest.mark.parametrize("noise", [0.3, "tied"])
def test_full_size(cu, noise):
    """N = 10^6, F = 128, S = 1024, y = X w* + 0.3 noise, against the fp64 streamed oracle"""
    import linreg_oracle as LO
    from oracle import elbo_oracle as O
    N, F, S = 1_000_000, 128, 1024
    g = torch.Generator().manual_seed(0)
    X = torch.randn(N, F, generator=g)
    wstar = torch.randn(F, generator=g) / F ** 0.5
    y = X @ wstar + 0.3 * torch.randn(N, generator=g)
    params = {"weights": (np.zeros((1, F), "f4"), O.softplus_inverse(np.full((1, F), 0.05)).astype("f4")),
              "nu": (np.array(np.log(0.3), "f4"), np.array(-2.0, "f4"))}
    r = cu.sample_range(S, seed=3, offset=5)
    eps = {"weights": cu.philox_normal(F, 0, r, DEV).cpu().numpy().reshape(S, 1, F),
           "nu": cu.philox_normal(1, 1, r, DEV).cpu().numpy().reshape(S)}
    kind = noise if isinstance(noise, float) else "lognormal"
    o64 = LO.linreg_elbo_streamed(X.numpy(), y.numpy(), params, eps, None, kind)
    o32 = LO.linreg_elbo_streamed(X.numpy(), y.numpy(), params, eps, None, kind, dtype=torch.float32)
    loss, grads = run(cu, X.numpy(), y.numpy(), params, noise, r, None, None, Xd=X.to(DEV))
    assert cu.last_variant() == "tcgen05-flash"
    literal_report("linreg N=1e6 F=128 S=1024 noise=%s" % noise, dict(grads, loss=np.array(loss)), dict(o64[1], loss=np.array(o64[0])),
                   dict(o32[1], loss=np.array(o32[0])))
    check_against_oracle(loss, grads, o32, o64, "linreg full size %s" % noise)


def api_loss_and_grads(ns, model, S, eps):
    from brancher_b200 import lowering
    with lowering.inject_noise(eps):
        loss = ns.inference.ReverseKL().compute_loss(model, model.posterior_model, None, S)
    loss.backward()
    grads = {v.name: v.link.parameter.grad.detach().cpu().numpy()[0, 0]
             for v in model.posterior_model.flatten() if getattr(v, "learnable", False) and hasattr(v.link, "parameter")}
    return float(loss.detach()), grads


def q_params(model, noise):
    val = {v.name: v.link.parameter.detach().cpu().numpy()[0, 0] for v in model.posterior_model.flatten()
           if getattr(v, "learnable", False) and hasattr(v.link, "parameter")}
    p = {"weights": (val["weights_loc"], val["weights_scale"])}
    if noise != 0.3:
        p["nu"] = (val["nu_loc"].reshape(()), val["nu_scale"].reshape(()))
    return p


@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("N,F,S", [(5000, 64, 128), (200, 6, 12)])
def test_api_compute_loss_matches_oracle(ns, noise, N, F, S):
    model, Q, d = lm.dense(ns, 7, N=N, F=F, noise=noise)
    rng = np.random.RandomState(1)
    eps = {"weights": rng.randn(S, 1, F).astype("f4"), "nu": rng.randn(S).astype("f4")}
    loss, grads = api_loss_and_grads(ns, model, S, eps if noise != 0.3 else {"weights": eps["weights"]})
    params = q_params(model, noise)
    o32, o64 = oracles(d["X"], d["y"], params, eps, d["prior"], noise)
    check_against_oracle(loss, grads, o32, o64, "linreg API %s" % noise)


@pytest.mark.parametrize("noise", NOISES)
def test_k1_twin_on_gpu(ns, noise):
    """the dense model (K2g) and its scalar-written twin (K1, the reference-pinned path) give the same loss and gradients"""
    N, S = 300, 16
    X, y, _, rng = lm.data(9, N, 3)
    mu0 = (0.3 * rng.randn(1, 3)).astype("float32")
    sg0 = (0.2 + 0.3 * rng.rand(1, 3)).astype("float32")
    dense, _, _ = lm.dense(ns, 9, N=N, F=3, noise=noise, mu0=mu0, sg0=sg0)
    twin, _ = lm.scalar_twin(ns, X, y, mu0, sg0, noise=noise)
    ew, enu = rng.randn(S, 1, 3).astype("f4"), rng.randn(S).astype("f4")
    ed = {"weights": ew, "nu": enu}
    et = {"w1": ew[:, 0, 0], "w2": ew[:, 0, 1], "w3": ew[:, 0, 2], "nu": enu}
    if noise == 0.3:
        ed.pop("nu"); et.pop("nu")
    ld, gd = api_loss_and_grads(ns, dense, S, ed)
    lt, gt = api_loss_and_grads(ns, twin, S, et)
    np.testing.assert_allclose(ld, lt, rtol=1e-5)
    for i in range(3):
        for part in ("loc", "scale"):
            a, b = gd["weights_" + part].reshape(-1)[i], gt["w%d_%s" % (i + 1, part)].reshape(())
            np.testing.assert_allclose(a, b, rtol=1e-4, atol=1e-5 * max(abs(b), 1.0))
    if noise != 0.3:
        for part in ("loc", "scale"):
            np.testing.assert_allclose(gd["nu_" + part].reshape(()), gt["nu_" + part].reshape(()), rtol=1e-4, atol=1e-5)


def learnable_values(model):
    return {v.name: v.link.parameter.detach().cpu().numpy().copy() for v in model.posterior_model.flatten()
            if getattr(v, "learnable", False) and hasattr(v.link, "parameter")}


@pytest.mark.parametrize("noise,N,F,S,opt,kw,iters", [
    (0.3, 300, 16, 32, "Adam", dict(lr=0.05), 30), ("tied", 300, 16, 32, "SGD", dict(lr=1e-4, momentum=0.9), 30),
    ("declared", 5000, 64, 128, "Adam", dict(lr=0.02), 20), ("tied", 5000, 64, 128, "Adam", dict(lr=0.02), 20)])
def test_graph_loop_equals_stepwise_loop(ns, noise, N, F, S, opt, kw, iters):
    from brancher_b200 import config, inference
    out = {}
    for mode in ("graph", "eager"):
        config.set_seed(123)
        model = lm.dense(ns, 3, N=N, F=F, noise=noise)[0]
        inference.fused_loop_enabled = mode == "graph"
        try:
            inference.perform_inference(model, number_iterations=iters, number_samples=S, optimizer=opt,
                                        inference_method=inference.ReverseKL(), **kw)
        finally:
            inference.fused_loop_enabled = True
        assert inference.last_loop == mode
        out[mode] = (np.asarray(model.diagnostics["loss curve"], dtype=np.float64).reshape(-1), learnable_values(model))
    cg, ce = out["graph"][0], out["eager"][0]
    assert cg.shape == ce.shape == (iters,) and np.isfinite(cg).all()
    np.testing.assert_allclose(cg, ce, rtol=2e-5, atol=1e-5 * np.abs(ce).max())
    for k, v in out["eager"][1].items():
        sc = max(np.abs(v).max(), 1e-6)
        np.testing.assert_allclose(out["graph"][1][k], v, rtol=1e-4, atol=1e-5 * sc, err_msg=k)


@pytest.mark.parametrize("noise", [0.3, "tied"])
def test_perform_inference_posterior_mean(ns, noise):
    """perform_inference reaches the fp64 oracle-trained posterior mean of w (and nu) within MC error"""
    from brancher_b200 import config
    import linreg_oracle as LO
    from oracle import elbo_oracle as O
    config.set_seed(123)
    N, F, S, iters, lr = 400, 4, 64, 400, 0.05
    mu0, sg0 = np.zeros((1, F), "f4"), np.full((1, F), 0.5, "f4")
    model, Q, d = lm.dense(ns, 11, N=N, F=F, noise=noise, mu0=mu0, sg0=sg0)
    ns.inference.perform_inference(model, number_iterations=iters, number_samples=S, optimizer="Adam", lr=lr)
    curve = model.diagnostics["loss curve"]
    assert np.isfinite(curve).all() and curve[-20:].mean() < curve[:20].mean()
    got = q_params(model, noise)
    p0 = {"weights": (mu0.astype("f8"), O.softplus_inverse(sg0)), "nu": (np.array(-1.0), O.softplus_inverse(0.5))}
    t = {k: [torch.tensor(np.asarray(a, "f8"), requires_grad=True) for a in p0[k]] for k in p0}
    opt = torch.optim.Adam([a for k in t for a in t[k]], lr=lr)
    rng = np.random.RandomState(0)
    kind = noise if noise == 0.3 else "lognormal"
    for _ in range(iters):
        eps = {"weights": rng.randn(S, 1, F), "nu": rng.randn(S)}
        _, gr = LO.linreg_elbo_streamed(d["X"], d["y"], {k: tuple(a.detach().numpy() for a in t[k]) for k in t}, eps, None, kind)
        opt.zero_grad()
        t["weights"][0].grad = torch.tensor(gr["weights_loc"]); t["weights"][1].grad = torch.tensor(gr["weights_scale"])
        if kind == "lognormal":
            t["nu"][0].grad = torch.tensor(gr["nu_loc"]); t["nu"][1].grad = torch.tensor(gr["nu_scale"])
        opt.step()
    sd = torch.nn.functional.softplus(t["weights"][1]).detach().numpy().reshape(-1)
    want = t["weights"][0].detach().numpy().reshape(-1)
    assert np.all(np.abs(got["weights"][0].reshape(-1) - want) < 4 * sd / np.sqrt(S) + 0.02), (got["weights"][0], want)
    if kind == "lognormal":
        sdn = float(torch.nn.functional.softplus(t["nu"][1].detach()))
        assert abs(float(got["nu"][0]) - float(t["nu"][0])) < 4 * sdn / np.sqrt(S) + 0.05, (got["nu"][0], float(t["nu"][0]))
