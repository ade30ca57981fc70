"""GPU: robust Bayesian linear regression (K2g with a Cauchy or Laplace likelihood, brn_linreg_elbo_fwd_bwd_lik) against the
oracle -- the one-pass tcgen05 kernel and the SIMT kernel, both noise modes (a fixed scale, a LogNormal latent tied or
declared), Philox noise, sample sharding, the prepared X, the API path, the scalar-written K1 twin, the graph-captured loop and
training on heavy-tailed data.

Laplace's gradient has a kink at r = 0: a residual closer to zero than the logits' error can take the opposite sign from the
fp64 oracle, and each such flip moves the weight gradient by 2 |x_b| / sigma_s / S.  Its checks add the streamed oracle's
rigorous bound of those contributions (robreg_oracle.KINK_REL) to the absolute term of both gates; the set is empty at the
small sizes, where the plain rule applies.  Cauchy is smooth and is held to the plain rule everywhere."""
import json

import numpy as np
import pytest
import torch

import model_zoo as zoo
import robreg_models as rm
from helpers import ATOL, RTOL, assert_close, check_against_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NOISES = [0.3, "tied", "declared"]
LIKS = list(rm.LIKELIHOODS)


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


def code(cu, lik):
    return cu.CAUCHY if lik == "cauchy" else cu.LAPLACE


def problem(N, F, S, noise, seed=0):
    X, y, _, rng = rm.data(seed, N, F)
    params = {"weights": ((0.3 * rng.randn(1, F)).astype("f4"), (rng.randn(1, F) - 1.5).astype("f4")),
              "nu": (np.array(-1.0, "f4"), np.array(-0.5, "f4"))}
    eps = {"weights": rng.randn(S, 1, F).astype("f4"), "nu": rng.randn(S).astype("f4")}
    prior = {"weights": None, "nu": (-1.2, 0.7)} if noise == "declared" else None
    return X, y, params, eps, prior


def run(cu, lik, X, y, params, noise, r, eps=None, prior=None, with_prior=True, prepared=None, Xd=None):
    F = X.shape[1]
    w = cu.MeanFieldVar(dev(params["weights"][0]), dev(params["weights"][1]), var_id=0,
                        eps=None if eps is None else dev(eps["weights"]).reshape(-1, F))
    nu = None
    if not isinstance(noise, float):
        pl = None if prior is None else dev(np.array([prior["nu"][0]], "f4"))
        ps = None if prior is None else dev(np.array([prior["nu"][1]], "f4"))
        nu = cu.MeanFieldVar(dev(params["nu"][0]).reshape(1), dev(params["nu"][1]).reshape(1), var_id=1, prior_loc=pl, prior_scale=ps,
                             eps=None if eps is None else dev(eps["nu"]).reshape(-1, 1))
    Xd = dev(X) if Xd is None else Xd
    loss = cu.linreg_elbo_fwd_bwd(Xd, dev(y), w, r, nu=nu, noise_scale=None if nu is not None else dev(np.array([noise], "f4")),
                                  with_prior=with_prior, prepared=prepared, likelihood=code(cu, lik))
    torch.cuda.synchronize()
    g = {"weights_loc": w.dmu.cpu().numpy().reshape(1, F), "weights_scale": w.drho.cpu().numpy().reshape(1, F)}
    if nu is not None:
        g["nu_loc"] = nu.dmu.cpu().numpy().reshape(()); g["nu_scale"] = nu.drho.cpu().numpy().reshape(())
    return loss.item(), g


def oracles(lik, X, y, params, eps, prior, noise, with_prior=True):
    """(o32, o64, kink bound or None): autograd oracles in fp32 / fp64 and, for Laplace, the streamed oracle's kink bound"""
    import robreg_oracle as RO
    kind = noise if isinstance(noise, float) else "lognormal"
    o32 = RO.robreg_elbo(X, y, params, eps, prior, kind, lik, torch.float32, with_prior=with_prior)
    o64 = RO.robreg_elbo(X, y, params, eps, prior, kind, lik, torch.float64, with_prior=with_prior)
    kb = None
    if lik == "laplace":
        kb = RO.robreg_elbo_streamed(X, y, params, eps, prior, kind, lik, with_prior=with_prior, kink=True)[2]
    return o32, o64, kb


def check(loss, grads, o32, o64, kb, what):
    """check_against_oracle's two gates, with the Laplace kink bound (per element) added to the absolute term"""
    if kb is None or kb["count"] == 0:
        check_against_oracle(loss, grads, o32, o64, what)
        return
    print("%s: %d residuals within the kink margin" % (what, kb["count"]))
    (l32, g32), (l64, g64) = o32, o64
    assert_close(loss, l64, what + " loss vs fp64 oracle")
    assert_close(loss, l32, what + " loss vs fp32 oracle", atol=ATOL + 2 * abs(l32 - l64))
    for k in g64:
        a = np.asarray(grads[k], dtype=np.float64).reshape(g64[k].shape)
        w64, w32 = np.asarray(g64[k], np.float64), np.asarray(g32[k], np.float64).reshape(g64[k].shape)
        sc = max(np.abs(w64).max(), np.abs(w32).max(), 1e-8)
        extra = np.asarray(kb.get(k, 0.0), np.float64)
        noise = np.abs(w32 - w64).max()
        for ref, floor, name in ((w64, 0.0, "fp64"), (w32, 2 * noise, "fp32")):
            err = np.abs(a - ref)
            bound = ATOL * sc + floor + extra + RTOL * np.abs(ref)
            assert (err <= bound).all(), "%s grad %s vs %s oracle (+ kink bound): max err %.3e, %d outside" % (
                what, k, name, err.max(), int((err > bound).sum()))


# (N, F, S): every N, F and S of the sweep at least once; flash-eligible F (multiple of 16) with N >= 4096 and S >= 64
CASES = [(1, 16, 7, "simt"), (63, 3, 1, "simt"), (64, 17, 128, "simt"), (1000, 100, 300, "simt"), (4097, 16, 128, "tcgen05-flash"),
         (4097, 48, 300, "tcgen05-flash"), (20000, 128, 128, "tcgen05-flash"), (20000, 100, 128, "simt"), (4097, 3, 7, "simt"),
         (20000, 48, 7, "simt")]


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("N,F,S,variant", CASES)
@pytest.mark.parametrize("noise", NOISES)
def test_kernel_vs_oracle_injected(cu, monkeypatch, lik, N, F, S, variant, noise):
    X, y, params, eps, prior = problem(N, F, S, noise, seed=N + F + S)
    o32, o64, kb = oracles(lik, X, y, params, eps, prior, noise)
    r = cu.sample_range(S)
    loss, g = run(cu, lik, X, y, params, noise, r, eps, prior)
    assert cu.last_variant() == variant
    what = "%s N=%d F=%d S=%d %s" % (lik, N, F, S, noise)
    check(loss, g, o32, o64, kb, what + " " + variant)
    # each variant forced on the same inputs
    for forced, want in (("simt", "simt"), ("tcgen05", "tcgen05-flash" if F % 16 == 0 else "simt")):
        monkeypatch.setenv("BRN_LINEAR_VARIANT", forced)
        loss2, g2 = run(cu, lik, X, y, params, noise, r, eps, prior)
        assert cu.last_variant() == want
        check(loss2, g2, o32, o64, kb, what + " forced " + forced)
    monkeypatch.delenv("BRN_LINEAR_VARIANT")


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("N,F,S", [(5000, 64, 96), (300, 5, 9)])
def test_philox_noise(cu, lik, noise, N, F, S):
    X, y, params, _, prior = problem(N, F, S, noise, seed=3)
    r = cu.sample_range(S, seed=11, offset=4)
    loss, g = run(cu, lik, X, y, params, noise, r, None, prior)
    eps = {"weights": cu.philox_normal(F, 0, r, DEV).cpu().numpy().reshape(S, 1, F),
           "nu": cu.philox_normal(1, 1, r, DEV).cpu().numpy().reshape(S)}
    check(loss, g, *oracles(lik, X, y, params, eps, prior, noise), "%s philox %s" % (lik, noise))


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("N,F,S", [(6000, 32, 256), (500, 7, 40)])
def test_shard_invariance(cu, lik, noise, N, F, S):
    X, y, params, _, prior = problem(N, F, S, noise, seed=4)
    full = run(cu, lik, X, y, params, noise, cu.sample_range(S, seed=2, offset=1), None, prior)
    parts = [run(cu, lik, X, y, params, noise, cu.sample_range(S, s0=s0, s_local=sl, seed=2, offset=1), None, prior)
             for s0, sl in ((0, S // 4), (S // 4, S // 2), (S // 4 + S // 2, S - S // 4 - S // 2))]
    np.testing.assert_allclose(sum(p[0] for p in parts), full[0], rtol=2e-6)
    for k in full[1]:
        tot = sum(p[1][k] for p in parts)
        np.testing.assert_allclose(tot, full[1][k], rtol=1e-5, atol=1e-6 * max(np.abs(full[1][k]).max(), 1e-6), err_msg=k)


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", [0.3, "tied"])
def test_prepared_x(cu, lik, noise):
    N, F, S = 8192, 64, 128
    X, y, params, eps, prior = problem(N, F, S, noise, seed=5)
    r = cu.sample_range(S)
    Xd = dev(X)
    plain = run(cu, lik, X, y, params, noise, r, eps, prior, Xd=Xd)
    px = cu.PreparedX()
    prep = run(cu, lik, X, y, params, noise, r, eps, prior, prepared=px, Xd=Xd)
    assert cu.last_variant() == "tcgen05-flash"
    # the same kernel on the same operands; only the order of the per-sample fp64 / noise-gradient atomics differs
    np.testing.assert_allclose(prep[0], plain[0], rtol=1e-12)
    for k in plain[1]:
        np.testing.assert_allclose(prep[1][k], plain[1][k], rtol=1e-6, err_msg=k)
    # X changes in place: the prepared form is rebuilt
    X2 = X * 1.5
    Xd.copy_(dev(X2))
    again = run(cu, lik, X2, y, params, noise, r, eps, prior, prepared=px, Xd=Xd)
    check(again[0], again[1], *oracles(lik, X2, y, params, eps, prior, noise), "%s prepared X after a change" % lik)


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", NOISES)
def test_zero_rows_and_without_prior(cu, lik, noise):
    F, S = 16, 70
    X, y, params, eps, prior = problem(0, F, S, noise)
    loss, g = run(cu, lik, X, y, params, noise, cu.sample_range(S), eps, prior)
    check(loss, g, *oracles(lik, X, y, params, eps, prior, noise), "%s N=0" % lik)
    X, y, params, eps, prior = problem(5000, 32, 80, noise)
    loss, g = run(cu, lik, X, y, params, noise, cu.sample_range(80), eps, prior, with_prior=False)
    check(loss, g, *oracles(lik, X, y, params, eps, prior, noise, with_prior=False), "%s with_prior=0" % lik)


def test_bad_arguments(cu):
    import ctypes
    X, y, params, eps, prior = problem(10, 4, 2, 0.3)
    w = cu.MeanFieldVar(dev(params["weights"][0]), dev(params["weights"][1]), var_id=0)
    with pytest.raises(cu.BrancherCudaError, match="unknown likelihood"):
        cu.linreg_elbo_fwd_bwd(dev(X), dev(y), w, cu.sample_range(2), noise_scale=dev(np.array([0.3], "f4")), likelihood=cu.BERNOULLI)
    with pytest.raises(cu.BrancherCudaError, match="exactly one"):
        cu.linreg_elbo_fwd_bwd(dev(X), dev(y), w, cu.sample_range(2), likelihood=cu.CAUCHY)
    lib = cu.lib()
    st = w.struct()
    args = (None, None, None, 10, 4, ctypes.byref(st), None, dev(np.array([0.3], "f4")).data_ptr(), ctypes.byref(cu.sample_range(2)),
            None, 0, 1, None, None)
    rc = lib.brn_linreg_elbo_fwd_bwd_lik(*(args[:3] + (cu.CAUCHY,) + args[3:]))
    assert rc < 0 and lib.brn_last_error()
    rc = lib.brn_linreg_elbo_fwd_bwd_lik(*(args[:3] + (7,) + args[3:]))
    assert rc < 0 and b"unknown likelihood" in lib.brn_last_error()


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", [0.3, "tied"])
def test_full_size(cu, lik, noise):
    """N = 10^6, F = 128, S = 1024, y = X w* + 0.3 standard-Cauchy noise (|z| beyond 10^4 occurs: the exponent-split log is
    exercised), against the fp64 streamed oracle; Laplace with the kink bound"""
    import robreg_oracle as RO
    import test_full_config_parity as T
    from oracle import elbo_oracle as O
    N, F, S = 1_000_000, 128, 1024
    g = torch.Generator().manual_seed(0)
    X = torch.randn(N, F, generator=g)
    wstar = torch.randn(F, generator=g) / F ** 0.5
    y = X @ wstar + 0.3 * torch.tan(np.pi * (torch.rand(N, generator=g, dtype=torch.float64) - 0.5)).float()     # standard Cauchy
    params = {"weights": (np.zeros((1, F), "f4"), O.softplus_inverse(np.full((1, F), 0.05)).astype("f4")),
              "nu": (np.array(np.log(0.3), "f4"), np.array(-2.0, "f4"))}
    r = cu.sample_range(S, seed=3, offset=5)
    eps = {"weights": cu.philox_normal(F, 0, r, DEV).cpu().numpy().reshape(S, 1, F),
           "nu": cu.philox_normal(1, 1, r, DEV).cpu().numpy().reshape(S)}
    kind = noise if isinstance(noise, float) else "lognormal"
    o64 = RO.robreg_elbo_streamed(X.numpy(), y.numpy(), params, eps, None, kind, lik, kink=lik == "laplace")
    o32 = RO.robreg_elbo_streamed(X.numpy(), y.numpy(), params, eps, None, kind, lik, dtype=torch.float32)
    kb = o64[2] if lik == "laplace" else None
    zmax = float(((y - X @ wstar).abs() / 0.3).max())
    assert zmax > 1e4, zmax
    loss, grads = run(cu, lik, X.numpy(), y.numpy(), params, noise, r, None, None, Xd=X.to(DEV))
    assert cu.last_variant() == "tcgen05-flash"
    what = "%s N=1e6 F=128 S=1024 noise=%s" % (lik, noise)
    T.literal_report(what, dict(grads, loss=np.array(loss)), dict(o64[1], loss=np.array(o64[0])), dict(o32[1], loss=np.array(o32[0])))
    if kb is not None:
        print(json.dumps({"config": what, "kink_count": kb["count"],
                          "kink_bound_over_scale": {k: float(kb[k].max() / np.abs(o64[1][k]).max()) for k in ("weights_loc", "weights_scale")}}))
    check(loss, grads, o32[:2], o64[:2], kb, what)


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


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", NOISES)
@pytest.mark.parametrize("N,F,S", [(5000, 64, 128), (200, 6, 12)])
def test_api_compute_loss_matches_oracle(ns, lik, noise, N, F, S):
    from brancher_b200 import _cuda as cu, lowering
    model, Q, d = rm.dense(ns, 7, N=N, F=F, likelihood=lik, noise=noise)
    assert lowering.get_plan(model, model.posterior_model).likelihood == code(cu, lik)
    rng = np.random.RandomState(1)
    eps = {"weights": rng.randn(S, 1, F).astype("f4"), "nu": rng.randn(S).astype("f4")}
    loss, grads = api_loss_and_grads(ns, model, S, eps if noise != 0.3 else {"weights": eps["weights"]})
    params = q_params(model, noise)
    check(loss, grads, *oracles(lik, d["X"], d["y"], params, eps, d["prior"], noise), "%s API %s" % (lik, noise))


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", NOISES)
def test_k1_twin_on_gpu(ns, lik, noise):
    """the dense model (K2g) and its scalar-written twin (K1, the reference-pinned path) give the same loss and gradients"""
    N, S = 300, 16
    X, y, _, rng = rm.data(9, N, 3)
    mu0 = (0.3 * rng.randn(1, 3)).astype("float32")
    sg0 = (0.2 + 0.3 * rng.rand(1, 3)).astype("float32")
    dense, _, _ = rm.dense(ns, 9, N=N, F=3, likelihood=lik, noise=noise, mu0=mu0, sg0=sg0)
    twin, _ = rm.scalar_twin(ns, X, y, mu0, sg0, likelihood=lik, noise=noise)
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


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise,N,F,S,opt,kw,iters", [
    (0.3, 300, 16, 32, "Adam", dict(lr=0.05), 30), ("tied", 300, 16, 32, "SGD", dict(lr=1e-4, momentum=0.9), 30),
    ("declared", 5000, 64, 128, "Adam", dict(lr=0.02), 20), ("tied", 5000, 64, 128, "Adam", dict(lr=0.02), 20)])
def test_graph_loop_equals_stepwise_loop(ns, lik, noise, N, F, S, opt, kw, iters):
    from brancher_b200 import inference
    out = {}
    for mode in ("graph", "eager"):
        from brancher_b200 import config
        config.set_seed(123)
        model = rm.dense(ns, 3, N=N, F=F, likelihood=lik, noise=noise)[0]
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


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", [0.3, "tied"])
def test_perform_inference_recovers_weights(ns, lik, noise):
    """on heavy-tailed data (y = X w* + 0.3 standard-Cauchy noise) perform_inference with the robust likelihood recovers w*
    (the least-squares estimate of the same data does not: it is checked to be further off)"""
    from brancher_b200 import config
    config.set_seed(123)
    N, F, S, iters = 2000, 4, 64, 400
    mu0, sg0 = np.zeros((1, F), "f4"), np.full((1, F), 0.5, "f4")
    model, Q, d = rm.dense(ns, 11, N=N, F=F, likelihood=lik, noise=noise, mu0=mu0, sg0=sg0)
    ns.inference.perform_inference(model, number_iterations=iters, number_samples=S, optimizer="Adam", lr=0.05)
    curve = np.asarray(model.diagnostics["loss curve"], dtype=np.float64)
    assert np.isfinite(curve).all() and curve[-20:].mean() < curve[:20].mean()
    got = q_params(model, noise)["weights"][0].reshape(-1)
    err = np.abs(got - d["wtrue"]).max()
    ls = np.linalg.lstsq(d["X"].astype("f8"), d["y"].astype("f8"), rcond=None)[0]
    assert err < 0.05, (got, d["wtrue"])
    assert err < np.abs(ls - d["wtrue"]).max(), (err, ls, d["wtrue"])
