"""GPU: regression particles -- brn_linreg_particles_loss_grad (K4a) and brn_linreg_vectors_loglik_grad (K6b) for the Normal,
Cauchy and Laplace likelihoods over BF.matmul(weights, x) at a fixed noise scale -- against the fp64 oracle on both kernel paths,
the argument checks, the full C4 size, and SVGD / MAP / WVGD through the public API."""
import json

import numpy as np
import pytest
import torch

import model_zoo as zoo
import regparticles_models as rm
import regparticles_oracle as ro
from helpers import ATOL, assert_close, check_against_oracle
from test_robreg_cuda import check

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LIKS = list(rm.LIKELIHOODS)
CODE = {"normal": 2, "cauchy": 3, "laplace": 4}
SIGMA = 0.3


@pytest.fixture(scope="module")
def cu():
    from brancher_b200 import _cuda
    _cuda.lib()
    assert torch.cuda.is_available()
    return _cuda


@pytest.fixture
def ns():
    from brancher_b200 import config
    config.set_device(DEV)
    return zoo.namespace("brancher_b200")


def dev(a, dtype=torch.float32):
    return torch.tensor(np.asarray(a), dtype=dtype, device=DEV)


def sig():
    return dev(np.array([SIGMA], "f4"))


def problem(lik, N, F, n, seed=0, spread=0.3):
    X, y, wtrue, rng = rm.data(seed, N, F, likelihood=lik)
    theta = (wtrue[None, None, :] + spread * rng.randn(n, 1, F)).astype("f4")
    return X, y, theta


def oracles(lik, X, y, theta, prior):
    o32 = ro.particles_loss_grad(X, y, theta, SIGMA, lik, prior, dtype=torch.float32)
    o64 = ro.particles_loss_grad(X, y, theta, SIGMA, lik, prior, dtype=torch.float64)
    kb = ro.particles_loss_grad_streamed(X, y, theta, SIGMA, lik, prior, kink=True)[2] if lik == "laplace" else None
    return (o32[0], {"G": o32[1]}), (o64[0], {"G": o64[1]}), kb


def run_particles(cu, lik, X, y, theta, prior, prepared=None):
    n, _, F = theta.shape
    pr = (None, None) if prior is None else (dev(np.full(F, prior[0], "f4")), dev(np.full(F, prior[1], "f4")))
    loss, G = cu.linreg_particles_loss_grad(dev(X).reshape(len(X), F), dev(y), CODE[lik], dev(theta).reshape(n, F), sig(), *pr,
                                            prepared=prepared)
    return loss.item(), G.cpu().numpy().reshape(theta.shape)


# (N, F, n, variant): N not a multiple of 64, n in {1, 7, 300}, F = 5 on the SIMT kernel, the one-pass kernel where K2g takes it
CASES = [(1000, 5, 7, "simt"), (777, 16, 1, "simt"), (4097, 48, 300, "simt"), (4097, 48, 300, "tcgen05-flash"),
         (5000, 128, 64, "tcgen05-flash"), (4100, 16, 7, "simt")]


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("N,F,n,variant", CASES)
@pytest.mark.parametrize("prior", [None, rm.PRIOR])
def test_particles_vs_oracle(cu, monkeypatch, lik, N, F, n, variant, prior):
    if variant == "simt" and N >= 4096 and n >= 64:
        monkeypatch.setenv("BRN_LINEAR_VARIANT", "simt")
    X, y, theta = problem(lik, N, F, n, seed=N + F + n)
    loss, G = run_particles(cu, lik, X, y, theta, prior)
    assert cu.last_variant() == variant
    o32, o64, kb = oracles(lik, X, y, theta, prior)
    check(loss, {"G": G}, o32, o64, kb, "%s particles N=%d F=%d n=%d %s" % (lik, N, F, n, variant))


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("N,F,n,variant", [(1000, 5, 7, "simt"), (4097, 48, 300, "tcgen05-flash")])
def test_vectors_vs_oracle(cu, lik, N, F, n, variant):
    X, y, V = problem(lik, N, F, n, seed=7 + N)
    Xd = dev(X)
    ll, G = cu.linreg_vectors_loglik_grad(Xd, dev(y), CODE[lik], dev(V).reshape(n, F), sig())
    assert cu.last_variant() == variant
    ll2, G2 = cu.linreg_vectors_loglik_grad(Xd, dev(y), CODE[lik], dev(V).reshape(n, F), sig(), want_grad=False)
    assert G2 is None
    l64, g64 = ro.vectors_loglik_grad(X, y, V, SIGMA, lik, dtype=torch.float64)
    kb = ro.particles_loss_grad_streamed(X, y, V, SIGMA, lik, kink=True)[2] if lik == "laplace" else {"G": 0.0}
    for got in (ll, ll2):
        assert_close(got.cpu().numpy(), l64, "%s ll" % lik, scale=np.abs(l64).max())
    sc = np.abs(g64).max()
    err = np.abs(G.cpu().numpy().reshape(V.shape) - g64)
    assert (err <= 1e-6 * sc + 1e-5 * np.abs(g64) + kb["G"]).all(), err.max() / sc


@pytest.mark.parametrize("lik", LIKS)
def test_prepared_x_matches_plain(cu, lik):
    """a prepared X gives what the per-call split of X gives; the loss only up to the order of its fp64 atomic sums"""
    X, y, theta = problem(lik, 5000, 64, 128, seed=5)
    a = run_particles(cu, lik, X, y, theta, rm.PRIOR)
    assert cu.last_variant() == "tcgen05-flash"
    b = run_particles(cu, lik, X, y, theta, rm.PRIOR, prepared=cu.PreparedX())
    np.testing.assert_allclose(b[0], a[0], rtol=1e-12)
    np.testing.assert_allclose(b[1], a[1], rtol=1e-6, atol=1e-6 * np.abs(a[1]).max())


@pytest.mark.parametrize("lik", LIKS)
def test_no_particles_and_no_rows(cu, lik):
    F = 8
    X, y, theta = problem(lik, 50, F, 3)
    loss, G = cu.linreg_particles_loss_grad(dev(X), dev(y), CODE[lik], torch.zeros((0, F), device=DEV), sig())
    assert loss.item() == 0.0 and G.shape == (0, F)
    ll, _ = cu.linreg_vectors_loglik_grad(dev(X), dev(y), CODE[lik], torch.zeros((0, F), device=DEV), sig())
    assert ll.numel() == 0
    X0, y0 = np.zeros((0, F), "f4"), np.zeros(0, "f4")
    loss, G = run_particles(cu, lik, X0, y0, theta, rm.PRIOR)
    l64, g64 = ro.particles_loss_grad(X0, y0, theta, SIGMA, lik, rm.PRIOR, dtype=torch.float64)
    assert_close(loss, l64, "N=0 loss")
    assert_close(G, g64, "N=0 G", scale=np.abs(g64).max())
    ll, G = cu.linreg_vectors_loglik_grad(dev(X0), dev(y0), CODE[lik], dev(theta).reshape(3, F), sig())
    assert (ll.cpu().numpy() == 0).all() and (G.cpu().numpy() == 0).all()


def test_bad_arguments(cu):
    lib = cu.lib()
    N, F, n = 5000, 64, 128
    X, y, theta = problem("normal", N, F, n)
    Xd, yd, th, G = dev(X), dev(y), dev(theta).reshape(n, F), torch.empty((n, F), device=DEV)
    loss, ll, s = torch.zeros(1, dtype=torch.float64, device=DEV), torch.zeros(n, dtype=torch.float64, device=DEV), sig()
    nbytes = lib.brn_linreg_vectors_workspace_bytes(N, F, n)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    px = cu.PreparedX().get(Xd, cu.GAUSSIAN, 1)
    assert px is not None

    def particles(lik=2, X=Xd.data_ptr(), px=None, F=F, noise=s.data_ptr(), ws_bytes=nbytes):
        return lib.brn_linreg_particles_loss_grad(X, px, yd.data_ptr(), lik, N, F, th.data_ptr(), n, None, None, noise, G.data_ptr(),
                                                  loss.data_ptr(), ws.data_ptr(), ws_bytes, None)

    def vectors(lik=2, X=Xd.data_ptr(), px=None, F=F, noise=s.data_ptr(), ws_bytes=nbytes):
        return lib.brn_linreg_vectors_loglik_grad(X, px, yd.data_ptr(), lik, N, F, th.data_ptr(), n, noise, G.data_ptr(), ll.data_ptr(),
                                                  ws.data_ptr(), ws_bytes, None)

    for fn in (particles, vectors):
        assert fn() == 0 and fn(px=px.data_ptr()) == 0
        torch.cuda.synchronize()
        for kw, msg in ((dict(lik=0), b"unknown likelihood"), (dict(lik=1), b"unknown likelihood"), (dict(lik=5), b"unknown likelihood"),
                        (dict(noise=None), b"NULL pointer"), (dict(F=129), b"exceeds the supported maximum"),
                        (dict(px=px.data_ptr() + 16), b"256-byte aligned"), (dict(X=None), b"NULL data pointer"),
                        (dict(ws_bytes=nbytes - 1), b"workspace too small")):
            assert fn(**kw) < 0, kw
            assert msg in lib.brn_last_error(), (kw, lib.brn_last_error())
    with pytest.raises(cu.BrancherCudaError, match="unknown likelihood"):
        cu.linreg_particles_loss_grad(Xd, yd, cu.BERNOULLI, th, s)


@pytest.mark.parametrize("lik", LIKS)
def test_full_size(cu, lik):
    """the C4 shape: n = 4096 particles, N = 65536 rows, F = 128, prepared X, against the fp64 streamed oracle (Laplace with the
    kink bound); the literal-box counts go to the parity report"""
    import test_full_config_parity as T
    n, N, F = 4096, 65536, 128
    X, y, theta = problem(lik, N, F, n, seed=11)
    loss, G = run_particles(cu, lik, X, y, theta, rm.PRIOR, prepared=cu.PreparedX())
    assert cu.last_variant() == "tcgen05-flash"
    o64 = ro.particles_loss_grad_streamed(X, y, theta, SIGMA, lik, rm.PRIOR, kink=lik == "laplace")
    o32 = ro.particles_loss_grad_streamed(X, y, theta, SIGMA, lik, rm.PRIOR, dtype=torch.float32)
    kb = o64[2] if lik == "laplace" else None
    what = "%s particles n=4096 N=65536 F=128 sigma=0.3" % lik
    T.literal_report(what, {"G": G, "loss": np.array(loss)}, {"G": o64[1], "loss": np.array(o64[0])},
                     {"G": o32[1], "loss": np.array(o32[0])})
    if kb is not None:
        print(json.dumps({"config": what, "kink_count": kb["count"], "kink_bound_over_scale": float(kb["G"].max() / np.abs(o64[1]).max())}))
    check(loss, {"G": G}, (o32[0], {"G": o32[1]}), (o64[0], {"G": o64[1]}), kb, what)


# ---------------------------------------------------------------------------------------------------------------------------
# public API
# ---------------------------------------------------------------------------------------------------------------------------
def _roots(models, name="weights"):
    return [[v for v in m.flatten() if v.name == name][0] for m in models]


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("scale", ["number", "root"])
def test_svgd_api_matches_oracle(ns, cu, lik, scale):
    """SVGD compute_loss -> backward -> correct_gradient == the oracle's gradient, then oracle.svgd_direction"""
    from oracle import elbo_oracle as O
    X, y, theta = problem(lik, 300, 6, 9, seed=21)
    model = rm.joint(ns, X, y, lik, scale)
    parts = rm.particles(ns, theta)
    m = ns.inference.SteinVariationalGradientDescent()
    m.check_model_compatibility(model, parts, None)
    loss = m.compute_loss(model, parts, None, 1)
    loss.backward()
    l64, g64 = ro.particles_loss_grad(X, y, theta, SIGMA, lik, rm.PRIOR, dtype=torch.float64)
    assert_close(float(loss.detach()), l64, "svgd loss")
    raw = np.stack([r.value.grad.cpu().numpy().reshape(1, 6) for r in _roots(parts)])
    assert_close(raw, g64, "svgd raw gradient", scale=np.abs(g64).max())
    m.correct_gradient(model, parts, None, 1)
    want, _ = O.svgd_direction(theta.reshape(9, 6), g64.reshape(9, 6))
    got = np.stack([r.value.grad.cpu().numpy().reshape(-1) for r in _roots(parts)])
    assert_close(got, want, "svgd direction", scale=np.abs(want).max())


@pytest.mark.parametrize("lik", LIKS)
def test_svgd_perform_inference_lowers_loss(ns, lik):
    X, y, theta = problem(lik, 400, 8, 6, seed=22, spread=1.0)
    model = rm.joint(ns, X, y, lik)
    parts = rm.particles(ns, theta)
    ns.inference.perform_inference(model, inference_method=ns.inference.SteinVariationalGradientDescent(), number_iterations=30,
                                   number_samples=1, optimizer="SGD", lr=2e-6, posterior_model=parts)
    curve = model.diagnostics["loss curve"]
    assert np.isfinite(curve).all() and curve[-1] < curve[0]


@pytest.mark.parametrize("lik", LIKS)
def test_map_api_matches_oracle(ns, cu, lik):
    X, y, theta = problem(lik, 500, 7, 1, seed=23)
    model, point = rm.map_model(ns, X, y, lik, w0=theta[0])
    m = ns.inference.MAP()
    m.check_model_compatibility(model, point, None)
    loss = m.compute_loss(model, point, None, 1)
    loss.backward()
    l64, g64 = ro.particles_loss_grad(X, y, theta, SIGMA, lik, rm.PRIOR, dtype=torch.float64)
    assert_close(float(loss.detach()), l64, "MAP loss")
    assert_close(_roots([point])[0].value.grad.cpu().numpy().reshape(1, 1, 7), g64, "MAP gradient", scale=np.abs(g64).max())


@pytest.mark.parametrize("lik", LIKS)
def test_map_dense_equals_scalar_twin(ns, cu, lik):
    """MAP on the dense model (K4a) == MAP on the scalar-written twin (K1), loss and gradient, both on the GPU"""
    X, y, theta = problem(lik, 200, 3, 1, seed=24)
    model, point = rm.map_model(ns, X, y, lik, w0=theta[0])
    twin, tpoint = rm.scalar_twin(ns, X, y, lik, w0=theta[0])
    m = ns.inference.MAP()
    assert m._plan(model, point)[0] == "particles" and m._plan(twin, tpoint)[0] == "dag"
    loss = m.compute_loss(model, point, None, 1)
    loss.backward()
    tloss = m.compute_loss(twin, tpoint, None, 1)
    tloss.backward()
    assert_close(float(loss.detach()), float(tloss.detach()), "MAP dense vs K1 loss")
    g = _roots([point])[0].value.grad.cpu().numpy().reshape(-1)
    tg = np.array([_roots([tpoint], "w%d" % (i + 1))[0].value.grad.cpu().numpy().reshape(()) for i in range(3)])
    assert_close(g, tg, "MAP dense vs K1 gradient", scale=np.abs(tg).max())


def test_map_perform_inference_recovers_weights(ns):
    X, y, wtrue, _ = rm.data(25, 4000, 6, noise_sd=0.3)
    model, point = rm.map_model(ns, X, y, "normal")
    # SGD below 2 / lambda_max of the Hessian X^T X / sigma^2 (about 4.8e4 here): plain gradient descent converges geometrically
    ns.inference.perform_inference(model, inference_method=ns.inference.MAP(), number_iterations=200, number_samples=1,
                                   optimizer="SGD", lr=1e-5)
    w = _roots([point])[0].value.detach().cpu().numpy().reshape(-1)
    wls = np.linalg.lstsq(X.astype(np.float64), y.astype(np.float64), rcond=None)[0]      # the N(0, 2) prior moves it by ~1e-5
    assert np.abs(w - wls).max() < 1e-3, (w, wls)
    assert np.abs(w - wtrue).max() < 0.05, (w, wtrue)


def _wvgd(ns, lik, n=3, S=40, seed=26, spread=1.0):
    X, y, theta = problem(lik, 200, 4, n, seed=seed, spread=spread)
    rng = np.random.RandomState(seed)
    loc = (theta + 0.05 * rng.randn(*theta.shape)).astype("f4")
    model = rm.joint(ns, X, y, lik)
    parts, smps = rm.particles(ns, theta), rm.samplers(ns, loc)
    rho = np.stack([r.value.detach().cpu().numpy().reshape(()) for r in _roots(smps, "weights_scale")]).astype("f4")
    eps = {"elbo": rng.randn(n, S, 1, 4).astype("f4"), "particle": rng.randn(n, S, 1, 4).astype("f4"),
           "post": rng.randn(n, S, 1, 4).astype("f4")}
    return X, y, theta, loc, rho, eps, model, parts, smps


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("spread", [0.3, 1.0])
def test_wvgd_api_matches_oracle(ns, cu, lik, spread):
    """spread 0.3: particles near the data's weights, both gates of check_against_oracle.  spread 1.0: particles far from them,
    where the importance weights are a softmax over log-likelihoods hundreds apart and the particle gradient is ill-conditioned:
    rounding the draws to fp32 alone moves the exact Laplace theta gradient by about 1.3e-5 of its scale, more than gate A's
    1e-6 -- no evaluation on fp32 draws can meet gate A there, so gate A gets the fp32 evaluation's own distance from fp64, the
    allowance gate B already has"""
    from brancher_b200 import lowering
    n, S = 3, 40
    X, y, theta, loc, rho, eps, model, parts, smps = _wvgd(ns, lik, n, S, spread=spread)
    m = ns.inference.WassersteinVariationalGradientDescent(variational_samplers=smps, particles=parts, biased=False)
    m.check_model_compatibility(model, parts, m.sampler_model)
    with lowering.inject_noise({"elbo": eps["elbo"], "particle": eps["particle"]}):
        loss = m.compute_loss(model, parts, m.sampler_model, S)
    loss.backward()
    o = {dt: ro.wvgd_loss(ro.loglik(X, y, SIGMA, lik, dt), theta, loc, rho, eps["elbo"], eps["particle"], dtype=dt)
         for dt in (torch.float32, torch.float64)}
    assert (m.accepted.cpu().numpy() == o[torch.float64][2]).all()
    got = {"loc": np.stack([r.value.grad.cpu().numpy().reshape(1, 4) for r in _roots(smps, "weights_loc")]),
           "rho": np.stack([r.value.grad.cpu().numpy().reshape(()) for r in _roots(smps, "weights_scale")]),
           "theta": np.stack([r.value.grad.cpu().numpy().reshape(1, 4) for r in _roots(parts)])}
    (l32, g32), (l64, g64) = o[torch.float32][:2], o[torch.float64][:2]
    what = "%s wvgd spread=%g" % (lik, spread)
    if spread < 1.0:
        check_against_oracle(float(loss.detach()), got, (l32, g32), (l64, g64), what)
    else:
        assert_close(float(loss.detach()), l64, what + " loss vs fp64 oracle", atol=ATOL + 2 * abs(l32 - l64))
        for k in g64:
            sc = max(np.abs(g64[k]).max(), 1e-8)
            cond = 2 * np.abs(np.asarray(g32[k], np.float64) - g64[k]).max() / sc
            assert_close(got[k], g64[k], "%s grad %s vs fp64 oracle (+ fp32 conditioning)" % (what, k), atol=ATOL + cond, scale=sc)
    with lowering.inject_noise({"post": eps["post"]}):
        m.number_post_samples = S
        m.post_process(model)
    w64, lz64, n64 = ro.wvgd_ensemble_weights(ro.loglik(X, y, SIGMA, lik), theta, loc, rho, eps["post"])
    w32, lz32, _ = ro.wvgd_ensemble_weights(ro.loglik(X, y, SIGMA, lik, torch.float32), theta, loc, rho, eps["post"], dtype=torch.float32)
    assert (m.accepted_post == n64).all()
    assert_close(m.log_normalizers, lz64, "%s wvgd logZ" % lik, rtol=1e-5, atol=1e-5 + 2 * np.abs(lz32 - lz64).max())
    assert_close(m.weights, w64, "%s wvgd weights" % lik, rtol=1e-4, atol=1e-7 + 2 * np.abs(w32 - w64).max())
