"""CPU: lowering of regression particle ensembles (SVGD, MAP, WVGD over Normal / Cauchy / Laplace(BF.matmul(weights, x), constant
scale)) to the particle family, its rejections, and the regression-particle oracle against itself and against oracle.elbo_oracle."""
import numpy as np
import pytest
import torch

import model_zoo as zoo
import regparticles_models as rm
import regparticles_oracle as ro

CODES = {"normal": 2, "cauchy": 3, "laplace": 4}       # cu.GAUSSIAN / CAUCHY / LAPLACE
NAMES = {"normal": "Normal", "cauchy": "Cauchy", "laplace": "Laplace"}


@pytest.fixture(scope="module")
def ns():
    from brancher_b200 import config
    config.set_device("cpu")
    yield zoo.namespace("brancher_b200")
    config.set_device("cuda:0" if torch.cuda.is_available() else "cpu")


def _check_plan(plan, likelihood, F):
    assert plan.family == "particles (K4, %s likelihood)" % NAMES[likelihood]
    assert plan.likelihood == CODES[likelihood] and plan.C == 1 and plan.shape == (1, F)
    np.testing.assert_allclose(plan.noise_scale().item(), 0.3, rtol=1e-6)
    np.testing.assert_allclose(plan.prior_loc.numpy(), np.full(F, rm.PRIOR[0]), rtol=1e-6)
    np.testing.assert_allclose(plan.prior_scale.numpy(), np.full(F, rm.PRIOR[1]), rtol=1e-6)


@pytest.mark.parametrize("likelihood", rm.LIKELIHOODS)
@pytest.mark.parametrize("scale", ["number", "root"])
def test_svgd_map_wvgd_lower(ns, likelihood, scale):
    from brancher_b200 import lowering
    X, y, _, rng = rm.data(1, 30, 5, likelihood=likelihood)
    theta = rng.randn(4, 1, 5)
    model = rm.joint(ns, X, y, likelihood, scale)
    parts = rm.particles(ns, theta)
    plan = lowering.get_particle_plan(model, parts)
    _check_plan(plan, likelihood, 5)
    assert len(plan.parameters()) == 4
    np.testing.assert_allclose(plan.stacked().numpy(), theta.reshape(4, 5), rtol=1e-6)
    wplan = lowering.get_wvgd_plan(model, parts, rm.samplers(ns, theta))
    assert wplan.pplan is plan and wplan.tied
    m = ns.inference.SteinVariationalGradientDescent()
    m.check_model_compatibility(model, parts, None)
    mmodel, point = rm.map_model(ns, X, y, likelihood, scale)
    kind, mplan = ns.inference.MAP()._plan(mmodel, point)
    assert kind == "particles"
    _check_plan(mplan, likelihood, 5)


def test_logistic_family_string_unchanged(ns):
    from brancher_b200 import lowering
    model, parts, _ = zoo.svgd_softmax(ns, 0, B=20, F=4, C=3, n=3)
    assert lowering.get_particle_plan(model, parts).family == "particles (K4)"


@pytest.mark.parametrize("likelihood", rm.LIKELIHOODS)
def test_scalar_twin_map_keeps_k1(ns, likelihood):
    X, y, _, _ = rm.data(2, 20, 3, likelihood=likelihood)
    model, point = rm.scalar_twin(ns, X, y, likelihood)
    kind, plan = ns.inference.MAP()._plan(model, point)
    assert kind == "dag" and plan.family.startswith("dag")


def _reject(ns, model, parts, match):
    from brancher_b200 import lowering
    with pytest.raises(lowering.UnsupportedModelError, match=match):
        lowering.lower_particles(model, parts)


def _build(ns, loc_fn, scale_fn, likelihood="normal", C=1, extra=(), prior=None, N=10, F=4):
    X = np.random.RandomState(0).randn(N, F, 1)
    x = ns.RootVariable(X, "x", is_observed=True)
    w = prior(C, F) if prior is not None else ns.NormalVariable(np.zeros((C, F)), np.ones((C, F)), "weights")
    yv = rm.variable(ns, likelihood)(loc_fn(w, x), scale_fn(), "y")
    model = ns.ProbabilisticModel([yv] + [f() for f in extra])
    yv.observe(np.zeros((N, C, 1)))
    return model, rm.particles(ns, np.zeros((2, C, F)))


@pytest.mark.parametrize("likelihood", rm.LIKELIHOODS)
def test_rejects_lognormal_noise_latent(ns, likelihood):
    model, parts = _build(ns, ns.BF.matmul, lambda: ns.LogNormalVariable(-1., 0.5, "nu"), likelihood)
    _reject(ns, model, parts, "lognormal-distributed noise latent is not lowered -- a particle holds one root")


def test_rejects_learnable_scale(ns):
    model, parts = _build(ns, ns.BF.matmul, lambda: ns.RootVariable(0.3, "sig", learnable=True))
    _reject(ns, model, parts, "learnable point-estimate noise scale")


def test_rejects_deterministic_scale(ns):
    model, parts = _build(ns, ns.BF.matmul, lambda: ns.BF.exp(ns.RootVariable(np.zeros(1), "z", is_observed=True)))
    _reject(ns, model, parts, "noise scale must be a constant")


def test_rejects_bias(ns):
    model, parts = _build(ns, lambda w, x: ns.BF.matmul(w, x) + ns.NormalVariable(0., 1., "b"), lambda: 0.3, "cauchy")
    _reject(ns, model, parts, "bias added to BF.matmul")


def test_rejects_multi_output(ns):
    model, parts = _build(ns, ns.BF.matmul, lambda: 0.3, "laplace", C=2)
    _reject(ns, model, parts, "multi-output")


def test_rejects_non_normal_prior(ns):
    model, parts = _build(ns, ns.BF.matmul, lambda: 0.3, prior=lambda C, F: ns.LaplaceVariable(np.zeros((C, F)), np.ones((C, F)),
                                                                                               "weights"))
    _reject(ns, model, parts, "only a Normal prior on the weights")


def test_rejects_extra_latents(ns):
    model, parts = _build(ns, ns.BF.matmul, lambda: 0.3, extra=(lambda: ns.NormalVariable(0., 1., "extra"),))
    _reject(ns, model, parts, "other than the weights")


def test_map_names_both_reasons(ns):
    model, _ = _build(ns, ns.BF.matmul, lambda: ns.RootVariable(0.3, "sig", learnable=True))
    point = ns.ProbabilisticModel([ns.RootVariable(np.zeros((1, 4)), name="weights", learnable=True)])
    model.set_posterior_model(point)
    from brancher_b200 import lowering
    with pytest.raises(lowering.UnsupportedModelError, match="learnable point-estimate noise scale.*nor as a scalar DAG"):
        ns.inference.MAP().check_model_compatibility(model, point, None)


def test_particle_loss_on_cpu_raises(ns):
    from brancher_b200 import lowering
    X, y, _, rng = rm.data(3, 10, 4)
    model = rm.joint(ns, X, y)
    plan = lowering.get_particle_plan(model, rm.particles(ns, rng.randn(2, 1, 4)))
    model.update_observed_submodel()
    empirical = model.observed_submodel._get_sample(1, observed=True, differentiable=False)
    with pytest.raises(RuntimeError, match="only on CUDA devices"):
        plan.loss(empirical)


@pytest.mark.parametrize("likelihood", rm.LIKELIHOODS)
@pytest.mark.parametrize("prior", [None, rm.PRIOR])
def test_streamed_oracle_matches_autograd_oracle(likelihood, prior):
    X, y, _, rng = rm.data(4, 300, 6, likelihood=likelihood)
    theta = rng.randn(5, 1, 6)
    l64, g64 = ro.particles_loss_grad(X, y, theta, 0.3, likelihood, prior, dtype=torch.float64)
    ls, gs = ro.particles_loss_grad_streamed(X, y, theta, 0.3, likelihood, prior, row_chunk=64)
    np.testing.assert_allclose(ls, l64, rtol=1e-12)
    np.testing.assert_allclose(gs, g64, rtol=1e-10, atol=1e-10 * np.abs(g64).max())
    ll, G = ro.vectors_loglik_grad(X, y, theta, 0.3, likelihood, dtype=torch.float64)
    want = l64 if prior is None else None
    if want is not None:
        np.testing.assert_allclose(-ll.sum(), want, rtol=1e-12)
        np.testing.assert_allclose(G, g64, rtol=1e-10, atol=1e-10 * np.abs(g64).max())


def test_laplace_kink_bound_counts_exact_zeros():
    X = np.eye(4, dtype="float32")
    theta = np.array([[[1.0, 2.0, 0.0, 0.0]]])
    y = np.array([1.0, 2.0, 0.5, -0.5], "float32")            # rows 0 and 1 sit exactly on the kink
    _, _, kb = ro.particles_loss_grad_streamed(X, y, theta, 0.5, "laplace", kink=True)
    assert kb["count"] == 2
    np.testing.assert_allclose(kb["G"].reshape(-1), [4.0, 4.0, 0.0, 0.0])


@pytest.mark.parametrize("tag", ["wvgd_softmax", "wvgd_softmax4"])
def test_wvgd_restatement_matches_oracle_package(tag):
    """with the logistic log-likelihood, the closure-taking WVGD restatements equal oracle.elbo_oracle's on its golden inputs"""
    import os
    import torch.distributions as D
    from helpers import GOLDEN
    from oracle import elbo_oracle as O
    g = np.load(os.path.join(GOLDEN, tag + ".npz"))
    Xt, yt = torch.as_tensor(g["X"], dtype=torch.float64), torch.as_tensor(g["y"], dtype=torch.long)
    ll_fn = lambda z: D.Categorical(logits=torch.einsum("scf,bf->sbc", z, Xt)).log_prob(yt[None, :]).sum(1)
    args = (g["theta"], g["loc"], g["rho"], g["eps_elbo"], g["eps_particle"])
    l0, g0, c0 = O.wvgd_loss(g["X"], g["y"], *args, dtype=torch.float64)
    l1, g1, c1 = ro.wvgd_loss(ll_fn, *args, dtype=torch.float64)
    assert l0 == l1 and (c0 == c1).all()
    for key in g0:
        np.testing.assert_array_equal(g0[key], g1[key])
    w0, z0, n0 = O.wvgd_ensemble_weights(g["X"], g["y"], g["theta"], g["loc"], g["rho"], g["eps_elbo"])
    w1, z1, n1 = ro.wvgd_ensemble_weights(ll_fn, g["theta"], g["loc"], g["rho"], g["eps_elbo"])
    np.testing.assert_array_equal(z0, z1)
    np.testing.assert_array_equal(w0, w1)
    assert (n0 == n1).all()
