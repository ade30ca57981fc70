"""CPU: lowering of robust Bayesian linear regression (Cauchy / Laplace likelihood over BF.matmul(weights, x)) to the K2g family,
its rejections, and the dense oracle against the streamed oracle and against the scalar-DAG semantics of the same model."""
import numpy as np
import pytest
import torch

import model_zoo as zoo
import robreg_models as rm

LIKS = list(rm.LIKELIHOODS)


@pytest.fixture(scope="module")
def ns():
    from brancher_b200 import config
    config.set_device("cpu")
    yield zoo.namespace("brancher_b200")
    config.set_device("cuda:0" if torch.cuda.is_available() else "cpu")


def _plan(model):
    from brancher_b200 import lowering
    return lowering.get_plan(model, model.posterior_model)


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", [0.3, "tied", "declared"])
def test_robreg_lowers(ns, lik, noise):
    from brancher_b200 import _cuda as cu, lowering
    model, Q, d = rm.dense(ns, 1, N=30, F=5, likelihood=lik, noise=noise)
    plan = _plan(model)
    assert isinstance(plan, lowering.LinregPlan)
    assert plan.likelihood == (cu.CAUCHY if lik == "cauchy" else cu.LAPLACE)
    assert plan.family == "linear regression (K2g, %s likelihood)" % lik.capitalize()
    assert [s.name for s in plan.latents] == (["weights"] if noise == 0.3 else ["weights", "nu"])
    assert plan.latents[0].shape == (1, 5) and plan.latents[0].tied
    if noise == 0.3:
        np.testing.assert_allclose(plan.noise_scale().item(), 0.3, rtol=1e-6)
    else:
        nu = plan.latents[1]
        assert nu.tied == (noise == "tied") and int(np.prod(nu.shape)) == 1
        if noise == "declared":
            np.testing.assert_allclose(nu.prior_loc.item(), -1.2, rtol=1e-6)
            np.testing.assert_allclose(nu.prior_scale.item(), 0.7, rtol=1e-6)


def test_normal_family_string_unchanged(ns):
    import linreg_models as lm
    from brancher_b200 import _cuda as cu
    plan = _plan(lm.dense(ns, 1, N=30, F=5, noise=0.3)[0])
    assert plan.family == "linear regression (K2g)" and plan.likelihood == cu.GAUSSIAN


def test_scalar_weights_keep_the_dag_family(ns):
    X, y, _, rng = rm.data(0, 20, 3)
    for lik in LIKS:
        model, _ = rm.scalar_twin(ns, X, y, np.zeros(3), 0.5 * np.ones(3), likelihood=lik, noise="tied")
        assert _plan(model).family.startswith("dag")


def _reject(build, match):
    from brancher_b200 import lowering
    model = build()
    with pytest.raises(lowering.UnsupportedModelError, match=match):
        lowering._lower_dense(model, model.posterior_model)
    with pytest.raises(lowering.UnsupportedModelError):
        lowering.lower(model, model.posterior_model)


def _build(ns, lik, loc_fn, scale_fn, C=1, q_extra=(), p_extra=(), w_prior=None):
    X = np.random.RandomState(0).randn(10, 4, 1)
    x = ns.RootVariable(X, "x", is_observed=True)
    w = (w_prior or (lambda: ns.NormalVariable(np.zeros((C, 4)), np.ones((C, 4)), "weights")))()
    y = rm.variable(ns, lik)(loc_fn(w, x), scale_fn(), "y")
    model = ns.ProbabilisticModel([y] + [f() for f in p_extra])
    y.observe(np.zeros((10, C, 1)))
    Q = [ns.NormalVariable(np.zeros((C, 4)), np.ones((C, 4)), "weights", learnable=True)] + [f() for f in q_extra]
    model.set_posterior_model(ns.ProbabilisticModel(Q))
    return model


@pytest.mark.parametrize("lik", LIKS)
def test_rejects_bias(ns, lik):
    _reject(lambda: _build(ns, lik, lambda w, x: ns.BF.matmul(w, x) + ns.NormalVariable(0., 1., "b"), lambda: 0.3,
                           q_extra=[lambda: ns.NormalVariable(0., 1., "b", learnable=True)]),
            "%s linear regression 'y': a bias .* append a column of ones" % lik.capitalize())


@pytest.mark.parametrize("lik", LIKS)
def test_rejects_learnable_scale(ns, lik):
    _reject(lambda: _build(ns, lik, ns.BF.matmul, lambda: ns.RootVariable(0.3, "sig", learnable=True)),
            "%s linear regression 'y': a learnable point-estimate" % lik.capitalize())


@pytest.mark.parametrize("lik", LIKS)
def test_rejects_deterministic_scale(ns, lik):
    z = {}

    def scale():
        z["z"] = ns.NormalVariable(0., 1., "z")
        return ns.BF.exp(z["z"])
    _reject(lambda: _build(ns, lik, ns.BF.matmul, scale, q_extra=[lambda: ns.NormalVariable(0., 1., "z", learnable=True)]),
            "%s linear regression 'y': the noise scale must be a constant" % lik.capitalize())


@pytest.mark.parametrize("lik", LIKS)
def test_rejects_normal_scale(ns, lik):
    _reject(lambda: _build(ns, lik, ns.BF.matmul, lambda: ns.NormalVariable(1., 0.1, "s"),
                           q_extra=[lambda: ns.NormalVariable(1., 0.1, "s", learnable=True)]),
            "%s linear regression 'y': a normal-distributed noise scale" % lik.capitalize())


@pytest.mark.parametrize("lik", LIKS)
def test_rejects_multi_output(ns, lik):
    _reject(lambda: _build(ns, lik, ns.BF.matmul, lambda: 0.3, C=2), "%s linear regression 'y': .*multi-output" % lik.capitalize())


@pytest.mark.parametrize("lik", LIKS)
def test_rejects_extra_latents(ns, lik):
    _reject(lambda: _build(ns, lik, ns.BF.matmul, lambda: 0.3, p_extra=[lambda: ns.NormalVariable(0., 1., "extra")],
                           q_extra=[lambda: ns.NormalVariable(0., 1., "extra", learnable=True)]),
            "%s linear regression 'y': latent variables other than the weights" % lik.capitalize())


@pytest.mark.parametrize("lik", LIKS)
def test_rejects_non_normal_weight_prior(ns, lik):
    """the mean-field reduction is closed-form for Normal priors on the weights only"""
    _reject(lambda: _build(ns, lik, ns.BF.matmul, lambda: 0.3,
                           w_prior=lambda: rm.variable(ns, lik)(np.zeros((1, 4)), np.ones((1, 4)), "weights")),
            "only Normal q / Normal prior")


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", [0.3, "lognormal"])
@pytest.mark.parametrize("prior", [None, {"weights": (0.1, 0.7)}, {"weights": None, "nu": (-1.2, 0.7)}])
@pytest.mark.parametrize("with_prior", [True, False])
def test_streamed_oracle_matches_autograd_oracle(lik, noise, prior, with_prior):
    import robreg_oracle as RO
    rng = np.random.RandomState(0)
    N, F, S = 50, 5, 7
    X, y, _, _ = rm.data(1, N, F)
    params = {"weights": (0.3 * rng.randn(1, F), rng.randn(1, F) - 1), "nu": (np.array(-0.5), np.array(0.2))}
    eps = {"weights": rng.randn(S, 1, F), "nu": rng.randn(S)}
    a = RO.robreg_elbo(X, y, params, eps, prior, noise, lik, torch.float64, with_prior=with_prior)
    b = RO.robreg_elbo_streamed(X, y, params, eps, prior, noise, lik, row_chunk=16, with_prior=with_prior)
    assert set(a[1]) == set(b[1])
    np.testing.assert_allclose(b[0], a[0], rtol=1e-12)
    for k in a[1]:
        np.testing.assert_allclose(np.asarray(b[1][k]).reshape(-1), np.asarray(a[1][k]).reshape(-1), rtol=1e-10, atol=1e-10)


def test_laplace_kink_bound():
    """the kink set is empty away from r = 0; a row placed exactly on one sample's prediction is in it, and the bound covers the
    jump of that row's sign (2 |x_b| / sigma_s / S on weights_loc)"""
    import robreg_oracle as RO
    rng = np.random.RandomState(2)
    N, F, S = 40, 4, 3
    X, y, _, _ = rm.data(3, N, F)
    params = {"weights": (0.3 * rng.randn(1, F), rng.randn(1, F) - 1)}
    eps = {"weights": rng.randn(S, 1, F)}
    _, _, kb = RO.robreg_elbo_streamed(X, y, params, eps, None, 0.5, "laplace", kink=True)
    assert kb["count"] == 0 and not kb["weights_loc"].any()
    w0 = (params["weights"][0] + np.log1p(np.exp(params["weights"][1])) * eps["weights"][0]).reshape(-1)
    y2 = y.astype("f8").copy()
    y2[5] = X[5].astype("f8") @ w0
    _, _, kb = RO.robreg_elbo_streamed(X, y2, params, eps, None, 0.5, "laplace", kink=True)
    assert kb["count"] >= 1
    np.testing.assert_allclose(kb["weights_loc"].reshape(-1), 2 * np.abs(X[5].astype("f8")) / 0.5 / S, rtol=1e-12)


@pytest.mark.parametrize("lik", LIKS)
@pytest.mark.parametrize("noise", [0.3, "tied", "declared"])
def test_dense_oracle_equals_scalar_dag_twin(ns, lik, noise):
    """The dense oracle on the F = 3 model equals the scalar-DAG program of its scalar-written twin (the K1 semantics the
    live-reference goldens pin), evaluated by oracle/dag_interp.py on the same noise and parameters."""
    import robreg_oracle as RO
    from oracle import dag_interp
    from brancher_b200.lowering import _observed_tensor
    N, S = 40, 6
    rng = np.random.RandomState(5)
    X, y, _, _ = rm.data(2, N, 3)
    mu0 = (0.3 * rng.randn(1, 3)).astype("float32")
    sg0 = (0.2 + 0.3 * rng.rand(1, 3)).astype("float32")
    model, Q = rm.scalar_twin(ns, X, y, mu0, sg0, likelihood=lik, noise=noise)
    plan = _plan(model)
    assert plan.family.startswith("dag")
    P = plan.prog
    ew = rng.randn(S, 1, 3)
    enu = rng.randn(S)
    eps_by = {"w%d" % (i + 1): ew[:, 0, i] for i in range(3)}
    eps_by["nu"] = enu
    eps = np.stack([eps_by[n] for n in P.eps_names], 1)
    names = {id(v._value): v.name for v in model.posterior_model.flatten()
             if getattr(v, "learnable", False) and isinstance(getattr(v, "_value", None), torch.nn.Parameter)}
    pv = np.array([float(p.detach().reshape(())) for p in P.params])
    cols = [np.broadcast_to(_observed_tensor(c).cpu().numpy().reshape(-1), (plan.n_rows,)) for c in P.columns]
    loss_dag, dp = dag_interp.run(P.ops, P.n_slots, pv, np.stack(cols, 1), eps)
    g_dag = {names[id(p)]: dp[i] for i, p in enumerate(P.params)}
    val = {v.name: float(v._value.detach().reshape(())) for v in model.posterior_model.flatten()
           if getattr(v, "learnable", False) and isinstance(getattr(v, "_value", None), torch.nn.Parameter)}
    params = {"weights": (np.array([[val["w%d_loc" % (i + 1)] for i in range(3)]]),
                          np.array([[val["w%d_scale" % (i + 1)] for i in range(3)]]))}
    if noise != 0.3:
        params["nu"] = (np.array(val["nu_loc"]), np.array(val["nu_scale"]))
    prior = {"weights": None, "nu": (-1.2, 0.7)} if noise == "declared" else None
    loss, g = RO.robreg_elbo(X, y, params, {"weights": ew, "nu": enu}, prior, "lognormal" if noise != 0.3 else 0.3, lik, torch.float64)
    np.testing.assert_allclose(loss, loss_dag, rtol=1e-6)
    for i in range(3):
        np.testing.assert_allclose(g["weights_loc"].reshape(-1)[i], g_dag["w%d_loc" % (i + 1)], rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(g["weights_scale"].reshape(-1)[i], g_dag["w%d_scale" % (i + 1)], rtol=1e-6, atol=1e-8)
    if noise != 0.3:
        np.testing.assert_allclose(g["nu_loc"], g_dag["nu_loc"], rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(g["nu_scale"], g_dag["nu_scale"], rtol=1e-6, atol=1e-8)
