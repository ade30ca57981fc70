"""CPU: lowering of Bayesian linear regression (Normal likelihood over BF.matmul(weights, x)) to the K2g family, its
rejections, and the dense oracle against the streamed oracle and against the scalar-DAG semantics of the same model."""
import numpy as np
import pytest
import torch

import linreg_models as lm
import model_zoo as zoo


@pytest.fixture(scope="module")
def ns():
    from brancher_b200 import config
    config.set_device("cpu")
    yield zoo.namespace("brancher_b200")
    config.set_device("cuda:0" if torch.cuda.is_available() else "cpu")


def _plan(model):
    from brancher_b200 import lowering
    return lowering.get_plan(model, model.posterior_model)


@pytest.mark.parametrize("noise", [0.3, "tied", "declared"])
def test_linreg_lowers(ns, noise):
    model, Q, d = lm.dense(ns, 1, N=30, F=5, noise=noise)
    plan = _plan(model)
    assert plan.family.startswith("linear regression")
    assert [s.name for s in plan.latents] == (["weights"] if noise == 0.3 else ["weights", "nu"])
    assert plan.latents[0].shape == (1, 5) and plan.latents[0].tied
    if noise == 0.3:
        np.testing.assert_allclose(plan.noise_scale().item(), 0.3, rtol=1e-6)
    else:
        nu = plan.latents[1]
        assert nu.tied == (noise == "tied") and int(np.prod(nu.shape)) == 1
        assert len(nu.parameters()) == 2
        if noise == "declared":
            np.testing.assert_allclose(nu.prior_loc.item(), -1.2, rtol=1e-6)
            np.testing.assert_allclose(nu.prior_scale.item(), 0.7, rtol=1e-6)


def test_logreg_and_scalar_regression_keep_their_families(ns):
    assert _plan(zoo.logreg(ns, 3, B=40, F=8, tied=True)[0]).family.startswith("linear (K2)")
    assert _plan(zoo.multivariate_regression(ns, 0, 20)[0]).family.startswith("dag")


def _reject(ns, build, match):
    from brancher_b200 import lowering
    model = build()
    with pytest.raises(lowering.UnsupportedModelError, match=match):
        lowering._lower_dense(model, model.posterior_model)
    with pytest.raises(lowering.UnsupportedModelError):
        lowering.lower(model, model.posterior_model)


def _model(ns, loc_fn, scale_fn, C=1, extra_q=(), N=10, F=4):
    X = np.random.RandomState(0).randn(N, F, 1)
    x = ns.RootVariable(X, "x", is_observed=True)
    w = ns.NormalVariable(np.zeros((C, F)), np.ones((C, F)), "weights")
    y = ns.NormalVariable(loc_fn(w, x), scale_fn(), "y")
    model = ns.ProbabilisticModel([y])
    y.observe(np.zeros((N, C, 1)) if C > 1 else np.zeros((N, 1, 1)))
    Q = [ns.NormalVariable(np.zeros((C, F)), np.ones((C, F)), "weights", learnable=True)] + [f() for f in extra_q]
    model.set_posterior_model(ns.ProbabilisticModel(Q))
    return model


def test_rejects_bias(ns):
    def build():
        b = ns.NormalVariable(0., 1., "b")
        X = np.random.RandomState(0).randn(10, 4, 1)
        x = ns.RootVariable(X, "x", is_observed=True)
        w = ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights")
        y = ns.NormalVariable(ns.BF.matmul(w, x) + b, 0.3, "y")
        model = ns.ProbabilisticModel([y])
        y.observe(np.zeros((10, 1, 1)))
        model.set_posterior_model(ns.ProbabilisticModel([ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights", learnable=True),
                                                         ns.NormalVariable(0., 1., "b", learnable=True)]))
        return model
    _reject(ns, build, "append a column of ones")


def test_rejects_learnable_scale(ns):
    _reject(ns, lambda: _model(ns, ns.BF.matmul, lambda: ns.RootVariable(0.3, "sig", learnable=True)), "learnable point-estimate")


def test_rejects_deterministic_scale(ns):
    def build():
        X = np.random.RandomState(0).randn(10, 4, 1)
        x = ns.RootVariable(X, "x", is_observed=True)
        w = ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights")
        z = ns.NormalVariable(0., 1., "z")
        y = ns.NormalVariable(ns.BF.matmul(w, x), ns.BF.exp(z), "y")
        model = ns.ProbabilisticModel([y])
        y.observe(np.zeros((10, 1, 1)))
        model.set_posterior_model(ns.ProbabilisticModel([ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights", learnable=True),
                                                         ns.NormalVariable(0., 1., "z", learnable=True)]))
        return model
    _reject(ns, build, "noise scale must be a constant")


def test_rejects_normal_scale(ns):
    def build():
        X = np.random.RandomState(0).randn(10, 4, 1)
        x = ns.RootVariable(X, "x", is_observed=True)
        w = ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights")
        s = ns.NormalVariable(1., 0.1, "s")
        y = ns.NormalVariable(ns.BF.matmul(w, x), s, "y")
        model = ns.ProbabilisticModel([y])
        y.observe(np.zeros((10, 1, 1)))
        model.set_posterior_model(ns.ProbabilisticModel([ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights", learnable=True),
                                                         ns.NormalVariable(1., 0.1, "s", learnable=True)]))
        return model
    _reject(ns, build, "normal-distributed noise scale")


def test_rejects_multi_output(ns):
    _reject(ns, lambda: _model(ns, ns.BF.matmul, lambda: 0.3, C=2), "multi-output")


def test_rejects_extra_latents(ns):
    def build():
        X = np.random.RandomState(0).randn(10, 4, 1)
        x = ns.RootVariable(X, "x", is_observed=True)
        w = ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights")
        extra = ns.NormalVariable(0., 1., "extra")
        y = ns.NormalVariable(ns.BF.matmul(w, x), 0.3, "y")
        model = ns.ProbabilisticModel([y, extra])
        y.observe(np.zeros((10, 1, 1)))
        model.set_posterior_model(ns.ProbabilisticModel([ns.NormalVariable(np.zeros((1, 4)), np.ones((1, 4)), "weights", learnable=True),
                                                         ns.NormalVariable(0., 1., "extra", learnable=True)]))
        return model
    _reject(ns, build, "other than the weights")


@pytest.mark.parametrize("noise", [0.3, "lognormal"])
@pytest.mark.parametrize("prior", [None, {"weights": (0.1, 0.7)}, {"weights": None, "nu": (-1.2, 0.7)}])
@pytest.mark.parametrize("with_prior", [True, False])
def test_streamed_oracle_matches_autograd_oracle(noise, prior, with_prior):
    import linreg_oracle as LO
    rng = np.random.RandomState(0)
    N, F, S = 50, 5, 7
    X, y, _, _ = lm.data(1, N, F)
    params = {"weights": (0.3 * rng.randn(1, F), rng.randn(1, F) - 1), "nu": (np.array(-0.5), np.array(0.2))}
    eps = {"weights": rng.randn(S, 1, F), "nu": rng.randn(S)}
    a = LO.linreg_elbo(X, y, params, eps, prior, noise, torch.float64, with_prior=with_prior)
    b = LO.linreg_elbo_streamed(X, y, params, eps, prior, noise, row_chunk=16, with_prior=with_prior)
    assert set(a[1]) == set(b[1])
    np.testing.assert_allclose(b[0], a[0], rtol=1e-12)
    for k in a[1]:
        np.testing.assert_allclose(np.asarray(b[1][k]).reshape(-1), np.asarray(a[1][k]).reshape(-1), rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize("noise", [0.3, "tied", "declared"])
def test_dense_oracle_equals_scalar_dag_twin(ns, noise):
    """The dense oracle on the F = 3 model equals the scalar-DAG program of its scalar-written twin (the K1 semantics the
    live-reference goldens pin), evaluated by oracle/dag_interp.py on the same noise and parameters."""
    import linreg_oracle as LO
    from oracle import dag_interp
    from brancher_b200.lowering import _observed_tensor
    N, S = 40, 6
    rng = np.random.RandomState(5)
    X, y, _, _ = lm.data(2, N, 3)
    mu0 = (0.3 * rng.randn(1, 3)).astype("float32")
    sg0 = (0.2 + 0.3 * rng.rand(1, 3)).astype("float32")
    model, Q = lm.scalar_twin(ns, X, y, mu0, sg0, noise=noise)
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

    pget = lambda n: float(g_dag_param(model, n))
    params = {"weights": (np.array([[pget("w%d_loc" % (i + 1)) for i in range(3)]]),
                          np.array([[pget("w%d_scale" % (i + 1)) for i in range(3)]]))}
    if noise != 0.3:
        params["nu"] = (np.array(pget("nu_loc")), np.array(pget("nu_scale")))
    prior = {"weights": None, "nu": (-1.2, 0.7)} if noise == "declared" else None
    loss, g = LO.linreg_elbo(X, y, params, {"weights": ew, "nu": enu}, prior, "lognormal" if noise != 0.3 else 0.3, torch.float64)
    np.testing.assert_allclose(loss, loss_dag, rtol=1e-6)
    for i in range(3):
        np.testing.assert_allclose(g["weights_loc"].reshape(-1)[i], g_dag["w%d_loc" % (i + 1)], rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(g["weights_scale"].reshape(-1)[i], g_dag["w%d_scale" % (i + 1)], rtol=1e-6, atol=1e-8)
    if noise != 0.3:
        np.testing.assert_allclose(g["nu_loc"], g_dag["nu_loc"], rtol=1e-6, atol=1e-8)
        np.testing.assert_allclose(g["nu_scale"], g_dag["nu_scale"], rtol=1e-6, atol=1e-8)


def g_dag_param(model, name):
    for v in model.posterior_model.flatten():
        if v.name == name and getattr(v, "learnable", False):
            return v._value.detach().reshape(())
    raise KeyError(name)
