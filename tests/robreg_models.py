"""Robust Bayesian linear regression models for the K2g Cauchy / Laplace tests, built through the public API (same conventions as
linreg_models.py): y ~ Cauchy / Laplace(BF.matmul(weights, x), noise) over a dense design matrix with heavy-tailed data, and
its scalar-written twin for F = 3 (w1 * x1 + w2 * x2 + w3 * x3), which lowers to the scalar-DAG family."""
import numpy as np

from linreg_models import _noise

LIKELIHOODS = ("cauchy", "laplace")


def variable(ns, likelihood):
    return ns.CauchyVariable if likelihood == "cauchy" else ns.LaplaceVariable


def data(seed, N, F, noise_sd=0.3):
    """y = X w* + noise_sd * standard-Cauchy noise"""
    rng = np.random.RandomState(seed)
    X = rng.randn(N, F).astype("float32")
    wtrue = rng.randn(F) / np.sqrt(F)
    y = (X @ wtrue + noise_sd * rng.standard_cauchy(N)).astype("float32")
    return X, y, wtrue, rng


def dense(ns, seed, N, F, likelihood="cauchy", noise="tied", tied_weights=True, mu0=None, sg0=None):
    """returns (model, Q, dict(X, y, prior, wtrue)); prior in the oracle's format (None = everything tied)"""
    X, y, wtrue, rng = data(seed, N, F)
    x = ns.RootVariable(X[:, :, None], "x", is_observed=True)
    if tied_weights:
        w = ns.NormalVariable(np.zeros((1, F)), 0.5 * np.ones((1, F)), "weights")
    else:
        w = ns.NormalVariable(ns.RootVariable(np.zeros((1, F)), "w_prior_loc"), ns.RootVariable(0.5 * np.ones((1, F)), "w_prior_scale"),
                              "weights")
    yv = variable(ns, likelihood)(ns.BF.matmul(w, x), _noise(ns, noise, q=False), "y")
    model = ns.ProbabilisticModel([yv])
    yv.observe(y.reshape(N, 1, 1))
    mu0 = (0.3 * rng.randn(1, F)).astype("float32") if mu0 is None else mu0
    sg0 = (0.2 + 0.3 * rng.rand(1, F)).astype("float32") if sg0 is None else sg0
    Q = [ns.NormalVariable(mu0.astype("float64"), sg0.astype("float64"), "weights", learnable=True)]
    if not isinstance(noise, (int, float)):
        Q.append(_noise(ns, noise, q=True))
    model.set_posterior_model(ns.ProbabilisticModel(Q))
    prior = {}
    if not tied_weights:
        prior["weights"] = (0.0, 0.5)
    if noise == "declared":
        prior["nu"] = (-1.2, 0.7)
    if prior and "weights" not in prior:
        prior["weights"] = None
    return model, Q, {"X": X, "y": y, "prior": prior or None, "wtrue": wtrue, "rng": rng}


def scalar_twin(ns, X, y, mu0, sg0, likelihood="cauchy", noise="tied"):
    """the same model for F = 3 with three scalar weights (w1 * x1 + w2 * x2 + w3 * x3) and tied Normal priors N(0, 0.5)"""
    N, F = X.shape
    assert F == 3
    xs = [ns.DeterministicVariable(X[:, i].astype("float64"), name="x%d" % (i + 1), is_observed=True) for i in range(F)]
    ws = [ns.NormalVariable(0., 0.5, name="w%d" % (i + 1)) for i in range(F)]
    mean = ws[0] * xs[0] + ws[1] * xs[1] + ws[2] * xs[2]
    yv = variable(ns, likelihood)(mean, _noise(ns, noise, q=False), name="y")
    model = ns.ProbabilisticModel([yv])
    Q = [ns.NormalVariable(float(mu0.reshape(-1)[i]), float(sg0.reshape(-1)[i]), name="w%d" % (i + 1), learnable=True)
         for i in range(F)]
    if not isinstance(noise, (int, float)):
        Q.append(_noise(ns, noise, q=True))
    model.set_posterior_model(ns.ProbabilisticModel(Q))
    yv.observe(y.reshape(N, 1, 1))
    return model, Q
