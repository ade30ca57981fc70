"""Regression particle models for the K4a / K6b regression tests, built through the public API: y ~ Normal / Cauchy / Laplace(
BF.matmul(weights, x), scale) over a dense design matrix with a constant scale, and the particle ensembles SVGD, MAP and WVGD
take (one learnable root named "weights" per particle; WVGD adds one learnable Normal sampler per particle)."""
import numpy as np

LIKELIHOODS = ("normal", "cauchy", "laplace")
PRIOR = (0.0, 2.0)


def variable(ns, likelihood):
    return {"normal": ns.NormalVariable, "cauchy": ns.CauchyVariable, "laplace": ns.LaplaceVariable}[likelihood]


def data(seed, N, F, noise_sd=0.3, likelihood="normal"):
    """y = X w* + noise_sd * (standard Normal, or standard Cauchy for the robust likelihoods)"""
    rng = np.random.RandomState(seed)
    X = rng.randn(N, F).astype("float32")
    wtrue = rng.randn(F) / np.sqrt(F)
    noise = rng.randn(N) if likelihood == "normal" else rng.standard_cauchy(N)
    y = (X @ wtrue + noise_sd * noise).astype("float32")
    return X, y, wtrue, rng


def scale_of(ns, form, value=0.3):
    """the constant scale forms: "number" (auto-named root behind a softplus) or "root" (a non-learnable RootVariable)"""
    return value if form == "number" else ns.RootVariable(value, "sigma")


def joint(ns, X, y, likelihood="normal", scale="number"):
    N, F = X.shape
    x = ns.RootVariable(X[:, :, None], "x", is_observed=True)
    w = ns.NormalVariable(PRIOR[0] * np.ones((1, F)), PRIOR[1] * np.ones((1, F)), "weights")
    yv = variable(ns, likelihood)(ns.BF.matmul(w, x), scale_of(ns, scale), "y")
    model = ns.ProbabilisticModel([yv])
    yv.observe(y.reshape(N, 1, 1))
    return model


def particles(ns, theta):
    """theta [n, 1, F] -> one single-root ProbabilisticModel per particle"""
    return [ns.ProbabilisticModel([ns.RootVariable(np.asarray(t, np.float64), name="weights", learnable=True)]) for t in theta]


def samplers(ns, loc, q_sigma=0.3):
    return [ns.ProbabilisticModel([ns.NormalVariable(loc=np.asarray(l, np.float64), scale=q_sigma, name="weights", learnable=True)])
            for l in loc]


def map_model(ns, X, y, likelihood="normal", scale="number", w0=None):
    """joint model with a one-root point-estimate posterior (MAP)"""
    model = joint(ns, X, y, likelihood, scale)
    w0 = np.zeros((1, X.shape[1])) if w0 is None else w0
    point = ns.ProbabilisticModel([ns.RootVariable(np.asarray(w0, np.float64), name="weights", learnable=True)])
    model.set_posterior_model(point)
    return model, point


def scalar_twin(ns, X, y, likelihood="normal", w0=None):
    """the same MAP problem for F = 3 with three scalar weights (w1 * x1 + w2 * x2 + w3 * x3), priors N(PRIOR); lowers to K1"""
    N, F = X.shape
    assert F == 3
    xs = [ns.DeterministicVariable(X[:, i].astype("float64"), name="x%d" % (i + 1), is_observed=True) for i in range(F)]
    ws = [ns.NormalVariable(PRIOR[0], PRIOR[1], name="w%d" % (i + 1)) for i in range(F)]
    yv = variable(ns, likelihood)(ws[0] * xs[0] + ws[1] * xs[1] + ws[2] * xs[2], 0.3, name="y")
    model = ns.ProbabilisticModel([yv])
    yv.observe(y.reshape(N, 1, 1))
    w0 = np.zeros(F) if w0 is None else np.asarray(w0).reshape(-1)
    point = ns.ProbabilisticModel([ns.RootVariable(float(w0[i]), name="w%d" % (i + 1), learnable=True) for i in range(F)])
    model.set_posterior_model(point)
    return model, point
