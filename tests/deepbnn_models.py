"""Deep Bayesian neural networks for the brn_bnn_deep_* tests: random parameters in the oracle's format, and the same network
built through the public API (BF.matmul / BF.tanh / BF.relu / BF.sigmoid, CategoricalVariable(logits=...))."""
import numpy as np

from deepbnn_oracle import layer_names
from oracle.elbo_oracle import softplus_inverse


def shapes_of(P, H, C):
    """{name: event shape} and the layer list of a P-H[0]-...-H[-1]-C network"""
    layers = layer_names(len(H))
    dims = [P] + list(H) + [C]
    shapes = {}
    for l, (wn, bn) in enumerate(layers):
        shapes[wn] = (dims[l + 1], dims[l])
        shapes[bn] = (dims[l + 1], 1)
    return shapes, layers


def random_net(seed, B, P, H, C, S, sigma=0.05, mu_scale=0.5, x_scale=1.0):
    """X [B, P], labels y [B], params {name: (mu, rho)}, injected noise {name: [S, *event]}, shapes, layers.
    mu_scale / sqrt(fan-in) keeps every layer's pre-activations of order one."""
    rng = np.random.RandomState(seed)
    shapes, layers = shapes_of(P, H, C)
    X = (x_scale * rng.rand(B, P)).astype("f4")
    y = rng.randint(0, C, size=B)
    params = {}
    for n, s in shapes.items():
        fan_in = s[1] if n.startswith("weights") else 1
        params[n] = ((mu_scale * rng.randn(*s) / np.sqrt(fan_in)).astype("f4"),
                     softplus_inverse(sigma * (1 + rng.rand(*s))).astype("f4"))
    eps = {n: rng.randn(S, *s).astype("f4") for n, s in shapes.items()}
    return X, y, params, eps, shapes, layers


def api_model(ns, seed, B, P, H, C, activations, tied=True, q_sigma=0.05, q_mu_scale=0.5):
    """the network through the public API; returns (model, Q, dict(X, y, shapes, layers, prior)).  tied: numeric prior
    hyper-parameters (the root names collide with q's); else the prior N(0, 2) is declared with distinctly named roots."""
    rng = np.random.RandomState(seed)
    shapes, layers = shapes_of(P, H, C)
    X = rng.rand(B, P, 1).astype("float32")
    y = rng.randint(0, C, size=(B,))
    x = ns.RootVariable(X, "x", is_observed=True)
    if tied:
        pv = {n: ns.NormalVariable(np.zeros(s), 2 * np.ones(s), n) for n, s in shapes.items()}
    else:
        pv = {n: ns.NormalVariable(ns.RootVariable(np.zeros(s), n + "_prior_loc"), ns.RootVariable(2 * np.ones(s), n + "_prior_scale"), n)
              for n, s in shapes.items()}
    h = x
    for l, (wn, bn) in enumerate(layers):
        pre = ns.BF.matmul(pv[wn], h) + pv[bn]
        h = getattr(ns.BF, activations[l])(pre) if l < len(activations) else pre
    k = ns.CategoricalVariable(logits=h, name="k")
    model = ns.ProbabilisticModel([k])
    k.observe(y)
    Q = []
    for n, s in shapes.items():
        fan_in = s[1] if n.startswith("weights") else 1
        mu0 = (q_mu_scale * rng.randn(*s) / np.sqrt(fan_in)).astype("float32")
        sg0 = (q_sigma * (1 + rng.rand(*s))).astype("float32")
        Q.append(ns.NormalVariable(mu0.astype("float64"), sg0.astype("float64"), n, learnable=True))
    model.set_posterior_model(ns.ProbabilisticModel(Q))
    prior = None if tied else {n: (0.0, 2.0) for n in shapes}
    return model, Q, {"X": X[:, :, 0], "y": y, "shapes": shapes, "layers": layers, "prior": prior, "x": x}
