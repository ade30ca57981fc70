"""CPU: lowering of Bayesian neural networks with two to four hidden layers to the K3 family (BNNPlan over brn_bnn_deep_*), its
rejections, the one-hidden-layer network still lowering as before, and the deep oracle tied to oracle.elbo_oracle.bnn_elbo."""
import numpy as np
import pytest
import torch

import deepbnn_models as dm
import model_zoo as zoo
from deepbnn_oracle import deep_bnn_elbo, layer_names


@pytest.fixture(scope="module")
def ns():
    from brancher_b200 import config
    config.set_device("cpu")
    yield zoo.namespace("brancher_b200")
    config.set_device("cuda:0" if torch.cuda.is_available() else "cpu")


def _plan(model):
    from brancher_b200 import lowering
    return lowering.get_plan(model, model.posterior_model)


@pytest.mark.parametrize("H,acts", [((9, 5), ("tanh", "relu")), ((21, 1, 7), ("sigmoid", "tanh", "relu")),
                                    ((128, 100, 3, 17), ("relu", "relu", "sigmoid", "tanh"))])
@pytest.mark.parametrize("tied", [True, False])
def test_deep_plan(ns, H, acts, tied):
    model, Q, d = dm.api_model(ns, 3, B=10, P=6, H=H, C=4, activations=acts, tied=tied)
    plan = _plan(model)
    L = len(H)
    assert plan.family == "bnn (K3, %d hidden layers)" % L
    assert plan.activations == list(acts)
    assert len(plan.layers) == L + 1 and plan.layers[-1][2] is None
    # latent order = Philox var_id order: W1, b1, W2, b2, ..., W_out, b_out
    assert [s.name for s in plan.latents] == [n for pair in layer_names(L) for n in pair]
    dims = [6] + list(H) + [4]
    assert [s.shape for s in plan.latents] == [s for l in range(L + 1) for s in ((dims[l + 1], dims[l]), (dims[l + 1], 1))]
    assert all(s.tied == tied for s in plan.latents)
    if not tied:
        for s in plan.latents:
            np.testing.assert_allclose(s.prior_loc.numpy().reshape(-1), 0.0)
            np.testing.assert_allclose(s.prior_scale.numpy().reshape(-1), 2.0)
    assert plan.x_var is d["x"]


@pytest.mark.parametrize("act", ["tanh", "relu", "sigmoid"])
def test_one_hidden_layer_keeps_its_plan(ns, act):
    model, Q, d = zoo.bnn(ns, 1, B=12, P=20, H=7, C=4, activation=act)
    plan = _plan(model)
    assert plan.family == "bnn (K3)"
    assert plan.activations == [act]
    assert [s.name for s in plan.latents] == ["weights1", "b1", "weights2", "b2"]
    assert [s.shape for s in plan.latents] == [(7, 20), (7, 1), (4, 7), (4, 1)]


def _rejected(model, *fragments):
    from brancher_b200 import lowering
    with pytest.raises(lowering.UnsupportedModelError) as e:
        _plan(model)
    for f in fragments:
        assert f in str(e.value), str(e.value)


def test_reject_five_hidden_layers(ns):
    model, Q, d = dm.api_model(ns, 4, B=8, P=5, H=(4, 4, 4, 4, 4), C=3, activations=("tanh",) * 5)
    _rejected(model, "5 hidden layers; at most 4")


def test_reject_width_over_128(ns):
    model, Q, d = dm.api_model(ns, 5, B=8, P=5, H=(16, 129), C=3, activations=("tanh", "relu"))
    _rejected(model, "hidden layer 2: width 129", "up to 128")


def test_reject_more_than_16_classes(ns):
    model, Q, d = dm.api_model(ns, 5, B=8, P=5, H=(16, 8), C=17, activations=("tanh", "relu"))
    _rejected(model, "17 classes; at most 16")


def _net_without_bias(ns, layer):
    """three-layer network whose layer `layer` (0-based, 2 = output) has no bias"""
    rng = np.random.RandomState(0)
    B, P, H, C = 8, 5, 4, 3
    x = ns.RootVariable(rng.rand(B, P, 1).astype("f4"), "x", is_observed=True)
    shapes = {"w1": (H, P), "b1": (H, 1), "w2": (H, H), "b2": (H, 1), "w3": (C, H), "b3": (C, 1)}
    if layer is not None:
        del shapes["b%d" % (layer + 1)]
    pv = {n: ns.NormalVariable(np.zeros(s), np.ones(s), n) for n, s in shapes.items()}
    h = x
    for l in range(3):
        pre = ns.BF.matmul(pv["w%d" % (l + 1)], h)
        if "b%d" % (l + 1) in pv:
            pre = pre + pv["b%d" % (l + 1)]
        h = ns.BF.tanh(pre) if l < 2 else pre
    k = ns.CategoricalVariable(logits=h, name="k")
    model = ns.ProbabilisticModel([k])
    k.observe(rng.randint(0, C, size=B))
    model.set_posterior_model(ns.ProbabilisticModel([ns.NormalVariable(np.zeros(s), np.ones(s), n, learnable=True)
                                                     for n, s in shapes.items()]))
    return model


def test_three_layer_reference_net_lowers(ns):
    assert _plan(_net_without_bias(ns, None)).family == "bnn (K3, 2 hidden layers)"


@pytest.mark.parametrize("layer", [0, 1, 2])
def test_reject_layer_without_bias(ns, layer):
    _rejected(_net_without_bias(ns, layer), "BF.matmul(w%d, ...) has no bias" % (layer + 1))


def test_reject_other_latent(ns):
    """a latent of the model that is not a weight or bias of the network"""
    rng = np.random.RandomState(1)
    shapes, layers = dm.shapes_of(5, (4, 3), 2)
    x = ns.RootVariable(rng.rand(6, 5, 1).astype("f4"), "x", is_observed=True)
    pv = {n: ns.NormalVariable(np.zeros(s), np.ones(s), n) for n, s in shapes.items()}
    h = ns.BF.tanh(ns.BF.matmul(pv["weights1"], x) + pv["b1"])
    h = ns.BF.relu(ns.BF.matmul(pv["weights2"], h) + pv["b2"])
    k = ns.CategoricalVariable(logits=ns.BF.matmul(pv["weights_out"], h) + pv["b_out"], name="k")
    model = ns.ProbabilisticModel([k, ns.NormalVariable(0.0, 1.0, "extra")])
    k.observe(rng.randint(0, 2, size=6))
    Q = [ns.NormalVariable(np.zeros(s), np.ones(s), n, learnable=True) for n, s in shapes.items()]
    model.set_posterior_model(ns.ProbabilisticModel(Q + [ns.NormalVariable(0.0, 1.0, "extra", learnable=True)]))
    _rejected(model, "latent(s) extra are neither weights nor biases")


@pytest.mark.parametrize("act", ["tanh", "relu", "sigmoid"])
@pytest.mark.parametrize("tied", [True, False])
def test_oracle_reproduces_bnn_elbo_at_one_hidden_layer(act, tied):
    """at L = 1 the deep oracle IS oracle.elbo_oracle.bnn_elbo (pinned by the reference's goldens): bit for bit, fp32 and fp64"""
    from oracle import elbo_oracle as O
    X, y, params, eps, shapes, layers = dm.random_net(7, B=33, P=12, H=(9,), C=5, S=6)
    assert layers == [("weights1", "b1"), ("weights2", "b2")]
    prior = None if tied else {n: (0.1, 1.5) for n in shapes}
    for dtype in (torch.float32, torch.float64):
        want = O.bnn_elbo(X, y, params, eps, prior, dtype=dtype, activation=act)
        got = deep_bnn_elbo(X, y, params, eps, layers, [act], prior, dtype=dtype)
        assert got[0] == want[0]
        for k in want[1]:
            assert np.array_equal(got[1][k], want[1][k]), k
        chunked = deep_bnn_elbo(X, y, params, eps, layers, [act], prior, dtype=dtype, sample_chunk=4)
        assert abs(chunked[0] - want[0]) <= 1e-5 * abs(want[0])


def test_oracle_fp32_tracks_fp64_at_depth():
    X, y, params, eps, shapes, layers = dm.random_net(8, B=40, P=10, H=(21, 1, 100), C=7, S=3)
    acts = ["relu", "sigmoid", "tanh"]
    l32, g32 = deep_bnn_elbo(X, y, params, eps, layers, acts)
    l64, g64 = deep_bnn_elbo(X, y, params, eps, layers, acts, dtype=torch.float64)
    assert abs(l32 - l64) <= 1e-5 * abs(l64)
    for k in g64:
        assert np.abs(g32[k] - g64[k]).max() <= 1e-4 * max(np.abs(g64[k]).max(), 1e-6), k


def test_softmax_regression_with_bias_is_not_a_bnn(ns):
    """Categorical(logits = BF.matmul(W, x) + b) has no hidden layer: it stays unsupported, as before the deep networks"""
    from brancher_b200 import lowering
    rng = np.random.RandomState(2)
    x = ns.RootVariable(rng.rand(9, 5, 1).astype("f4"), "x", is_observed=True)
    W = ns.NormalVariable(np.zeros((3, 5)), np.ones((3, 5)), "W")
    b = ns.NormalVariable(np.zeros((3, 1)), np.ones((3, 1)), "b")
    k = ns.CategoricalVariable(logits=ns.BF.matmul(W, x) + b, name="k")
    model = ns.ProbabilisticModel([k])
    k.observe(rng.randint(0, 3, size=9))
    model.set_posterior_model(ns.ProbabilisticModel([ns.NormalVariable(np.zeros((3, 5)), np.ones((3, 5)), "W", learnable=True),
                                                     ns.NormalVariable(np.zeros((3, 1)), np.ones((3, 1)), "b", learnable=True)]))
    with pytest.raises(lowering.UnsupportedModelError) as e:
        _plan(model)
    assert "not recognised by any fused kernel family" in str(e.value)
