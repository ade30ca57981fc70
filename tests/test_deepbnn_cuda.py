"""GPU: Bayesian neural networks with two to four hidden layers (brn_bnn_deep_*) against the autograd oracle
(tests/deepbnn_oracle.py) under the repository's parity rule, helpers.check_against_oracle.  ReLU networks leave out the data
rows whose pre-activation, at any hidden layer and sample, lies within RELU_MARGIN of the kink (fp32 rounding may put such a
unit on the other side); the number left out is printed."""
import numpy as np
import pytest
import torch

import deepbnn_models as dm
import model_zoo as zoo
from deepbnn_oracle import deep_bnn_elbo, deep_bnn_forward
from helpers import assert_close, check_against_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
RELU_MARGIN = 1e-4         # absolute, as test_bnn_tcgen05_activations


@pytest.fixture(scope="module")
def cu():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from brancher_b200 import _cuda
    _cuda.lib()
    return _cuda


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.asarray(a), dtype=dtype).to(DEV).contiguous()


def names_of(layers):
    return [n for pair in layers for n in pair]


def make_vars(cu, params, eps, names, prior=None):
    out = []
    for i, n in enumerate(names):
        mu, rho = params[n]
        e = None if eps is None else dev(eps[n]).reshape(np.asarray(eps[n]).shape[0], -1)
        pl = ps = None
        if prior is not None:
            pl, ps = dev(np.broadcast_to(prior[n][0], np.shape(mu)).copy()), dev(np.broadcast_to(prior[n][1], np.shape(mu)).copy())
        out.append(cu.MeanFieldVar(dev(mu), dev(rho), var_id=i, prior_loc=pl, prior_scale=ps, eps=e))
    return out


def run_deep(cu, X, y, params, eps, layers, acts, prior=None, r=None, with_prior=True):
    names = names_of(layers)
    S = next(iter(eps.values())).shape[0] if eps is not None else r.s_local
    vs = make_vars(cu, params, eps, names, prior)
    loss = cu.bnn_deep_elbo_fwd_bwd(dev(X), dev(y, torch.int32), vs, r or cu.sample_range(S), acts, with_prior=with_prior)
    grads = {}
    for v, n in zip(vs, names):
        grads[n + "_loc"] = v.dmu.cpu().numpy().reshape(np.shape(params[n][0]))
        grads[n + "_scale"] = v.drho.cpu().numpy().reshape(np.shape(params[n][1]))
    return loss.item(), grads


def philox_eps(cu, r, shapes, layers):
    S = r.s_local
    return {n: cu.philox_normal(int(np.prod(shapes[n])), i, r, DEV).cpu().numpy().reshape((S,) + shapes[n])
            for i, n in enumerate(names_of(layers))}


def drop_kink_rows(X, y, params, eps, layers, acts, what):
    if "relu" not in acts:
        return X, y
    _, margin = deep_bnn_forward(X, params, eps, layers, acts, sample_chunk=16)
    keep = margin > RELU_MARGIN
    print("%s: %d of %d rows within %.0e of a ReLU kink left out" % (what, (~keep).sum(), len(keep), RELU_MARGIN))
    assert keep.sum() >= len(keep) // 2
    return X[keep], y[keep]


def check(cu, X, y, params, eps, layers, acts, prior=None, with_prior=True, r=None, what="", sample_chunk=None):
    o32 = deep_bnn_elbo(X, y, params, eps, layers, acts, prior, sample_chunk=sample_chunk, with_prior=with_prior)
    o64 = deep_bnn_elbo(X, y, params, eps, layers, acts, prior, dtype=torch.float64, sample_chunk=sample_chunk, with_prior=with_prior)
    loss, grads = run_deep(cu, X, y, params, None if r is not None else eps, layers, acts, prior, r=r, with_prior=with_prior)
    check_against_oracle(loss, grads, o32, o64, what)
    return loss, grads, o32, o64


CASES = [  # B, P, H, C, S, activations, prior, with_prior
    (130, 37, (21, 100), 5, 3, ("tanh", "sigmoid"), "tied", 1),
    (257, 30, (1, 128, 21), 16, 2, ("sigmoid", "tanh", "tanh"), "declared", 1),
    (77, 33, (100, 21, 128, 1), 1, 3, ("tanh", "sigmoid", "tanh", "sigmoid"), "tied", 0),
    (200, 64, (50, 30), 7, 4, ("relu", "relu"), "declared", 1),
    (128, 16, (8, 9, 10), 3, 5, ("relu", "tanh", "sigmoid"), "tied", 1),
    (1, 5, (3, 2), 2, 1, ("tanh", "tanh"), "declared", 0),
    (300, 50, (100, 60, 33), 10, 3, ("sigmoid", "relu", "tanh"), "declared", 1),
]


@pytest.mark.parametrize("B,P,H,C,S,acts,prior,with_prior", CASES)
def test_deep_random_shapes(cu, B, P, H, C, S, acts, prior, with_prior):
    """ragged B, widths 1..128 mixed in one net, P not a multiple of 4, C 1..16, depths 2-4, every activation, tied and
    declared priors, with_prior = 0"""
    X, y, params, eps, shapes, layers = dm.random_net(B * 5 + sum(H), B, P, H, C, S)
    pr = None if prior == "tied" else {n: (0.05, 1.5) for n in shapes}
    what = "deep bnn %s" % ((B, P, H, C, S, acts, prior, with_prior),)
    X, y = drop_kink_rows(X, y, params, eps, layers, acts, what)
    check(cu, X, y, params, eps, layers, list(acts), pr, bool(with_prior), what=what)


@pytest.mark.parametrize("H,P,variant", [((100, 60), 50, "simt"), ((100, 60), 50, "tcgen05"), ((100, 60), 50, None),
                                         ((97, 128, 40), 64, "tcgen05"), ((21, 30), 48, "tcgen05"), ((90, 12), 64, "simt")])
def test_deep_layer1_variants(cu, monkeypatch, H, P, variant):
    """both layer-1 variants, forced through BRN_BNN_VARIANT; H1 = 100 takes tcgen05 by default"""
    if variant is None:
        monkeypatch.delenv("BRN_BNN_VARIANT", raising=False)
    else:
        monkeypatch.setenv("BRN_BNN_VARIANT", variant)
    B, C, S = 300, 10, 5
    X, y, params, eps, shapes, layers = dm.random_net(P + sum(H), B, P, H, C, S)
    acts = ["tanh"] * len(H)
    check(cu, X, y, params, eps, layers, acts, what="deep bnn variant %s %s" % (variant, H))
    assert cu.last_variant() == (variant or "tcgen05")


@pytest.mark.parametrize("variant", ["simt", "tcgen05"])
def test_deep_philox_and_shard_invariance(cu, monkeypatch, variant):
    """Philox noise re-materialised with philox_normal for the oracle; two sample ranges sum to the whole"""
    monkeypatch.setenv("BRN_BNN_VARIANT", variant)
    B, P, H, C, S = 150, 40, (100, 50, 20), 6, 10
    X, y, params, _, shapes, layers = dm.random_net(31, B, P, H, C, S)
    acts = ["tanh", "sigmoid", "tanh"]
    r = cu.sample_range(S, seed=99, offset=3)
    eps = philox_eps(cu, r, shapes, layers)
    loss, grads, _, _ = check(cu, X, y, params, eps, layers, acts, r=r, what="deep bnn philox " + variant)
    la, ga = run_deep(cu, X, y, params, None, layers, acts, r=cu.sample_range(S, s0=0, s_local=4, seed=99, offset=3))
    lb, gb = run_deep(cu, X, y, params, None, layers, acts, r=cu.sample_range(S, s0=4, s_local=6, seed=99, offset=3))
    assert_close(la + lb, loss, "sharded loss", rtol=1e-6)
    for k in grads:
        assert_close(ga[k] + gb[k], grads[k], "sharded grad " + k, rtol=1e-5, atol=1e-6, scale=np.abs(grads[k]).max())
    # s_local = 0 leaves every output untouched
    l0, g0 = run_deep(cu, X, y, params, None, layers, acts, r=cu.sample_range(S, s0=S, s_local=0, seed=99, offset=3))
    assert l0 == 0.0 and all(not np.any(v) for v in g0.values())


@pytest.mark.parametrize("noise", ["philox", "injected"])
def test_deep_full_config(cu, noise):
    """784-100-100-10 tanh, B = 1024, S = 256, q sigma 0.01, tied prior; the literal report goes to the full-config jsonl"""
    from test_full_config_parity import literal_report
    B, P, H, C, S = 1024, 784, (100, 100), 10, 256
    X, y, params, _, shapes, layers = dm.random_net(2027, B, P, H, C, 1, sigma=0.01, mu_scale=0.5)
    acts = ["tanh", "tanh"]
    r = cu.sample_range(S, seed=7, offset=11)
    eps = philox_eps(cu, r, shapes, layers)
    o64 = deep_bnn_elbo(X, y, params, eps, layers, acts, None, dtype=torch.float64, sample_chunk=8)
    o32 = deep_bnn_elbo(X, y, params, eps, layers, acts, None, sample_chunk=8)
    loss, grads = run_deep(cu, X, y, params, None if noise == "philox" else eps, layers, acts, r=r if noise == "philox" else None)
    assert cu.last_variant() == "tcgen05"
    literal_report("deep bnn 784-100-100-10 tanh B=1024 S=256 (%s)" % noise, dict(grads, loss=np.array(loss)),
                   dict(o64[1], loss=np.array(o64[0])), dict(o32[1], loss=np.array(o32[0])))
    check_against_oracle(loss, grads, o32, o64, "deep full config (%s)" % noise)


@pytest.mark.parametrize("B,P,H,C,S,variant,acts", [(300, 50, (100, 64), 10, 6, "tcgen05", ("tanh", "relu")),
                                                    (77, 33, (21, 5, 128), 4, 5, "simt", ("sigmoid", "tanh", "tanh"))])
def test_deep_predict_matches_forward_oracle(cu, monkeypatch, B, P, H, C, S, variant, acts):
    """bnn_deep_predict: logits vs the oracle's fp64 forward pass on the re-materialised Philox weights, probs = MC mean of the
    softmax, class draws distributed as the probabilities"""
    monkeypatch.setenv("BRN_BNN_VARIANT", variant)
    X, y, params, _, shapes, layers = dm.random_net(B + sum(H), B, P, H, C, S)
    r = cu.sample_range(S, seed=21, offset=4)
    mv = make_vars(cu, params, None, names_of(layers))
    logits, labels, probs = cu.bnn_deep_predict(dev(X), mv, r, list(acts))
    assert cu.last_variant() == variant
    eps = philox_eps(cu, r, shapes, layers)
    a, margin = deep_bnn_forward(X, params, eps, layers, list(acts))
    keep = margin > RELU_MARGIN if "relu" in acts else np.ones(B, bool)
    print("deep predict %s: %d of %d rows within %.0e of a ReLU kink left out" % (acts, (~keep).sum(), B, RELU_MARGIN))
    assert_close(logits.cpu().numpy()[:, keep], a[:, keep], "predict logits", scale=np.abs(a).max())
    e = np.exp(a - a.max(-1, keepdims=True))
    p = e / e.sum(-1, keepdims=True)
    assert_close(probs.cpu().numpy()[keep], p.mean(0)[keep], "predict probs", rtol=1e-5, atol=1e-6)
    lab = labels.cpu().numpy()
    assert lab.shape == (S, B) and lab.min() >= 0 and lab.max() < C
    freq = np.bincount(lab.reshape(-1), minlength=C) / lab.size
    want = p.reshape(-1, C).mean(0)
    assert np.all(np.abs(freq - want) <= 5 * np.sqrt(want * (1 - want) / lab.size) + 1e-3), (freq, want)


# ------------------------------------------------------------------------------------------------ public API
@pytest.fixture(scope="module")
def ns():
    from brancher_b200 import config
    config.set_device(DEV)
    return zoo.namespace("brancher_b200")


def _q_params(model, names):
    """{name: (mu, rho)} of the posterior's learnable roots, in the oracle's format"""
    by = {v.name: v for v in model.posterior_model.flatten()}
    return {n: (by[n].roots["loc"].value.detach().cpu().numpy().reshape(-1).astype("f4"),
                by[n].roots["scale"].value.detach().cpu().numpy().reshape(-1).astype("f4")) for n in names}


@pytest.mark.parametrize("tied", [True, False])
def test_deep_api_reverse_kl_matches_oracle(ns, tied):
    """ReverseKL().compute_loss + backward through the public API with injected noise vs the oracle"""
    from brancher_b200 import lowering
    H, C, S, acts = (100, 30, 12), 6, 4, ("tanh", "sigmoid", "tanh")
    model, Q, d = dm.api_model(ns, 13, B=90, P=20, H=H, C=C, activations=acts, tied=tied)
    layers, shapes = d["layers"], d["shapes"]
    rng = np.random.RandomState(5)
    eps = {n: rng.randn(S, *shapes[n]).astype("f4") for n in shapes}
    with lowering.inject_noise(eps):
        loss = ns.inference.ReverseKL().compute_loss(model, model.posterior_model, None, S)
    assert lowering.get_plan(model, model.posterior_model).family == "bnn (K3, 3 hidden layers)"
    loss.backward()
    by = {v.name: v for v in model.posterior_model.flatten()}
    grads = {}
    for n in shapes:
        grads[n + "_loc"] = by[n].roots["loc"].value.grad.detach().cpu().numpy().reshape(shapes[n])
        grads[n + "_scale"] = by[n].roots["scale"].value.grad.detach().cpu().numpy().reshape(shapes[n])
    params = {n: (m.reshape(shapes[n]), r.reshape(shapes[n])) for n, (m, r) in _q_params(model, list(shapes)).items()}
    o32 = deep_bnn_elbo(d["X"], d["y"], params, eps, layers, list(acts), d["prior"])
    o64 = deep_bnn_elbo(d["X"], d["y"], params, eps, layers, list(acts), d["prior"], dtype=torch.float64)
    check_against_oracle(float(loss.detach()), grads, o32, o64, "deep bnn via API")


def test_deep_api_perform_inference_and_predictive(ns):
    from brancher_b200 import config, inference
    config.set_seed(3)
    model, Q, d = dm.api_model(ns, 17, B=200, P=16, H=(32, 24), C=4, activations=("relu", "tanh"))
    inference.perform_inference(model, number_iterations=60, number_samples=8, optimizer="Adam", lr=0.01,
                                inference_method=inference.ReverseKL())
    curve = np.asarray(model.diagnostics["loss curve"]).reshape(-1)
    assert curve.shape == (60,) and np.isfinite(curve).all() and curve[-10:].mean() < curve[:10].mean()
    out = model.get_posterior_predictive(12, {d["x"]: d["X"][:25]})
    assert tuple(out["logits"].shape) == (12, 25, 4) and tuple(out["samples"].shape) == (12, 25)
    p = out["probs"].cpu().numpy()
    assert p.shape == (25, 4) and np.allclose(p.sum(1), 1.0, atol=1e-5)
    np.testing.assert_allclose(p, torch.softmax(out["logits"], -1).mean(0).cpu().numpy(), rtol=1e-5, atol=1e-6)


def test_deep_graph_loop_equals_stepwise_loop(ns):
    """the CUDA-graph-captured training loop over the deep evaluation equals the step-by-step loop (as tests/test_fused_loop.py)"""
    from brancher_b200 import config, inference
    out = {}
    for mode in ("graph", "eager"):
        config.set_seed(123)
        model, Q, d = dm.api_model(ns, 19, B=130, P=40, H=(100, 40, 17), C=10, activations=("tanh", "sigmoid", "tanh"))
        inference.fused_loop_enabled = mode == "graph"
        try:
            inference.perform_inference(model, number_iterations=12, number_samples=6, optimizer="Adam", lr=1e-3,
                                        inference_method=inference.ReverseKL())
        finally:
            inference.fused_loop_enabled = True
        assert inference.last_loop == mode
        vals = {v.name: v.link.parameter.detach().cpu().numpy().copy() for v in model.posterior_model.flatten()
                if getattr(v, "learnable", False) and hasattr(v.link, "parameter")}
        out[mode] = (np.asarray(model.diagnostics["loss curve"], dtype=np.float64).reshape(-1), vals)
    cg, ce = out["graph"][0], out["eager"][0]
    assert cg.shape == ce.shape == (12,) and np.isfinite(cg).all()
    np.testing.assert_allclose(cg, ce, rtol=2e-5, atol=1e-5 * np.abs(ce).max())
    for k, v in out["eager"][1].items():
        np.testing.assert_allclose(out["graph"][1][k], v, rtol=1e-4, atol=1e-5 * max(np.abs(v).max(), 1e-6), err_msg=k)


def test_deep_forced_tcgen05_rejects_wide_first_layer(cu, monkeypatch):
    """BRN_BNN_VARIANT=tcgen05 with H1 above the instantiated tile is an error, as for brn_bnn_elbo_fwd_bwd_act, and writes nothing"""
    monkeypatch.setenv("BRN_BNN_VARIANT", "tcgen05")
    X, y, params, eps, shapes, layers = dm.random_net(3, 40, 20, (120, 16), 4, 2)
    vs = make_vars(cu, params, eps, names_of(layers))
    with pytest.raises(cu.BrancherCudaError, match="BRN_BNN_VARIANT=tcgen05 needs H\\[0\\] <= 104 \\(got 120\\)"):
        cu.bnn_deep_elbo_fwd_bwd(dev(X), dev(y, torch.int32), vs, cu.sample_range(2), ["tanh", "tanh"])
    assert all(not v.dmu.any() and not v.drho.any() for v in vs)
