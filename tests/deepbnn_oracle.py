"""Autograd oracle of the Bayesian neural network with 1..4 hidden layers (the brn_bnn_deep_* networks): the ELBO and its
gradients, restated on the oracle package's mean-field machinery (oracle.elbo_oracle.MeanFieldNormal).

    h_0 = x,  h_l = act_l(W_l h_{l-1} + b_l)  (l = 1..L),  logits = W_out h_L + b_out,  k ~ Categorical(logits) observed

`layers` names the (weights, bias) variables from the input layer outward, the output layer last; `activations` holds one of
"tanh" / "relu" / "sigmoid" per hidden layer.  Weights have event shape [n_out, n_in], biases [n_out, 1].  With one hidden layer
and the names weights1, b1, weights2, b2 this is oracle.elbo_oracle.bnn_elbo operation for operation."""
import numpy as np
import torch
import torch.distributions as D

from oracle.elbo_oracle import MeanFieldNormal, _t

ACT = {"tanh": torch.tanh, "relu": torch.relu, "sigmoid": torch.sigmoid}


def layer_names(n_hidden):
    """(weights, bias) names of a network with n_hidden hidden layers: weights1, b1, ..., weights_out, b_out (the two-layer
    network keeps weights2, b2)"""
    names = [("weights%d" % (l + 1), "b%d" % (l + 1)) for l in range(n_hidden)]
    return names + [("weights%d" % (n_hidden + 1), "b%d" % (n_hidden + 1)) if n_hidden == 1 else ("weights_out", "b_out")]


def _forward(Xt, w, sl, layers, activations):
    """logits [s, B, C] and the pre-activations of every hidden layer"""
    pres = []
    h = None
    for l, (wn, bn) in enumerate(layers):
        if l == 0:
            pre = torch.einsum("shp,bp->sbh", w[wn][sl], Xt) + w[bn][sl, :, 0].unsqueeze(1)
        else:
            pre = torch.einsum("sch,sbh->sbc", w[wn][sl], h) + w[bn][sl, :, 0].unsqueeze(1)
        if l == len(layers) - 1:
            return pre, pres
        pres.append(pre)
        h = ACT[activations[l]](pre)


def deep_bnn_elbo(X, y, params, eps, layers, activations, prior=None, dtype=torch.float32, sample_chunk=None, with_prior=True):
    """(loss = -ELBO, {name_loc / name_scale: gradient}) as oracle.elbo_oracle.bnn_elbo returns them"""
    assert len(activations) == len(layers) - 1
    q = MeanFieldNormal(params, eps, prior, dtype)
    w = q.sample()
    Xt = _t(X, dtype)
    yt = _t(y, torch.int64)
    S = q.S
    step = sample_chunk or S
    lls = []
    for s0 in range(0, S, step):
        a, _ = _forward(Xt, w, slice(s0, s0 + step), layers, activations)
        lp = D.Categorical(logits=a).log_prob(yt.unsqueeze(0))      # [s,B]
        lls.append(lp.sum(dim=1))
    per_sample = torch.cat(lls)
    if with_prior:
        per_sample = per_sample + q.log_prior()
    elbo = per_sample.mean()
    if with_prior:
        elbo = elbo + q.entropy()
    loss = -elbo
    loss.backward()
    return float(loss.detach()), q.grads()


def deep_bnn_forward(X, params, eps, layers, activations, sample_chunk=None):
    """fp64 forward pass without gradients: (logits [S, B, C], smallest |pre-activation| of each row over every hidden layer
    and sample [B]) -- the second for leaving rows at a ReLU kink out of a comparison"""
    with torch.no_grad():
        q = MeanFieldNormal(params, eps, None, torch.float64)
        w = q.sample()
        Xt = _t(X, torch.float64)
        step = sample_chunk or q.S
        logits, margin = [], torch.full((Xt.shape[0],), float("inf"), dtype=torch.float64)
        for s0 in range(0, q.S, step):
            a, pres = _forward(Xt, w, slice(s0, s0 + step), layers, activations)
            logits.append(a)
            for p in pres:
                margin = torch.minimum(margin, p.abs().amin(dim=(0, 2)))
        return torch.cat(logits).numpy(), margin.numpy()
