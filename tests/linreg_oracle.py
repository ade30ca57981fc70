"""TEST INFRASTRUCTURE ONLY: the oracle of Bayesian linear regression (K2g), in the conventions of oracle/elbo_oracle.py --
`loss = -ELBO` as a python float and gradients keyed by the reference's parameter names (`<var>_loc`, `<var>_scale` = d loss /
d rho).  `linreg_elbo` restates the objective with torch.distributions and autograd; `linreg_elbo_streamed` is the fp64
row-streamed version with the gradient written out by hand, pinned against it in tests/test_linreg_lowering.py."""
import math

import numpy as np
import torch
import torch.distributions as D
import torch.nn.functional as F

from oracle.elbo_oracle import MeanFieldNormal, F_softplus, _t


def linreg_elbo(X, y, params, eps, prior=None, noise="lognormal", dtype=torch.float32, with_prior=True):
    """Bayesian linear regression: y_b ~ Normal(BF.matmul(weights, x)_b, sigma) over N observed rows (summed,
    variables.py:513-514), weights [1, F] mean-field Normal as in `logreg_elbo`.

    noise: a number -> sigma is that constant (the auto-named root `y_scale`, non-learnable);
           "lognormal" -> sigma = nu, a scalar LogNormal latent: q(nu) = LogNormal(m, softplus(rho)) from params["nu"] and
           eps["nu"] [S]; p(nu) = LogNormal with q's roots (tied, prior None or no "nu" entry) or prior["nu"] = (loc, scale).
    log p(nu) and H[q(nu)] are torch's LogNormal (TransformedDistribution) terms -- Normal.log_prob(log nu) - log nu and
    Normal.entropy() + loc -- the order the scalar-DAG family composes them in.
    prior: None (everything tied) or {"weights": (loc, scale) or None (tied), optionally "nu": (loc, scale)}.
    """
    wprior = {"weights": prior["weights"]} if prior is not None and prior.get("weights") is not None else None
    q = MeanFieldNormal({"weights": params["weights"]}, {"weights": eps["weights"]}, wprior, dtype)
    w = q.sample()["weights"]                       # [S,1,F]
    S = q.S
    Xt = _t(X, dtype)
    yt = _t(y, dtype).reshape(-1)
    loc = torch.einsum("scf,bf->sb", w, Xt)
    if noise == "lognormal":
        m = _t(params["nu"][0], dtype, True)
        rho = _t(params["nu"][1], dtype, True)
        sg = F.softplus(rho).reshape(())
        e = _t(eps["nu"], dtype).reshape(S)
        nu = torch.exp(m.reshape(()) + e * sg)      # LogNormal rsample: exp(loc + eps * scale)
        sigma = nu[:, None]
    else:
        sigma = torch.tensor(float(noise), dtype=dtype)
    ll = D.Normal(loc, sigma).log_prob(yt[None, :]).sum(dim=1)
    per_sample = ll
    if with_prior:
        per_sample = per_sample + q.log_prior()
        if noise == "lognormal":
            if prior is not None and "nu" in prior:
                a, b = _t(prior["nu"][0], dtype).reshape(()), _t(prior["nu"][1], dtype).reshape(())
            else:
                a, b = m.reshape(()), sg
            per_sample = per_sample + D.LogNormal(a, b).log_prob(nu)
    elbo = per_sample.mean()
    if with_prior:
        elbo = elbo + q.entropy()
        if noise == "lognormal":
            elbo = elbo + D.LogNormal(m.reshape(()), sg).entropy()
    loss = -elbo
    loss.backward()
    g = q.grads()
    if noise == "lognormal":
        g["nu_loc"] = m.grad.detach().numpy().copy()
        g["nu_scale"] = rho.grad.detach().numpy().copy()
    return float(loss.detach()), g


def linreg_elbo_streamed(X, y, params, eps, prior=None, noise="lognormal", dtype=torch.float64, row_chunk=65536,
                         with_prior=True):
    """`linreg_elbo` with the rows streamed and the gradient written out by hand.  Per sample, with residuals
    r_sb = y_b - w_s . x_b, R_s = sum_b r_sb^2, G_s = sum_b r_sb x_b and sigma_s = exp(u_s), u_s = m + softplus(rho) e_s:
        ll_s = -R_s / (2 sigma_s^2) - N log sigma_s - N/2 log(2 pi)
        d ll_s / d w_s = G_s / sigma_s^2,   d ll_s / d u_s = R_s / sigma_s^2 - N
    log p(nu_s) = Normal(a, b).log_prob(u_s) - u_s (tied: a = m, b = softplus(rho), differentiated through both),
    H[q(nu)] = 1/2 + log sqrt(2 pi) + log softplus(rho) + m."""
    mu, rho = (_t(a, dtype) for a in params["weights"])
    e = _t(eps["weights"], dtype)                                   # [S, 1, F]
    S, F = e.shape[0], e.shape[-1]
    sg = F_softplus(rho)
    w = (mu + sg * e).reshape(S, F)
    Xt = torch.as_tensor(np.asarray(X))
    yt = torch.as_tensor(np.asarray(y)).reshape(-1)
    N = Xt.shape[0]
    R = torch.zeros(S, dtype=dtype)
    G = torch.zeros(S, F, dtype=dtype)
    with torch.no_grad():
        for r0 in range(0, N, row_chunk):
            xb = Xt[r0:r0 + row_chunk].to(dtype)
            rb = yt[r0:r0 + row_chunk].to(dtype)[None, :] - w @ xb.T        # [S, rows]
            R += (rb * rb).sum(1)
            G += rb @ xb
    c = 0.5 * math.log(2 * math.pi)
    if noise == "lognormal":
        m, rn = (_t(a, dtype).reshape(()) for a in params["nu"])
        sgn = F_softplus(rn)
        en = _t(eps["nu"], dtype).reshape(S)
        u = m + sgn * en
        sigma = torch.exp(u)
    else:
        u = torch.full((S,), math.log(float(noise)), dtype=dtype)
        sigma = torch.exp(u)
    inv_s2 = 1.0 / (sigma * sigma)
    ll = -0.5 * R * inv_s2 - N * u - N * c
    gw = G * inv_s2[:, None]                                        # d ll_s / d w_s
    e2 = e.reshape(S, -1)
    muf, sgf, rhof = mu.reshape(-1), sg.reshape(-1), rho.reshape(-1)
    if not with_prior:
        lp = torch.zeros(S, dtype=dtype)
        dlp_dmu = dlp_dsg = torch.zeros(S, F, dtype=dtype)
        ent = 0.0
        dent = torch.zeros_like(sgf)
    elif prior is None or prior.get("weights") is None:                                           # tied: log N(w; mu, sg) = -eps^2/2 - log sg - c
        lp = (-0.5 * e2 * e2 - torch.log(sgf) - c).sum(1)
        dlp_dmu = torch.zeros(S, F, dtype=dtype)
        dlp_dsg = (-1.0 / sgf).expand(S, -1)
        ent = (0.5 + c + torch.log(sgf)).sum()
        dent = 1.0 / sgf
    else:
        a = torch.as_tensor(np.broadcast_to(np.asarray(prior["weights"][0], dtype=np.float64), tuple(mu.shape)).copy()).to(dtype).reshape(-1)
        b = torch.as_tensor(np.broadcast_to(np.asarray(prior["weights"][1], dtype=np.float64), tuple(mu.shape)).copy()).to(dtype).reshape(-1)
        d = w - a
        lp = (-0.5 * d * d / (b * b) - torch.log(b) - c).sum(1)
        g = -d / (b * b)
        dlp_dmu, dlp_dsg = g, g * e2
        ent = (0.5 + c + torch.log(sgf)).sum()
        dent = 1.0 / sgf
    elbo_s = ll + lp
    dE_dmu = (gw + dlp_dmu).mean(0)
    dE_dsg = (gw * e2 + dlp_dsg).mean(0) + dent
    grads = {"weights_loc": (-dE_dmu).reshape(tuple(mu.shape)).numpy(),
             "weights_scale": (-dE_dsg * torch.sigmoid(rhof)).reshape(tuple(mu.shape)).numpy()}
    if noise == "lognormal":
        gu = R * inv_s2 - N                                         # d ll_s / d u_s
        gm, gs = gu, gu * en
        ent_nu = 0.0
        if with_prior:
            if prior is not None and "nu" in prior:
                pa, pb = float(np.asarray(prior["nu"][0]).reshape(-1)[0]), float(np.asarray(prior["nu"][1]).reshape(-1)[0])
                dd = u - pa
                lpn = -0.5 * dd * dd / pb ** 2 - math.log(pb) - c - u
                gpu = -dd / pb ** 2 - 1.0
                gm, gs = gm + gpu, gs + gpu * en
            else:                                                   # a = m, b = sgn: the eps-dependent parts cancel
                lpn = -0.5 * en * en - torch.log(sgn) - c - u
                gm, gs = gm - 1.0, gs - 1.0 / sgn - en
            elbo_s = elbo_s + lpn
            ent_nu = 0.5 + c + torch.log(sgn) + m
            gm, gs = gm + 1.0, gs + 1.0 / sgn
        ent = ent + ent_nu
        grads["nu_loc"] = np.asarray(float(-gm.mean()))
        grads["nu_scale"] = np.asarray(float(-gs.mean() * torch.sigmoid(rn)))
    loss = -(elbo_s.mean() + ent)
    return float(loss), grads
