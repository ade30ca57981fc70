"""TEST INFRASTRUCTURE ONLY: the oracle of robust Bayesian linear regression (K2g with a Cauchy or Laplace likelihood), in the
conventions of tests/linreg_oracle.py -- `loss = -ELBO` as a python float and gradients keyed by the reference's parameter
names.  `robreg_elbo` restates the objective with torch.distributions and autograd; `robreg_elbo_streamed` is the fp64
row-streamed version with the gradient written out by hand, pinned against it in tests/test_robreg_lowering.py.  The prior and
entropy terms of the weights and of the LogNormal noise latent are those of the Normal likelihood (linreg_oracle.py)."""
import math

import numpy as np
import torch
import torch.distributions as D
import torch.nn.functional as F

from oracle.elbo_oracle import MeanFieldNormal, F_softplus, _t

LIKELIHOODS = {"cauchy": D.Cauchy, "laplace": D.Laplace}

# Laplace kink margin: a residual within KINK_REL * (|y_b| + sum_f |w_sf x_bf|) of zero may take the opposite sign in the
# kernel, whose logits carry a relative error of about 1e-6 (2^-20) of sum_f |w_sf x_bf| (3xFP16 operands): 2^-18 is 4x that.
KINK_REL = 2.0 ** -18


def robreg_elbo(X, y, params, eps, prior=None, noise="lognormal", likelihood="cauchy", dtype=torch.float32, with_prior=True):
    """y_b ~ Cauchy / Laplace(BF.matmul(weights, x)_b, sigma) over N observed rows (summed), weights [1, F] mean-field Normal;
    noise, prior and with_prior as in linreg_oracle.linreg_elbo."""
    wprior = {"weights": prior["weights"]} if prior is not None and prior.get("weights") is not None else None
    q = MeanFieldNormal({"weights": params["weights"]}, {"weights": eps["weights"]}, wprior, dtype)
    w = q.sample()["weights"]                       # [S,1,F]
    S = q.S
    loc = torch.einsum("scf,bf->sb", w, _t(X, dtype))
    yt = _t(y, dtype).reshape(-1)
    if noise == "lognormal":
        m = _t(params["nu"][0], dtype, True)
        rho = _t(params["nu"][1], dtype, True)
        sg = F.softplus(rho).reshape(())
        nu = torch.exp(m.reshape(()) + _t(eps["nu"], dtype).reshape(S) * sg)
        sigma = nu[:, None]
    else:
        sigma = torch.tensor(float(noise), dtype=dtype)
    per_sample = LIKELIHOODS[likelihood](loc, sigma).log_prob(yt[None, :]).sum(dim=1)
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


def robreg_elbo_streamed(X, y, params, eps, prior=None, noise="lognormal", likelihood="cauchy", dtype=torch.float64,
                         row_chunk=65536, with_prior=True, kink=False):
    """`robreg_elbo` with the rows streamed and the gradient written out by hand.  Per sample, with r_sb = y_b - w_s . x_b,
    z = r / sigma_s and u_s = log sigma_s:
        Cauchy   ll_s = -N (log pi + u_s) - Lam_s,   d ll_s / d w_s = (2 / sigma_s) G_s,   d ll_s / d u_s = 2 T_s - N
                 Lam_s = sum_b log1p(z^2), T_s = sum_b z^2 / (1 + z^2), G_s = sum_b z / (1 + z^2) x_b
        Laplace  ll_s = -N (log 2 + u_s) - A_s / sigma_s,   d ll_s / d w_s = G_s / sigma_s,   d ll_s / d u_s = A_s / sigma_s - N
                 A_s = sum_b |r|, G_s = sum_b sign(r) x_b (sign(0) = 0)
    kink=True (Laplace) also returns a third value: {"weights_loc", "weights_scale": per-element bounds of what the residuals
    with |r_sb| <= KINK_REL (|y_b| + sum_f |w_sf x_bf|) contribute to those gradients if their sign flips, "count": their
    number}."""
    mu, rho = (_t(a, dtype) for a in params["weights"])
    e = _t(eps["weights"], dtype)                                   # [S, 1, F]
    S, Fn = e.shape[0], e.shape[-1]
    sg = F_softplus(rho)
    w = (mu + sg * e).reshape(S, Fn)
    Xt = torch.as_tensor(np.asarray(X))
    yt = torch.as_tensor(np.asarray(y)).reshape(-1)
    N = Xt.shape[0]
    c = 0.5 * math.log(2 * math.pi)
    if noise == "lognormal":
        m, rn = (_t(a, dtype).reshape(()) for a in params["nu"])
        sgn = F_softplus(rn)
        en = _t(eps["nu"], dtype).reshape(S)
        u = m + sgn * en
    else:
        u = torch.full((S,), math.log(float(noise)), dtype=dtype)
    sigma = torch.exp(u)
    P = torch.zeros(S, dtype=dtype)                                 # Lam_s or A_s
    T = torch.zeros(S, dtype=dtype)
    G = torch.zeros(S, Fn, dtype=dtype)
    kb = torch.zeros(S, Fn, dtype=dtype)                            # sum over the kink set of |x_b| / sigma_s, per sample
    count = 0
    with torch.no_grad():
        for r0 in range(0, N, row_chunk):
            xb = Xt[r0:r0 + row_chunk].to(dtype)
            yb = yt[r0:r0 + row_chunk].to(dtype)
            rb = yb[None, :] - w @ xb.T                             # [S, rows]
            if likelihood == "cauchy":
                z = rb / sigma[:, None]
                zz = z * z
                P += torch.log1p(zz).sum(1)
                T += (zz / (1 + zz)).sum(1)
                G += (z / (1 + zz)) @ xb
            else:
                P += rb.abs().sum(1)
                G += torch.sign(rb) @ xb
                if kink:
                    K = rb.abs() <= KINK_REL * (yb.abs()[None, :] + w.abs() @ xb.abs().T)
                    count += int(K.sum())
                    kb += (K.to(dtype) / sigma[:, None]) @ xb.abs()
    if likelihood == "cauchy":
        ll = -N * (math.log(math.pi) + u) - P
        gw = (2.0 / sigma)[:, None] * G
        gu = 2.0 * T - N
    else:
        ll = -N * (math.log(2.0) + u) - P / sigma
        gw = G / sigma[:, None]
        gu = P / sigma - N
    e2 = e.reshape(S, -1)
    muf, sgf, rhof = mu.reshape(-1), sg.reshape(-1), rho.reshape(-1)
    if not with_prior:
        lp = torch.zeros(S, dtype=dtype)
        dlp_dmu = dlp_dsg = torch.zeros(S, Fn, dtype=dtype)
        ent = 0.0
        dent = torch.zeros_like(sgf)
    elif prior is None or prior.get("weights") is None:             # tied: log N(w; mu, sg) = -eps^2/2 - log sg - c
        lp = (-0.5 * e2 * e2 - torch.log(sgf) - c).sum(1)
        dlp_dmu = torch.zeros(S, Fn, dtype=dtype)
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
    loss = float(-(elbo_s.mean() + ent))
    if not kink:
        return loss, grads
    bound = {"weights_loc": (2.0 * kb.sum(0) / S).reshape(tuple(mu.shape)).numpy(),
             "weights_scale": (2.0 * (kb * e2.abs()).sum(0) / S * torch.sigmoid(rhof)).reshape(tuple(mu.shape)).numpy(),
             "count": count}
    return loss, grads, bound
