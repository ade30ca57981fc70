"""TEST INFRASTRUCTURE ONLY: the oracle of regression particles (K4a / K6b with a Normal, Cauchy or Laplace likelihood over
BF.matmul(weights, x) at a fixed noise scale sigma).  Per particle theta_k [1, F], ll_k = sum_b log p(y_b | theta_k . x_b, sigma)
with torch.distributions' log_prob, and the particle loss is a SUM over the particles (SteinVariationalGradientDescent.compute_loss,
inference.py:292-299; MAP, inference.py:251-274):
    loss = sum_k [ -ll_k - sum_f log N(theta_kf; prior_loc, prior_scale) ]      G = d loss / d theta
`particles_loss_grad` restates it with autograd; `particles_loss_grad_streamed` is the fp64 row-streamed version with the
gradient written out by hand, pinned against it in tests/test_regparticles_lowering.py.  `wvgd_loss` / `wvgd_ensemble_weights`
restate oracle.elbo_oracle's WVGD objectives, whose log-likelihoods are the logistic ones, for any log-likelihood closure; with the
logistic closure they are pinned against the originals in tests/test_regparticles_lowering.py."""
import math

import numpy as np
import torch
import torch.distributions as D
import torch.nn.functional as F

from oracle.elbo_oracle import _t, voronoi_owner
from robreg_oracle import KINK_REL

LIKELIHOODS = {"normal": D.Normal, "cauchy": D.Cauchy, "laplace": D.Laplace}


def loglik(X, y, sigma, likelihood, dtype=torch.float64):
    """z [S, 1, F] weight vectors -> ll [S], summed over the rows"""
    Xt, yt = _t(X, dtype), _t(y, dtype).reshape(-1)
    dist = LIKELIHOODS[likelihood]
    return lambda z: dist(torch.einsum("scf,bf->sb", z, Xt), torch.tensor(float(sigma), dtype=dtype)).log_prob(yt[None, :]).sum(1)


def particles_loss_grad(X, y, theta, sigma, likelihood, prior=None, dtype=torch.float32):
    """theta [n, 1, F]; prior = (loc, scale) broadcastable to [1, F] or None.  Returns (loss, G [n, 1, F])."""
    th = _t(theta, dtype, requires_grad=True)
    loss = -loglik(X, y, sigma, likelihood, dtype)(th).sum() if len(X) else (th * 0).sum()
    if prior is not None:
        loss = loss - D.Normal(_t(prior[0], dtype), _t(prior[1], dtype)).log_prob(th).sum()
    loss.backward()
    return float(loss.detach()), th.grad.detach().numpy().copy()


def vectors_loglik_grad(X, y, V, sigma, likelihood, dtype=torch.float32):
    """V [n, 1, F] -> (ll [n], G [n, 1, F] = -d ll / d V), autograd"""
    v = _t(V, dtype, requires_grad=True)
    ll = loglik(X, y, sigma, likelihood, dtype)(v)
    (-ll.sum()).backward()
    return ll.detach().numpy().copy(), v.grad.detach().numpy().copy()


def particles_loss_grad_streamed(X, y, theta, sigma, likelihood, prior=None, dtype=torch.float64, row_chunk=16384, kink=False):
    """`particles_loss_grad` with the rows streamed and the gradient written out by hand, r_kb = y_b - theta_k . x_b, z = r / sigma:
        Normal   ll_k = -sum r^2 / (2 sigma^2) - N log sigma - N/2 log(2 pi)   d ll_k / d theta_k = sum r x / sigma^2
        Cauchy   ll_k = -N (log pi + log sigma) - sum log1p(z^2)            d ll_k / d theta_k = (2 / sigma) sum z / (1 + z^2) x
        Laplace  ll_k = -N (log 2 + log sigma) - sum |r| / sigma            d ll_k / d theta_k = sum sign(r) x / sigma
    kink=True (Laplace) also returns a third value: {"G": [n, 1, F] bound of what the residuals with
    |r_kb| <= KINK_REL (|y_b| + sum_f |theta_kf x_bf|) contribute to G if their sign flips, sum 2 |x_bf| / sigma over them,
    "count": their number} -- the rule of robreg_oracle without the 1/S factor."""
    th = _t(theta, dtype).reshape(np.asarray(theta).shape[0], -1)     # [n, F]
    Xt = torch.as_tensor(np.asarray(X))
    yt = torch.as_tensor(np.asarray(y)).reshape(-1)
    N = Xt.shape[0]
    sd = float(sigma)
    P = torch.zeros(th.shape[0], dtype=dtype)
    G = torch.zeros_like(th)
    kb = torch.zeros_like(th)
    count = 0
    with torch.no_grad():
        for r0 in range(0, N, row_chunk):
            xb = Xt[r0:r0 + row_chunk].to(dtype)
            yb = yt[r0:r0 + row_chunk].to(dtype)
            rb = yb[None, :] - th @ xb.T
            if likelihood == "normal":
                P += (rb * rb).sum(1)
                G += rb @ xb
            elif likelihood == "cauchy":
                z = rb / sd
                zz = z * z
                P += torch.log1p(zz).sum(1)
                G += (z / (1 + zz)) @ xb
            else:
                P += rb.abs().sum(1)
                G += torch.sign(rb) @ xb
                if kink:
                    K = rb.abs() <= KINK_REL * (yb.abs()[None, :] + th.abs() @ xb.abs().T)
                    count += int(K.sum())
                    kb += K.to(dtype) @ xb.abs()
        if likelihood == "normal":
            ll = -P / (2 * sd * sd) - N * (math.log(sd) + 0.5 * math.log(2 * math.pi))
            gll = G / (sd * sd)
        elif likelihood == "cauchy":
            ll = -N * (math.log(math.pi) + math.log(sd)) - P
            gll = (2.0 / sd) * G
        else:
            ll = -N * (math.log(2.0) + math.log(sd)) - P / sd
            gll = G / sd
        loss = -ll.sum()
        Gl = -gll
        if prior is not None:
            a = torch.as_tensor(np.broadcast_to(np.asarray(prior[0], np.float64), (1, th.shape[1])).copy()).to(dtype).reshape(-1)
            b = torch.as_tensor(np.broadcast_to(np.asarray(prior[1], np.float64), (1, th.shape[1])).copy()).to(dtype).reshape(-1)
            d = th - a
            loss = loss - (-0.5 * d * d / (b * b) - torch.log(b) - 0.5 * math.log(2 * math.pi)).sum()
            Gl = Gl + d / (b * b)
    shape = np.asarray(theta).shape
    out = (float(loss), Gl.numpy().reshape(shape))
    if not kink:
        return out
    return out + ({"G": (2.0 * kb / sd).numpy().reshape(shape), "count": count},)


def wvgd_loss(ll_fn, theta, loc, rho, eps_elbo, eps_particle, prior=None, dtype=torch.float32, biased=False, first_column_only=True):
    """oracle.elbo_oracle.wvgd_loss (same objective and return values; see its docstring) with the log-likelihood a closure
    ll_fn(z [S, C, F]) -> [S] in `dtype` (`loglik` for regression) instead of (X, y, likelihood)."""
    n = len(theta)
    th, lc, rh = _t(theta, dtype, True), _t(loc, dtype, True), _t(rho, dtype, True)
    e1, e2 = _t(eps_elbo, dtype), _t(eps_particle, dtype)
    total = 0.0
    counts = np.zeros((n, 2), np.int64)
    for k in range(n):
        sg = F.softplus(rh[k])
        q = D.Normal(lc[k], sg.expand_as(lc[k]))
        pr = q if prior is None else D.Normal(_t(prior[0], dtype), _t(prior[1], dtype))
        z = lc[k] + sg * e1[k]
        acc = torch.as_tensor(voronoi_owner(z.detach().float().numpy(), th.detach().float().numpy(), first_column_only) == k)
        counts[k, 0] = int(acc.sum())
        za = z[acc]
        logq = q.log_prob(za).sum((1, 2))
        norm = -q.log_prob(za.detach()).sum((1, 2)).mean().detach()
        elbo = (ll_fn(za) + pr.log_prob(za).sum((1, 2)) - (logq + norm)).mean()
        z2 = (lc[k] + sg * e2[k]).detach()
        acc2 = torch.as_tensor(voronoi_owner(z2.float().numpy(), th.detach().float().numpy(), first_column_only) == k)
        counts[k, 1] = int(acc2.sum())
        z2a = z2[acc2]
        if biased:
            w = torch.full((z2a.shape[0],), 1.0 / eps_particle.shape[1], dtype=dtype)
        else:
            w = torch.softmax((ll_fn(z2a) + pr.log_prob(z2a).sum((1, 2)) - q.log_prob(z2a).sum((1, 2))).detach(), 0)
        total = total - elbo + (w * ((th[k][None] - z2a) ** 2).sum((1, 2))).sum()
    total.backward()
    return float(total.detach()), {"loc": lc.grad.numpy().copy(), "rho": rh.grad.numpy().copy(), "theta": th.grad.numpy().copy()}, counts


def wvgd_ensemble_weights(ll_fn, theta, loc, rho, eps, prior=None, dtype=torch.float64, first_column_only=True):
    """oracle.elbo_oracle.wvgd_ensemble_weights with the log-likelihood a closure, as for `wvgd_loss`.
    Returns (weights [n], logZ [n], counts [n])."""
    n = len(theta)
    logZ, counts = np.zeros(n), np.zeros(n, np.int64)
    with torch.no_grad():
        for k in range(n):
            lc = _t(loc[k], dtype)
            sg = F.softplus(_t(rho[k], dtype))
            q = D.Normal(lc, sg.expand_as(lc))
            pr = q if prior is None else D.Normal(_t(prior[0], dtype), _t(prior[1], dtype))
            z = lc + sg * _t(eps[k], dtype)
            acc = torch.as_tensor(voronoi_owner(z.float().numpy(), np.asarray(theta, np.float32), first_column_only) == k)
            counts[k] = int(acc.sum())
            za = z[acc]
            logw = ll_fn(za) + pr.log_prob(za).sum((1, 2)) - q.log_prob(za).sum((1, 2))
            logZ[k] = float(torch.logsumexp(logw, 0)) if counts[k] else -np.inf
    w = np.exp(logZ - logZ.max())
    return w / w.sum(), logZ, counts
