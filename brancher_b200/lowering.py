"""Graph matcher: lowers a (joint model, posterior model) pair to a fused CUDA kernel family.

The reference evaluates the ELBO by walking the model graph in Python, one torch op at a time
(variables.py:843-870, 486-570).  Here the pair is inspected ONCE: its expression trees are
pattern-matched against the kernel families of include/brancher_cuda.h and a `Plan` is cached on the
joint model.  `Plan.elbo(S, empirical_samples)` then runs one fused forward+backward evaluation and
returns a 0-d tensor wired into autograd (so `loss.backward()` fills `.grad` of every learnable
`ParameterModule.parameter`, the contract of optimizers.py:34-51).

Families
  LinearPlan  K2  observed Binomial(1)/Bernoulli/Categorical with logits = BF.matmul(W, x), W mean-field Normal
  LinregPlan  K2g observed Normal / Cauchy / Laplace(BF.matmul(W, x), sigma), W [1, F] mean-field Normal, sigma constant or a
              LogNormal latent
  BNNPlan     K3  observed Categorical with logits = BF.matmul(W_out, h_L) + b_out, h_l = act_l(BF.matmul(W_l, h_{l-1}) + b_l),
              h_0 = x, act_l in {BF.tanh, BF.relu, BF.sigmoid}: one hidden layer (brn_bnn_*, any width) or 2..4 hidden layers
              of width <= 128 (brn_bnn_deep_*); every weight and bias a mean-field Normal latent
  ParticlePlan / WvgdPlan  K4 / K6  particle ensembles (SVGD, MAP, WVGD) of the K2 graph, or of the K2g graph at a constant
              noise scale
Unrecognised graphs raise `UnsupportedModelError` -- there is no eager / CPU fallback for the ELBO.
"""
import contextlib

import numpy as np
import torch

from brancher_b200 import config, distributed
from brancher_b200.variables import (RootVariable, RandomVariable, VarRef, Const, Call, evaluate)


class UnsupportedModelError(NotImplementedError):
    pass


# ---------------------------------------------------------------------------------------------------
# noise injection (parity testing): {q variable name: tensor (S, *event)} of standard normals
# ---------------------------------------------------------------------------------------------------
_INJECTED = None


@contextlib.contextmanager
def inject_noise(eps_by_name):
    """Within the context every fused evaluation uses the given standard-normal draws instead of Philox
    (the counterpart of overriding `Qvar.distribution._get_sample` in the reference, SURVEY §8c)."""
    global _INJECTED
    prev, _INJECTED = _INJECTED, dict(eps_by_name)
    try:
        yield
    finally:
        _INJECTED = prev


# ---------------------------------------------------------------------------------------------------
# expression pattern helpers
# ---------------------------------------------------------------------------------------------------
def _is_call(e, name, nargs=None):
    return isinstance(e, Call) and e.name == name and (nargs is None or len(e.args) == nargs) and not e.kwargs


def _const_value(e):
    if isinstance(e, Const) and isinstance(e.value, (int, float)):
        return float(e.value)
    return None


def _strip_zero_add(e):
    """x + 0.0 / 0.0 + x -> x   (RightHalfLine(0.).forward_transform writes `0. + softplus(x)`)."""
    if _is_call(e, "add", 2):
        a, b = e.args
        if _const_value(b) == 0.0:
            return a
        if _const_value(a) == 0.0:
            return b
    return e


def _as_root(e):
    return e.var if isinstance(e, VarRef) and isinstance(e.var, RootVariable) else None


def _softplus_root(e):
    e = _strip_zero_add(e)
    if _is_call(e, "softplus", 1):
        return _as_root(e.args[0])
    return None


def _commutative_add(e):
    if _is_call(e, "add", 2):
        a, b = e.args
        return [(a, b), (b, a)]
    return []


def _var(e):
    return e.var if isinstance(e, VarRef) else None


# ---------------------------------------------------------------------------------------------------
class MeanFieldSpec:
    """One latent: q = Normal(root_loc, softplus(root_scale)) (learnable roots) and p = Normal prior of the
    same name, tied by root-name collision or declared."""
    kind, kind_name = "normal", "Normal"

    def __init__(self, name, q_var, p_var, q_names):
        self.name = name
        if not isinstance(q_var, RandomVariable):          # MAP's point estimate reaches here when its particle lowering fails
            raise UnsupportedModelError("latent %r: q is a point estimate (a root), not a %s variable" % (name, self.kind_name))
        lq = q_var.partial_links
        if q_var.distribution.kind != self.kind or p_var.distribution.kind != self.kind:
            raise UnsupportedModelError("latent %r: only %s q / %s prior are lowered to the mean-field kernels"
                                        % (name, self.kind_name, self.kind_name))
        self.loc_root = _as_root(lq["loc"].expr)
        self.scale_root = _softplus_root(lq["scale"].expr)
        if self.loc_root is None or self.scale_root is None:
            raise UnsupportedModelError("latent %r: q's loc/scale must be (learnable) roots" % name)
        self.shape = tuple(self.loc_root._value.shape[2:])
        if self.scale_root._value.numel() != self.loc_root._value.numel():
            raise UnsupportedModelError("latent %r: q's scale has %d elements, its loc %d -- the mean-field kernels need one "
                                        "scale per element (pass a scale array of the variable's shape)"
                                        % (name, self.scale_root._value.numel(), self.loc_root._value.numel()))
        lp = p_var.partial_links
        p_loc_root, p_scale_sp = _as_root(lp["loc"].expr), _softplus_root(lp["scale"].expr)
        p_scale_raw = _as_root(lp["scale"].expr)
        p_scale_root = p_scale_sp or p_scale_raw
        if p_loc_root is None or p_scale_root is None:
            raise UnsupportedModelError("latent %r: the prior's loc/scale must be constants" % name)
        tied_loc = p_loc_root.name in q_names
        tied_scale = p_scale_root.name in q_names
        if tied_loc != tied_scale:
            raise UnsupportedModelError("latent %r: prior loc/scale roots are tied to q inconsistently" % name)
        if tied_loc and not (p_loc_root.name == self.loc_root.name and p_scale_root.name == self.scale_root.name
                             and p_scale_sp is not None):
            raise UnsupportedModelError("latent %r: unexpected root-name collision pattern" % name)
        self.tied = tied_loc
        self._p_loc_root, self._p_scale_root, self._p_scale_softplus = p_loc_root, p_scale_root, p_scale_sp is not None
        if not self.tied and (getattr(p_loc_root, "learnable", False) or getattr(p_scale_root, "learnable", False)):
            # ReverseKL optimises the joint model's learnable parameters too (learnable_model = True); the fused kernels
            # return no gradient for a prior's own hyper-parameters, so training them silently would freeze them
            raise UnsupportedModelError("latent %r: learnable hyper-parameters of an untied prior are not lowered" % name)

    # the declared prior is read at EVALUATION time (a constant root may be re-assigned between evaluations)
    @property
    def prior_loc(self):
        return None if self.tied else self._p_loc_root.value.detach()

    @property
    def prior_scale(self):
        if self.tied:
            return None
        sc = self._p_scale_root.value.detach()
        return torch.nn.functional.softplus(sc) if self._p_scale_softplus else sc

    def parameters(self):
        return [self.loc_root.value, self.scale_root.value]

    def make(self, cu, var_id, eps, sinks=(None, None)):
        mu, rho = self.loc_root.value, self.scale_root.value
        if not self.tied:
            pl = self.prior_loc.expand(mu.shape).reshape(-1).contiguous()
            ps = self.prior_scale.expand(mu.shape).reshape(-1).contiguous()
        else:
            pl = ps = None
        return cu.MeanFieldVar(mu, rho, var_id=var_id, prior_loc=pl, prior_scale=ps, eps=eps, dmu=sinks[0], drho=sinks[1])


class LogNormalSpec(MeanFieldSpec):
    """A scalar latent with q = LogNormal(root_loc, softplus(root_scale)) and a LogNormal prior of the same name, tied or
    declared: the noise scale of the linear-regression family (brn_mf_var read as a LogNormal, Philox var_id 1)."""
    kind, kind_name = "lognormal", "LogNormal"

    def __init__(self, name, q_var, p_var, q_names):
        super().__init__(name, q_var, p_var, q_names)
        if int(np.prod(self.shape)) != 1:
            raise UnsupportedModelError("latent %r: the LogNormal noise scale must be a scalar (shape %s)" % (name, self.shape))


class _FusedELBO(torch.autograd.Function):
    """autograd node of one fused evaluation: forward runs the kernels (loss and all gradients at once),
    backward hands the stored gradients out."""

    @staticmethod
    def forward(ctx, runner, *params):
        loss, grads = runner()
        ctx.grads = grads
        return (-loss).to(torch.float32).reshape(())          # the reference's estimator returns +ELBO

    @staticmethod
    def backward(ctx, g):
        return (None,) + tuple((-g) * gr if gr is not None else None for gr in ctx.grads)


class Plan:
    family = "?"

    def __init__(self, joint, posterior):
        self.joint, self.posterior = joint, posterior
        self.latents = []        # MeanFieldSpec in kernel order

    def _eps(self, S_local, s0):
        out = []
        for spec in self.latents:
            if _INJECTED is None:
                out.append(None)
                continue
            if spec.name not in _INJECTED:
                raise KeyError("inject_noise: no noise given for q variable %r" % spec.name)
            e = torch.as_tensor(_INJECTED[spec.name], dtype=torch.float32, device=config.device)
            e = e.reshape(e.shape[0], -1)
            out.append(e[s0:s0 + S_local].contiguous())
        return out

    def elbo(self, number_samples, empirical_samples):
        if config.device.type != "cuda":
            raise RuntimeError("brancher_b200 evaluates the ELBO only on CUDA devices (no CPU fallback); "
                               "config.device is %s" % config.device)
        from brancher_b200 import _cuda as cu
        cu.lib()
        s0, S_local = distributed.shard(number_samples)
        r = cu.sample_range(number_samples, s0=s0, s_local=S_local, seed=config.seed, offset=config.next_offset())
        params = [p for spec in self.latents for p in spec.parameters()]

        def runner():
            flat, sinks = cu.flat_grad_views([int(np.prod(spec.shape)) for spec in self.latents], config.device)
            mvars = [spec.make(cu, i, eps, sk) for i, (spec, eps, sk) in enumerate(zip(self.latents, self._eps(S_local, s0), sinks))]
            loss = self._launch(cu, mvars, r, empirical_samples)
            if distributed.world_size() > 1:
                # ONE collective on the flat buffer the kernels accumulated into; the fp64 loss rides in its spare tail as a
                # (hi, lo) fp32 pair
                distributed.all_reduce_flat(flat, loss)
            grads = []
            for spec, v in zip(self.latents, mvars):
                grads += [v.dmu.reshape(spec.loc_root.value.shape), v.drho.reshape(spec.scale_root.value.shape)]
            return loss, [g if p.requires_grad else None for g, p in zip(grads, params)]

        return _FusedELBO.apply(runner, *params)

    def static_evaluation(self, number_samples, empirical_samples, offset_dev):
        """One evaluation as a replayable launch sequence over PERSISTENT buffers (what a CUDA graph captures): returns an
        object with `.params` (the learnable leaf tensors), `.grads` (views of one flat buffer, aligned with params),
        `.loss` (fp64 [1]) and `.launch()`.  The Philox offset of replay i is base + offset_dev[0] (read on the device)."""
        from types import SimpleNamespace
        from brancher_b200 import _cuda as cu
        cu.lib()
        if distributed.world_size() != 1 or _INJECTED is not None:
            return None
        r = cu.sample_range(number_samples, seed=config.seed, offset=config.next_offset(), offset_dev=offset_dev)
        flat, sinks = cu.flat_grad_views([int(np.prod(spec.shape)) for spec in self.latents], config.device)
        loss = torch.zeros(1, dtype=torch.float64, device=config.device)
        mvars = [spec.make(cu, i, None, sk) for i, (spec, sk) in enumerate(zip(self.latents, sinks))]
        params, grads = [], []
        for spec, v in zip(self.latents, mvars):
            params += [spec.loc_root.value, spec.scale_root.value]
            grads += [v.dmu, v.drho]

        def launch():
            flat.zero_()
            loss.zero_()
            self._launch(cu, mvars, r, empirical_samples, loss=loss)

        return SimpleNamespace(params=params, grads=grads, loss=loss, launch=launch)

    def _launch(self, cu, mvars, r, empirical_samples, loss=None):
        raise NotImplementedError


def _data_matrix(t, what):
    """(1, B, P, 1) / (1, B, P) observed tensor -> [B, P] fp32 contiguous."""
    if not torch.is_tensor(t) or t.shape[0] != 1:
        raise UnsupportedModelError("%s: expected an observed tensor with a singleton sample axis" % what)
    return t.reshape(t.shape[1], -1).to(torch.float32).contiguous()


class LinearPlan(Plan):
    family = "linear (K2)"

    def __init__(self, joint, posterior, k, w_spec, x_var, likelihood, C):
        super().__init__(joint, posterior)
        self.k, self.x_var, self.likelihood, self.C = k, x_var, likelihood, C
        self.latents = [w_spec]
        self._prepared_x = None      # fp16-pair form of a fixed observed matrix, rebuilt when the matrix changes

    def _launch(self, cu, mvars, r, empirical, loss=None):
        X = _data_matrix(empirical[self.x_var], "x")
        if self._prepared_x is None:
            self._prepared_x = cu.PreparedX()
        yv = empirical[self.k].reshape(-1)
        if self.likelihood == cu.BERNOULLI:
            y = yv.to(torch.float32).contiguous()
        else:
            y = yv.to(torch.int32).contiguous()
        return cu.linear_elbo_fwd_bwd(X, y, self.likelihood, mvars[0], self.C, r, loss=loss, prepared=self._prepared_x)


class LinregPlan(Plan):
    family = "linear regression (K2g)"

    def __init__(self, joint, posterior, k, w_spec, x_var, nu_spec=None, scale=None, likelihood=None):
        """scale: (root, softplus) of a constant noise scale, or a number; None when nu_spec is given.
        likelihood: cu.GAUSSIAN (None), cu.CAUCHY or cu.LAPLACE"""
        super().__init__(joint, posterior)
        from brancher_b200 import _cuda as cu
        self.likelihood = cu.GAUSSIAN if likelihood is None else likelihood
        if self.likelihood != cu.GAUSSIAN:
            self.family = "linear regression (K2g, %s likelihood)" % {cu.CAUCHY: "Cauchy", cu.LAPLACE: "Laplace"}[self.likelihood]
        self.k, self.x_var = k, x_var
        self.latents = [w_spec] + ([nu_spec] if nu_spec is not None else [])
        self._scale = scale
        self._prepared_x = None

    def noise_scale(self):
        return _noise_scale_tensor(self._scale)

    def _launch(self, cu, mvars, r, empirical, loss=None):
        X = _data_matrix(empirical[self.x_var], "x")
        if self._prepared_x is None:
            self._prepared_x = cu.PreparedX()
        y = empirical[self.k].reshape(-1).to(torch.float32).contiguous()
        nu = mvars[1] if len(mvars) > 1 else None
        return cu.linreg_elbo_fwd_bwd(X, y, mvars[0], r, nu=nu, noise_scale=None if nu is not None else self.noise_scale(),
                                      loss=loss, prepared=self._prepared_x, likelihood=self.likelihood)


class BNNPlan(Plan):
    family = "bnn (K3)"

    def __init__(self, joint, posterior, k, layers, x_var):
        """layers: [(weights spec, bias spec, activation of the layer's output)] from the input layer outward; the last one is
        the output layer (activation None).  Two layers (one hidden) run on brn_bnn_*, more on brn_bnn_deep_*."""
        super().__init__(joint, posterior)
        self.k, self.x_var, self.layers = k, x_var, layers
        self.latents = [spec for W, b, _ in layers for spec in (W, b)]          # weights1, b1, weights2, b2, ...
        self.activations = [act for _, _, act in layers[:-1]]
        if len(self.activations) > 1:
            self.family = "bnn (K3, %d hidden layers)" % len(self.activations)

    def _launch(self, cu, mvars, r, empirical, loss=None):
        X = _data_matrix(empirical[self.x_var], "x")
        y = empirical[self.k].reshape(-1).to(torch.int32).contiguous()
        if len(self.activations) == 1:
            return cu.bnn_elbo_fwd_bwd(X, y, mvars, r, loss=loss, activation=self.activations[0])
        return cu.bnn_deep_elbo_fwd_bwd(X, y, mvars, r, self.activations, loss=loss)

    def predict(self, X, number_samples):
        """Batched posterior-predictive pass (SURVEY 8(f)3; replaces the per-image loop around
        ProbabilisticModel._get_posterior_sample, variables.py:796-812): X [B, P] -> dict(logits [S, B, C],
        samples int32 [S, B] ~ Categorical(logits), probs [B, C] = MC mean of softmax(logits))."""
        if config.device.type != "cuda":
            raise RuntimeError("brancher_b200 evaluates the posterior predictive only on CUDA devices (no CPU fallback)")
        from brancher_b200 import _cuda as cu
        cu.lib()
        X = torch.as_tensor(X, dtype=torch.float32, device=config.device)
        X = X.reshape(-1, int(np.prod(self.latents[0].shape[1:]))).contiguous()
        r = cu.sample_range(number_samples, seed=config.seed, offset=config.next_offset())
        mvars = [spec.make(cu, i, None) for i, spec in enumerate(self.latents)]
        if len(self.activations) == 1:
            logits, labels, probs = cu.bnn_predict(X, mvars, r, activation=self.activations[0])
        else:
            logits, labels, probs = cu.bnn_deep_predict(X, mvars, r, self.activations)
        return {"logits": logits, "samples": labels, "probs": probs, "sample_range": r}


# ---------------------------------------------------------------------------------------------------
def _latent_random_variables(model):
    return [v for v in model._flatten() if isinstance(v, RandomVariable) and not v.is_observed
            and v.distribution.kind not in ("deterministic", "empirical")]


def _observed_likelihood_nodes(model):
    return [v for v in model._flatten() if isinstance(v, RandomVariable) and v.is_observed
            and v.distribution.kind not in ("deterministic", "empirical")]


def _is_data(var):
    return var is not None and var.is_observed and (isinstance(var, RootVariable) or
                                                    var.distribution.kind in ("deterministic", "empirical"))


def _lower_dense(joint, posterior):
    from brancher_b200 import _cuda as cu
    q_names = {v.name for v in posterior._flatten()}
    q_by_name = {v.name: v for v in posterior._flatten()}
    latents = _latent_random_variables(joint)
    liks = _observed_likelihood_nodes(joint)
    for v in latents:
        if v.name not in q_by_name:
            raise UnsupportedModelError("latent variable %r has no counterpart in the posterior model" % v.name)
    if len(liks) != 1:
        raise UnsupportedModelError("fused families need exactly one observed likelihood node, found %d" % len(liks))
    k = liks[0]
    kind = k.distribution.kind
    if kind in ("normal", "cauchy", "laplace"):
        return _lower_linreg(joint, posterior, k, latents, q_by_name, q_names)
    if "logits" not in k.partial_links:
        raise UnsupportedModelError("likelihood %r: only logits= parametrisations are lowered" % k.name)
    if kind == "binomial":
        tc = _as_root(k.partial_links["total_count"].expr)
        if tc is None or float(tc.value.reshape(-1)[0]) != 1.0 or tc.value.numel() != 1:
            raise UnsupportedModelError("Binomial likelihood is lowered only for total_count=1")
    if kind not in ("binomial", "bernoulli", "categorical"):
        raise UnsupportedModelError("likelihood kind %r is not lowered" % kind)
    logits = k.partial_links["logits"].expr
    spec = lambda var: MeanFieldSpec(var.name, q_by_name[var.name], var, q_names)

    # K2: logits = matmul(W, x)
    if _is_call(logits, "matmul", 2):
        W, x = _var(logits.args[0]), _var(logits.args[1])
        if W in latents and _is_data(x) and len(latents) == 1:
            ws = spec(W)
            if len(ws.shape) != 2:
                raise UnsupportedModelError("linear family: weights must be a [C, F] matrix")
            C = ws.shape[0]
            if kind != "categorical" and C != 1:
                raise UnsupportedModelError("Binomial/Bernoulli logistic regression needs weights of shape [1, F]")
            return LinearPlan(joint, posterior, k, ws, x, cu.CATEGORICAL if kind == "categorical" else cu.BERNOULLI, C)

    # K3: logits = matmul(W_out, h_L) + b_out, h_l = act(matmul(W_l, h_{l-1}) + b_l), h_0 = x
    if kind == "categorical":
        mlp = _match_mlp(logits, latents)
        if mlp is not None and len(mlp[1]) > 1:        # one layer (no hidden layer) is softmax regression with a bias: not K3
            return _bnn_plan(joint, posterior, k, latents, spec, *mlp)
    raise UnsupportedModelError("model graph is not recognised by any fused kernel family "
                                "(linear K2, bnn K3); likelihood link: %s" % k.partial_links["logits"].string)


BNN_ACTIVATIONS = ("tanh", "relu", "sigmoid")
BNN_DEEP_MAX_HIDDEN, BNN_DEEP_MAX_WIDTH, BNN_MAX_CLASSES = 4, 128, 16


def _match_mlp(e, latents, inner=False):
    """e = matmul(W, h) + b (either order of the sum) with W, b latents and h the data or act(<the same form>): returns
    (x, layers), layers = [(W, b, activation applied to the layer's input)] from the input layer outward (None for the first),
    or None.  A latent matmul without a bias where a layer is expected raises (`inner`: e sits inside an activation)."""
    for mm, be in _commutative_add(e):
        b, W = _var(be), _var(mm.args[0]) if _is_call(mm, "matmul", 2) else None
        if not (W in latents and b in latents):
            continue
        h = mm.args[1]
        if _is_data(_var(h)):
            return _var(h), [(W, b, None)]
        act = next((a for a in BNN_ACTIVATIONS if _is_call(h, a, 1)), None)
        sub = _match_mlp(h.args[0], latents, inner=True) if act is not None else None
        if sub is not None:
            return sub[0], sub[1] + [(W, b, act)]
    if _is_call(e, "matmul", 2) and _var(e.args[0]) in latents:
        h = e.args[1]
        if (inner and _is_data(_var(h))) or any(_is_call(h, a, 1) for a in BNN_ACTIVATIONS):
            raise UnsupportedModelError("bnn family: the layer BF.matmul(%s, ...) has no bias; every layer of the network needs a "
                                        "Normal bias latent (BF.matmul(W, h) + b)" % _var(e.args[0]).name)
    return None


def _bnn_plan(joint, posterior, k, latents, spec, x, layers):
    """BNNPlan of a matched network (x, layers from _match_mlp), or UnsupportedModelError with the reason."""
    n_hidden = len(layers) - 1
    variables = [v for W, b, _ in layers for v in (W, b)]
    if len(set(variables)) != len(variables):
        raise UnsupportedModelError("bnn family: a latent appears in more than one layer (%s)" % ", ".join(v.name for v in variables))
    others = [v.name for v in latents if v not in variables]
    if others:
        raise UnsupportedModelError("bnn family: latent(s) %s are neither weights nor biases of the network" % ", ".join(sorted(others)))
    if n_hidden > BNN_DEEP_MAX_HIDDEN:
        raise UnsupportedModelError("bnn family: %d hidden layers; at most %d are lowered" % (n_hidden, BNN_DEEP_MAX_HIDDEN))
    specs = [(spec(W), spec(b)) for W, b, _ in layers]
    if n_hidden > 1:
        for l, (ws, bs) in enumerate(specs):
            what = "hidden layer %d" % (l + 1) if l < n_hidden else "output layer"
            if len(ws.shape) != 2 or int(np.prod(bs.shape)) != ws.shape[0]:
                raise UnsupportedModelError("bnn family, %s: weights %s of shape %s and bias %s of shape %s do not form a layer"
                                            % (what, ws.name, ws.shape, bs.name, bs.shape))
            if l > 0 and ws.shape[1] != specs[l - 1][0].shape[0]:
                raise UnsupportedModelError("bnn family, %s: weights %s take %d inputs, the layer below has %d units"
                                            % (what, ws.name, ws.shape[1], specs[l - 1][0].shape[0]))
            if l < n_hidden and ws.shape[0] > BNN_DEEP_MAX_WIDTH:
                raise UnsupportedModelError("bnn family, %s: width %d; networks with more than one hidden layer are lowered for "
                                            "widths up to %d" % (what, ws.shape[0], BNN_DEEP_MAX_WIDTH))
        if specs[-1][0].shape[0] > BNN_MAX_CLASSES:
            raise UnsupportedModelError("bnn family: %d classes; at most %d are lowered" % (specs[-1][0].shape[0], BNN_MAX_CLASSES))
    acts = [layers[l + 1][2] for l in range(n_hidden)] + [None]
    return BNNPlan(joint, posterior, k, [(ws, bs, a) for (ws, bs), a in zip(specs, acts)], x)


REGRESSION_KINDS = {"normal": "Normal", "cauchy": "Cauchy", "laplace": "Laplace"}


def _constant_scale(scale, what, k):
    """The constant noise scale of likelihood node k: (root, softplus?) for a non-learnable scalar root (an auto-named root sits
    behind a softplus), a float for a number, None for anything else.  Shared by the mean-field and the particle regressions."""
    root, sp = _softplus_root(scale), True
    if root is None:
        root, sp = _as_root(scale), False
    if root is not None and not root.is_observed:
        if getattr(root, "learnable", False):
            raise UnsupportedModelError("%s %r: a learnable point-estimate noise scale (root %r) is not "
                                        "lowered" % (what, k.name, root.name))
        if root._value.numel() != 1:
            raise UnsupportedModelError("%s %r: the noise scale must be a scalar" % (what, k.name))
        return (root, sp)
    return _const_value(scale)


def _noise_scale_tensor(scale):
    """a constant scale of _constant_scale as a 1-element device tensor, recomputed from its root at every evaluation (a constant
    root may be re-assigned between evaluations; inside a captured graph this is one more captured kernel)"""
    if isinstance(scale, float):
        return torch.full((1,), scale, dtype=torch.float32, device=config.device)
    root, sp = scale
    v = root.value.detach().reshape(-1)[:1].to(device=config.device, dtype=torch.float32)
    return (torch.nn.functional.softplus(v) if sp else v).contiguous()


def _lower_linreg(joint, posterior, k, latents, q_by_name, q_names):
    """K2g: observed Normal / Cauchy / Laplace(loc = matmul(W, x), scale) with W the [1, F] mean-field Normal weights and x
    data; scale a non-learnable constant (a root, behind softplus when auto-named, or a number) or a scalar LogNormal latent."""
    from brancher_b200 import _cuda as cu
    kind = k.distribution.kind
    likelihood = {"normal": cu.GAUSSIAN, "cauchy": cu.CAUCHY, "laplace": cu.LAPLACE}[kind]
    lik_name = {"normal": "Normal", "cauchy": "Cauchy", "laplace": "Laplace"}[kind]
    what = "linear regression" if kind == "normal" else "%s linear regression" % lik_name
    loc, scale = k.partial_links["loc"].expr, k.partial_links["scale"].expr
    if not _is_call(loc, "matmul", 2):
        for a, b in _commutative_add(loc):
            if _is_call(a, "matmul", 2):
                raise UnsupportedModelError("%s %r: a bias added to BF.matmul(weights, x) is not lowered -- "
                                            "append a column of ones to x instead" % (what, k.name))
        raise UnsupportedModelError("likelihood %r: a %s likelihood is lowered for loc = BF.matmul(weights, x) only"
                                    % (k.name, lik_name))
    W, x = _var(loc.args[0]), _var(loc.args[1])
    if W not in latents or not _is_data(x):
        raise UnsupportedModelError("%s %r: loc must be BF.matmul(weights, x) with weights a latent and x data" % (what, k.name))
    ws = MeanFieldSpec(W.name, q_by_name[W.name], W, q_names)
    if len(ws.shape) != 2 or ws.shape[0] != 1:
        raise UnsupportedModelError("%s %r: weights must have shape [1, F] (multi-output regression is not "
                                    "lowered), got %s" % (what, k.name, ws.shape))
    nu_spec, const = None, None
    nu = _var(scale)
    if nu is not None and nu in latents:
        if nu.distribution.kind != "lognormal":
            raise UnsupportedModelError("%s %r: a %s-distributed noise scale is not lowered (a LogNormal "
                                        "latent or a constant is)" % (what, k.name, nu.distribution.kind))
        nu_spec = LogNormalSpec(nu.name, q_by_name[nu.name], nu, q_names)
    else:
        const = _constant_scale(scale, what, k)
        if const is None:
            raise UnsupportedModelError("%s %r: the noise scale must be a constant or a scalar LogNormal latent "
                                        "(deterministic or data-dependent scales are not lowered)" % (what, k.name))
    extra = [v.name for v in latents if v is not W and v is not nu]
    if extra:
        raise UnsupportedModelError("%s %r: latent variables other than the weights and the noise scale are not "
                                    "lowered: %s" % (what, k.name, sorted(extra)))
    return LinregPlan(joint, posterior, k, ws, x, nu_spec=nu_spec, scale=const, likelihood=likelihood)


# ---------------------------------------------------------------------------------------------------
# K1: scalar-DAG family
# ---------------------------------------------------------------------------------------------------
_DAG = dict(CONST=0, PARAM=1, DATA=2, EPS=3, ADD=4, SUB=5, MUL=6, DIV=7, NEG=8, POWI=9, EXP=10, LOG=11, LOG1P=12,
            SIGMOID=13, SOFTPLUS=14, TANH=15, SIN=16, COS=17, RELU=18, SQRT=19, ABS=20, CLAMP_UNIT=21, NORMAL_LP=22,
            NORMAL_ENTROPY=23, ACC_SAMPLE=24, ACC_ROW=25)             # include/brancher_cuda.h: enum brn_dag_opcode
_DAG_UNIFORM_HEADER, _DAG_LEVEL = 26, 27                                  # layout markers of the device table (not operations)
_DAG_BINARY = {"add": "ADD", "sub": "SUB", "mul": "MUL", "truediv": "DIV"}
_DAG_UNARY = {"exp": "EXP", "log": "LOG", "log1p": "LOG1P", "sigmoid": "SIGMOID", "softplus": "SOFTPLUS", "tanh": "TANH",
              "sin": "SIN", "cos": "COS", "relu": "RELU", "sqrt": "SQRT", "abs": "ABS", "neg": "NEG"}
_DAG_LOC_SCALE = ("normal", "lognormal", "logitnormal")      # kinds a q variable may have (pathwise sample from one normal draw)
_DAG_LOC_SCALE_P = _DAG_LOC_SCALE + ("cauchy", "laplace")     # kinds of the joint model's nodes (log-probability only)
DAG_MAX_SLOTS, DAG_MAX_PARAMS = 2048, 2048


class DagProgram:
    """Straight-line SSA program for brn_dag_elbo_fwd_bwd (one op = (opcode, dst, a, b, c, imm))."""

    def __init__(self):
        self.ops, self.n_slots = [], 0
        self.params, self._pidx = [], {}      # nn.Parameter (numel 1) per PARAM index
        self.columns = []                     # observed Variable per DATA column
        self.col_rows = []                    # rows of that column at lowering time (1 = broadcast)
        self.eps_names = []                   # q variable name per EPS stream
        self.rowdep = {}                      # slot -> depends on a multi-row DATA column
        self._cse = {}                        # (op, operands, imm) -> slot

    _PURE_SKIP = ("EPS", "DATA", "ACC_SAMPLE", "ACC_ROW")      # not hash-consed: streams / columns are allocated per call,
    _COMMUTATIVE = ("ADD", "MUL")                               # accumulations are side effects

    def emit(self, op, a=0, b=0, c=0, imm=0.0, rowdep=None):
        # common-subexpression elimination (the program is pure SSA): the same op on the same operands is computed once --
        # the graph walk re-derives e.g. softplus(rho) for q's sample, q's entropy and p's tied log-prob, and repeats
        # every literal.  K1 is a serial interpreter, so every op removed is latency removed (README AR(1): 556 -> fewer ops).
        if op not in self._PURE_SKIP:
            if op in self._COMMUTATIVE and b < a:
                a, b = b, a
            key = (op, a, b, c, float(np.float32(imm)))
            hit = self._cse.get(key)
            if hit is not None:
                return hit
        else:
            key = None
        dst = self.n_slots
        self.n_slots += 1
        self.ops.append((_DAG[op], dst, a, b, c, float(imm)))
        if rowdep is None:
            rowdep = any(self.rowdep.get(x, False) for x in (a, b, c)) if op not in ("CONST", "PARAM", "DATA", "EPS") else False
        self.rowdep[dst] = rowdep
        if key is not None:
            self._cse[key] = dst
        return dst

    def const(self, v):
        return self.emit("CONST", imm=float(v))

    def param(self, p):
        if p.numel() != 1:
            raise UnsupportedModelError("scalar-DAG family: learnable parameters must be scalars (got shape %s)" % (tuple(p.shape),))
        if id(p) not in self._pidx:
            self._pidx[id(p)] = len(self.params)
            self.params.append(p)
        return self.emit("PARAM", a=self._pidx[id(p)])

    def data(self, var, rows):
        self.columns.append(var)
        self.col_rows.append(rows)
        return self.emit("DATA", a=len(self.columns) - 1, rowdep=rows > 1)

    def eps(self, name):
        self.eps_names.append(name)
        return self.emit("EPS", a=len(self.eps_names) - 1)

    def device_ops(self):
        """The table the kernel walks (include/brancher_cuda.h: UNIFORM_HEADER / LEVEL markers): the sample-independent ops --
        those that depend on parameters and constants only, e.g. softplus(rho), analytic entropies -- are hoisted to the
        front and grouped by dependency level, so the kernel evaluates them once per CTA with the lanes of a warp working
        on a level in parallel; the per-sample ops follow in their original (topological) order.  `self.ops` itself stays
        the plain program (what oracle/dag_interp.py interprets)."""
        inv = {v: k for k, v in _DAG.items()}
        level = {}                       # slot -> dependency level of the uniform op that defines it
        uniform, rest = [], []
        for o in self.ops:
            op, dst, a_, b_, c_ = inv[o[0]], o[1], o[2], o[3], o[4]
            if op in ("CONST", "PARAM"):
                lv = 0
            elif op in ("EPS", "DATA", "ACC_SAMPLE", "ACC_ROW"):
                lv = None
            else:
                ins = (a_, b_, c_) if op == "NORMAL_LP" else ((a_, b_) if op in ("ADD", "SUB", "MUL", "DIV") else (a_,))
                lv = None if any(x not in level for x in ins) else 1 + max(level[x] for x in ins)
            if lv is None:
                rest.append(o)
            else:
                level[dst] = lv
                uniform.append((lv, o))
        if not uniform:
            return list(self.ops)
        # per-sample segment: the leaves (noise draws, data loads) first -- the kernel issues them back to back -- and every
        # ACC_SAMPLE / ACC_ROW whose operand is produced by a per-sample non-leaf op is folded into that op as a flag
        # (bit 6 / bit 7 of the opcode byte): one interpreted op less per accumulated term
        eps_ops = [o for o in rest if inv[o[0]] == "EPS"]
        data_ops = [o for o in rest if inv[o[0]] == "DATA"]
        body = [o for o in rest if inv[o[0]] not in ("EPS", "DATA")]
        producer = {o[1]: i for i, o in enumerate(body) if not inv[o[0]].startswith("ACC")}
        fused, flags = set(), {}
        for i, o in enumerate(body):
            op = inv[o[0]]
            if op.startswith("ACC") and o[2] in producer:
                bit = 0x40 if op == "ACC_SAMPLE" else 0x80
                j = producer[o[2]]
                if not flags.get(j, 0) & bit:
                    flags[j] = flags.get(j, 0) | bit
                    fused.add(i)
        body = [((o[0] | flags.get(i, 0),) + tuple(o[1:])) for i, o in enumerate(body) if i not in fused]
        if len(eps_ops) > 65535 or len(data_ops) > 65535:
            return list(self.ops)
        rest = eps_ops + data_ops + body
        out, prev = [], 0
        for lv in sorted({l for l, _ in uniform}):
            ops_lv = sorted((o for l, o in uniform if l == lv), key=lambda o: o[0])       # same opcodes side by side: less divergence
            for k in range(0, len(ops_lv), 65535):
                chunk = ops_lv[k:k + 65535]
                out.append((_DAG_LEVEL, 0, len(chunk), prev, 0, 0.0))
                out.extend(chunk)
                prev = len(chunk)
        if len(out) > 65535:             # header count is a 16-bit field: keep such programs in the plain layout
            return list(self.ops)
        return [(_DAG_UNIFORM_HEADER, 0, len(out), len(eps_ops), len(data_ops), 0.0)] + out + rest

    def table(self):
        ops = self.device_ops()
        t = np.zeros(len(ops), dtype=np.dtype([("opcode", "<i4"), ("dst", "<i4"), ("a", "<i4"), ("b", "<i4"),
                                               ("c", "<i4"), ("imm", "<f4")]))
        for i, o in enumerate(ops):
            t[i] = o
        return t


def _observed_tensor(var):
    t = var._observed_value if isinstance(var, RandomVariable) else var._value
    if not torch.is_tensor(t):
        raise UnsupportedModelError("scalar-DAG family: observed value of %r is not a tensor" % var.name)
    if t.dim() < 2 or t.shape[0] != 1 or int(np.prod(t.shape[2:])) != 1:
        raise UnsupportedModelError("scalar-DAG family: observed %r must hold scalars per data row (shape %s)" % (var.name, tuple(t.shape)))
    return t


class DagPlan(Plan):
    family = "dag (K1)"

    def __init__(self, joint, posterior):
        super().__init__(joint, posterior)
        P = self.prog = DagProgram()
        q_vars = posterior._flatten()
        self.q_by_name = {v.name: v for v in q_vars}
        if len(self.q_by_name) != len(q_vars):
            raise UnsupportedModelError("scalar-DAG family: duplicate variable names in the posterior model")
        self._q, self._p, self._qinfo = {}, {}, {}
        # q sampling, in name order (noise stream k = k-th sampled q variable in this order)
        for v in q_vars:
            self.q_value(v)
        terms = []
        # log p(x, z) with q's samples re-assigned BY NAME (utilities.py:282-309), roots included
        for v in joint._flatten():
            if not isinstance(v, RandomVariable) or v.distribution.kind in ("deterministic", "empirical"):
                continue
            kind = v.distribution.kind
            if kind in ("binomial", "bernoulli"):
                lp = self.bernoulli_log_prob(v)
            elif kind in _DAG_LOC_SCALE_P:
                x = self.p_value(v)
                loc = self.compile(v.partial_links["loc"].expr, self.p_value)
                scale = self.compile(v.partial_links["scale"].expr, self.p_value)
                lp = self.log_prob(kind, x, loc, scale)
            else:
                raise UnsupportedModelError("scalar-DAG family: distribution %r of %r is not lowered" % (kind, v.name))
            if P.rowdep[lp] and not v.is_observed:
                raise UnsupportedModelError("scalar-DAG family: latent %r has a per-row log-probability (local latents are "
                                            "not lowered)" % v.name)
            terms.append(("ACC_ROW" if P.rowdep[lp] else "ACC_SAMPLE", lp))
        # entropy of q: analytic where torch has it, else -log q (variables.py:156-162, 744-749)
        for v in q_vars:
            info = self._qinfo.get(v.name)
            if info is None:
                continue
            kind, loc, scale, z = info
            if kind == "normal":
                h = P.emit("NORMAL_ENTROPY", a=scale)
            elif kind == "lognormal":
                h = P.emit("ADD", a=P.emit("NORMAL_ENTROPY", a=scale), b=loc)
            else:
                h = P.emit("NEG", a=self.log_prob(kind, z, loc, scale))
            if P.rowdep[h]:
                raise UnsupportedModelError("scalar-DAG family: q variable %r depends on per-row data (amortised posteriors are "
                                            "not lowered)" % v.name)
            terms.append(("ACC_SAMPLE", h))
        for op, slot in terms:
            P.emit(op, a=slot)
        if P.n_slots > DAG_MAX_SLOTS or len(P.params) > DAG_MAX_PARAMS:
            raise UnsupportedModelError("scalar-DAG family: program too large (%d slots, %d parameters)" % (P.n_slots, len(P.params)))
        rows = [r for r in P.col_rows if r > 1]
        if rows and any(r != rows[0] for r in rows):
            raise UnsupportedModelError("scalar-DAG family: observed variables disagree on the number of data rows %s" % sorted(set(rows)))
        self.n_rows = rows[0] if rows else 1
        self._ops_dev = None

    # -- values ------------------------------------------------------------------------------------
    def _root_value(self, var):
        P = self.prog
        if var.is_observed:
            return P.data(var, _observed_tensor(var).shape[1])
        if var.learnable:
            return P.param(var._value)
        t = var._value
        if not torch.is_tensor(t) or t.numel() != 1:
            raise UnsupportedModelError("scalar-DAG family: constant %r is not a scalar" % var.name)
        return P.const(float(t.reshape(-1)[0]))

    def q_value(self, var):
        if id(var) in self._q:
            return self._q[id(var)]
        P = self.prog
        if isinstance(var, RootVariable):
            slot = self._root_value(var)
        elif var.distribution.kind == "deterministic":
            slot = self.compile(var.partial_links["value"].expr, self.q_value)
        elif var.distribution.kind in _DAG_LOC_SCALE:
            kind = var.distribution.kind
            loc = self.compile(var.partial_links["loc"].expr, self.q_value)
            scale = self.compile(var.partial_links["scale"].expr, self.q_value)
            u = P.emit("ADD", a=loc, b=P.emit("MUL", a=P.eps(var.name), b=scale))       # torch Normal.rsample: loc + eps * scale
            slot = u if kind == "normal" else P.emit("EXP" if kind == "lognormal" else "SIGMOID", a=u)
            self._qinfo[var.name] = (kind, loc, scale, slot)
        else:
            raise UnsupportedModelError("scalar-DAG family: q variable %r (%s) is not lowered" % (var.name, var.distribution.kind))
        self._q[id(var)] = slot
        return slot

    def p_value(self, var):
        if id(var) in self._p:
            return self._p[id(var)]
        P = self.prog
        if var.name in self.q_by_name and not var.is_observed:
            slot = self.q_value(self.q_by_name[var.name])               # by-name re-assignment (collision quirk included)
        elif isinstance(var, RootVariable):
            slot = self._root_value(var)
        elif var.distribution.kind == "deterministic" and not var.has_observed_value:
            slot = self.compile(var.partial_links["value"].expr, self.p_value)      # incl. observed regressors (observed root)
        elif var.is_observed:
            if not var.has_observed_value:
                raise UnsupportedModelError("scalar-DAG family: %r is observed through a random dataset" % var.name)
            slot = P.data(var, _observed_tensor(var).shape[1])
        else:
            raise UnsupportedModelError("latent variable %r has no counterpart in the posterior model" % var.name)
        self._p[id(var)] = slot
        return slot

    # -- expressions -------------------------------------------------------------------------------
    def compile(self, e, value_of):
        P = self.prog
        if isinstance(e, VarRef):
            return value_of(e.var)
        if isinstance(e, Const) or isinstance(e, (int, float, np.floating, np.integer)):
            v = e.value if isinstance(e, Const) else e
            if isinstance(v, np.ndarray) or torch.is_tensor(v):
                if int(np.prod(v.shape)) != 1:
                    raise UnsupportedModelError("scalar-DAG family: non-scalar constant in a link")
                v = float(np.asarray(v).reshape(-1)[0])
            if not isinstance(v, (int, float, np.floating, np.integer)):
                raise UnsupportedModelError("scalar-DAG family: constant %r in a link" % (v,))
            return P.const(v)
        if isinstance(e, Call) and not e.kwargs:
            if e.name in _DAG_BINARY and len(e.args) == 2:
                return P.emit(_DAG_BINARY[e.name], a=self.compile(e.args[0], value_of), b=self.compile(e.args[1], value_of))
            if e.name == "pow" and len(e.args) == 2:
                ex = e.args[1].value if isinstance(e.args[1], Const) else e.args[1]
                if isinstance(ex, (int, float, np.floating, np.integer)):
                    return P.emit("POWI", a=self.compile(e.args[0], value_of), imm=float(ex))
            if e.name in _DAG_UNARY and len(e.args) == 1:
                return P.emit(_DAG_UNARY[e.name], a=self.compile(e.args[0], value_of))
        raise UnsupportedModelError("scalar-DAG family: link expression %s is not lowered" % getattr(e, "name", type(e).__name__))

    def bernoulli_log_prob(self, v):
        """Observed Bernoulli / Binomial(total_count = 1) node with a `logits` link, as torch evaluates it
        (distributions.py:561-592; torch Binomial.log_prob with n = 1: the three lgamma terms vanish):
            y l - (max(l, 0) + log1p(exp(-|l|)))."""
        P = self.prog
        links = v.partial_links
        if not v.is_observed:
            raise UnsupportedModelError("scalar-DAG family: discrete latent %r has no pathwise gradient (not lowered)" % v.name)
        if "logits" not in links:
            raise UnsupportedModelError("scalar-DAG family: %r must be parameterised by logits" % v.name)
        if v.distribution.kind == "binomial":
            n = _const_value(links["total_count"].expr)
            if n is None:
                root = _as_root(links["total_count"].expr)
                n = float(root._value.reshape(-1)[0]) if root is not None and root._value.numel() == 1 else None
            if n != 1.0:
                raise UnsupportedModelError("scalar-DAG family: Binomial %r is lowered for total_count = 1 only" % v.name)
        y = self.p_value(v)
        l = self.compile(links["logits"].expr, self.p_value)
        norm = P.emit("ADD", a=P.emit("RELU", a=l), b=P.emit("LOG1P", a=P.emit("EXP", a=P.emit("NEG", a=P.emit("ABS", a=l)))))
        return P.emit("SUB", a=P.emit("MUL", a=y, b=l), b=norm)

    def log_prob(self, kind, x, loc, scale):
        """The op sequence torch evaluates: Normal.log_prob, and TransformedDistribution.log_prob =
        base.log_prob(T^-1(y)) - log|det J| for ExpTransform / SigmoidTransform (distributions.py:493-507 pattern)."""
        P = self.prog
        if kind == "normal":
            return P.emit("NORMAL_LP", a=x, b=loc, c=scale)
        if kind == "lognormal":
            lx = P.emit("LOG", a=x)                                   # ExpTransform: inv = log y, log|det J| = x
            return P.emit("SUB", a=P.emit("NORMAL_LP", a=lx, b=loc, c=scale), b=lx)
        if kind == "cauchy":            # torch Cauchy.log_prob: -log(pi) - log(scale) - log1p(((x - loc) / scale)^2)
            zz = P.emit("DIV", a=P.emit("SUB", a=x, b=loc), b=scale)
            t = P.emit("SUB", a=P.const(-float(np.log(np.pi))), b=P.emit("LOG", a=scale))
            return P.emit("SUB", a=t, b=P.emit("LOG1P", a=P.emit("MUL", a=zz, b=zz)))
        if kind == "laplace":           # torch Laplace.log_prob: -log(2 scale) - |x - loc| / scale
            t = P.emit("NEG", a=P.emit("LOG", a=P.emit("MUL", a=P.const(2.0), b=scale)))
            return P.emit("SUB", a=t, b=P.emit("DIV", a=P.emit("ABS", a=P.emit("SUB", a=x, b=loc)), b=scale))
        yc = P.emit("CLAMP_UNIT", a=x)                                # SigmoidTransform._inverse: clamp, log y - log1p(-y)
        u = P.emit("SUB", a=P.emit("LOG", a=yc), b=P.emit("LOG1P", a=P.emit("NEG", a=yc)))
        ladj = P.emit("SUB", a=P.emit("NEG", a=P.emit("SOFTPLUS", a=P.emit("NEG", a=u))), b=P.emit("SOFTPLUS", a=u))
        return P.emit("SUB", a=P.emit("NORMAL_LP", a=u, b=loc, c=scale), b=ladj)

    # -- evaluation --------------------------------------------------------------------------------
    def elbo(self, number_samples, empirical_samples):
        if config.device.type != "cuda":
            raise RuntimeError("brancher_b200 evaluates the ELBO only on CUDA devices (no CPU fallback); "
                               "config.device is %s" % config.device)
        from brancher_b200 import _cuda as cu
        cu.lib()
        P = self.prog
        s0, S_local = distributed.shard(number_samples)
        r = cu.sample_range(number_samples, s0=s0, s_local=S_local, seed=config.seed, offset=config.next_offset())
        params = list(P.params)

        def runner():
            dev = config.device
            if self._ops_dev is None or self._ops_dev.device != dev:
                self._ops_dev = torch.from_numpy(P.table().view(np.uint8)).to(dev)
            cols = []
            for var, rows in zip(P.columns, P.col_rows):
                t = empirical_samples[var] if var in empirical_samples else _observed_tensor(var)
                t = t.reshape(-1).to(torch.float32)
                if t.numel() != rows:
                    raise ValueError("observed %r now has %d rows, the lowered plan expects %d" % (var.name, t.numel(), rows))
                cols.append(t.expand(self.n_rows) if rows == 1 else t)
            data = torch.stack(cols, dim=1).contiguous() if cols else None
            eps = None
            if _INJECTED is not None:
                missing = [n for n in P.eps_names if n not in _INJECTED]
                if missing:
                    raise KeyError("inject_noise: no noise given for q variables %s" % missing)
                eps = torch.stack([torch.as_tensor(_INJECTED[n], dtype=torch.float32, device=dev).reshape(-1)[s0:s0 + S_local]
                                   for n in P.eps_names], dim=1).contiguous()
            pvec = torch.stack([p.detach().reshape(()) for p in params]) if params else torch.zeros(0, device=dev)
            loss, g = cu.dag_elbo_fwd_bwd(self._ops_dev, self._ops_dev.numel() // 24, P.n_slots, pvec, data, self.n_rows, eps, len(P.eps_names), r)
            loss, grads = distributed.all_reduce_partials(loss, [g])
            g = grads[0]
            return loss, [g[i].reshape(p.shape) if p.requires_grad else None for i, p in enumerate(params)]

        return _FusedELBO.apply(runner, *params)

    def static_evaluation(self, number_samples, empirical_samples, offset_dev):
        """see Plan.static_evaluation"""
        from types import SimpleNamespace
        from brancher_b200 import _cuda as cu
        cu.lib()
        P = self.prog
        if distributed.world_size() != 1 or _INJECTED is not None or not P.params:
            return None
        dev = config.device
        r = cu.sample_range(number_samples, seed=config.seed, offset=config.next_offset(), offset_dev=offset_dev)
        if self._ops_dev is None or self._ops_dev.device != dev:
            self._ops_dev = torch.from_numpy(P.table().view(np.uint8)).to(dev)
        cols = []
        for var, rows in zip(P.columns, P.col_rows):
            t = empirical_samples[var] if var in empirical_samples else _observed_tensor(var)
            t = t.reshape(-1).to(torch.float32)
            if t.numel() != rows:
                raise ValueError("observed %r now has %d rows, the lowered plan expects %d" % (var.name, t.numel(), rows))
            cols.append(t.expand(self.n_rows) if rows == 1 else t)
        data = torch.stack(cols, dim=1).contiguous() if cols else None
        params = list(P.params)
        dparams = torch.zeros(len(params), dtype=torch.float32, device=dev)
        loss = torch.zeros(1, dtype=torch.float64, device=dev)
        flat_params = [p.detach().reshape(-1) for p in params]

        def launch():
            dparams.zero_()
            loss.zero_()
            pvec = torch.cat(flat_params)
            cu.dag_elbo_fwd_bwd(self._ops_dev, self._ops_dev.numel() // 24, P.n_slots, pvec, data, self.n_rows, None,
                                len(P.eps_names), r, loss=loss, dparams=dparams)

        return SimpleNamespace(params=params, grads=[dparams[i:i + 1] for i in range(len(params))], loss=loss, launch=launch)


# ---------------------------------------------------------------------------------------------------
# K5: amortised VAE family (examples/VAE_playground.py:30-80)
# ---------------------------------------------------------------------------------------------------
def _module_call(expr):
    """ModuleCall(nn.Module, [one argument]) -> (module, argument expr) or None"""
    from brancher_b200.variables import ModuleCall
    if isinstance(expr, ModuleCall) and isinstance(expr.fn, torch.nn.Module) and len(expr.args) == 1 and not expr.kwargs:
        return expr.fn, expr.args[0]
    return None


def _index_of(expr, key):
    """Index(VarRef(var), key) -> var (a DeterministicVariable holding a dict-valued module output) or None"""
    from brancher_b200.variables import Index
    if isinstance(expr, Index) and expr.key == key and isinstance(expr.base, VarRef):
        return expr.base.var
    return None


def _identify_relu_mlp(module, n_in, heads, what):
    """Recover the layer structure of a user-written nn.Module (its __call__ is opaque Python, functions.py:9-45) for the K5
    kernels: hidden layers Linear -> ReLU in registration order, then one Linear per requested head.  `heads` maps the
    module's output keys to a post-processing tag: "id" (the raw head) or "softplus+c" (softplus(head) + constant c, the
    encoder's sd, VAE_playground.py:44-46).  The hypothesis is VERIFIED numerically on a random probe batch, so a module that
    computes anything else is rejected instead of silently mis-lowered.  Returns (hidden [(Linear)], {key: Linear}, c)."""
    linears = [m for m in module.modules() if isinstance(m, torch.nn.Linear)]
    nh = len(heads)
    if len(linears) < nh + 1:
        raise UnsupportedModelError("%s: expected at least %d nn.Linear layers, found %d" % (what, nh + 1, len(linears)))
    hidden, head_layers = linears[:-nh], linears[-nh:]
    dims = [n_in] + [l.out_features for l in hidden]
    if any(l.in_features != d for l, d in zip(hidden, dims[:-1])) or any(h.in_features != dims[-1] for h in head_layers):
        raise UnsupportedModelError("%s: the nn.Linear layers do not form a chain %s -> heads" % (what, dims))
    import itertools
    dev = hidden[0].weight.device
    g = torch.Generator().manual_seed(1234)
    probe = torch.rand(6, n_in, generator=g).to(dev)
    with torch.no_grad():
        try:
            out = module(probe.unsqueeze(-1)) if what.startswith("encoder") else module(probe)
        except Exception as exc:
            raise UnsupportedModelError("%s: probing the module failed (%s)" % (what, exc))
        if not isinstance(out, dict) or any(k not in out for k in heads):
            raise UnsupportedModelError("%s: the module must return a dict with keys %s" % (what, sorted(heads)))
        h = probe
        for l in hidden:
            h = torch.relu(torch.nn.functional.linear(h, l.weight, l.bias))
        for perm in itertools.permutations(head_layers):
            ok, c_found = True, 0.0
            for (key, tag), l in zip(sorted(heads.items()), perm):
                raw = torch.nn.functional.linear(h, l.weight, l.bias)
                got = out[key].reshape(raw.shape)
                if tag == "id":
                    ok = ok and torch.allclose(got, raw, rtol=1e-5, atol=1e-6)
                else:
                    d = got - torch.nn.functional.softplus(raw)
                    c_found = round(float(d.median()), 6)
                    ok = ok and float((d - c_found).abs().max()) < 1e-5 and c_found > -1e-6
            if ok:
                return hidden, dict(zip(sorted(heads), perm)), max(c_found, 0.0)
    raise UnsupportedModelError("%s: the module is not a ReLU MLP with linear heads %s (numerical probe mismatch)" % (what, sorted(heads)))


class VaePlan:
    """x ~ Binomial(1, logits = decoder(z)["mean"]), z ~ N(0, I); q: x = minibatch of an EmpiricalVariable,
    z ~ N(encoder(x)["mean"], encoder(x)["sd"]) -- examples/VAE_playground.py:65-80 -> brn_vae_elbo_fwd_bwd (K5).
    The same minibatch is shared by all MC samples (SURVEY 8d C5); gradients land in the nn.Modules' parameters."""
    family = "vae (K5)"

    def __init__(self, joint, posterior, x_q, z_name, enc, dec):
        self.joint, self.posterior, self.x_q, self.z_name = joint, posterior, x_q, z_name
        (self.enc_hidden, enc_heads, self.sd_offset), (self.dec_hidden, dec_heads, _) = enc, dec
        self.enc_mean, self.enc_sd, self.dec_out = enc_heads["mean"], enc_heads["sd"], dec_heads["mean"]
        self._net = None

    def layers(self):
        return list(self.enc_hidden) + [self.enc_mean, self.enc_sd] + list(self.dec_hidden) + [self.dec_out]

    def parameters(self):
        return [p for l in self.layers() for p in (l.weight, l.bias)]

    def _network(self, cu):
        key = tuple(p.data_ptr() for p in self.parameters())
        if self._net is None or self._net_key != key:
            wb = lambda l: (l.weight, l.bias)
            self._net = cu.VaeNet([wb(l) for l in self.enc_hidden], wb(self.enc_mean), wb(self.enc_sd),
                                  [wb(l) for l in self.dec_hidden], wb(self.dec_out), sd_offset=self.sd_offset)
            self._net_key = key
        return self._net

    def static_minibatch(self):
        """True when every evaluation sees the same rows (EmpiricalVariable(indices=...) with constant indices)"""
        idx = [p for p in self.x_q.parents if p.name.endswith("_indices")]
        return bool(idx) and all(isinstance(p, RootVariable) for p in idx)

    def _minibatch(self, empirical_samples):
        # x is observed in q, not in p: the reference draws it as part of the sampler (gradient_estimators.py:41), ONE draw
        # shared by all MC samples here (SURVEY 8d C5)
        t = empirical_samples[self.x_q] if self.x_q in empirical_samples else \
            self.x_q._get_sample(1, observed=False, differentiable=False)[self.x_q]
        if not torch.is_tensor(t) or t.shape[0] != 1:
            raise UnsupportedModelError("vae family: the minibatch must be shared by all MC samples (singleton sample axis), got "
                                        "shape %s" % (tuple(t.shape),))
        return t.reshape(t.shape[1], -1).to(torch.float32).contiguous()

    def _run(self, cu, net, X, r, eps, loss=None):
        row0, nb = distributed.shard(X.shape[0])
        net.zero_grads()
        loss = cu.vae_elbo_fwd_bwd(X[row0:row0 + nb].contiguous(), net, r, eps=None if eps is None else eps[:, row0:row0 + nb],
                                   var_id=0, row0=row0, B_total=X.shape[0], add_constant=(distributed.rank() == 0), loss=loss)
        if distributed.world_size() > 1:
            distributed.all_reduce_flat(net.flat, loss)
        return loss

    def elbo(self, number_samples, empirical_samples):
        if config.device.type != "cuda":
            raise RuntimeError("brancher_b200 evaluates the ELBO only on CUDA devices (no CPU fallback); "
                               "config.device is %s" % config.device)
        from brancher_b200 import _cuda as cu
        cu.lib()
        r = cu.sample_range(number_samples, seed=config.seed, offset=config.next_offset())
        params = self.parameters()

        def runner():
            net = self._network(cu)
            X = self._minibatch(empirical_samples)
            eps = None
            if _INJECTED is not None:
                if self.z_name not in _INJECTED:
                    raise KeyError("inject_noise: no noise given for q variable %r" % self.z_name)
                eps = torch.as_tensor(_INJECTED[self.z_name], dtype=torch.float32, device=config.device).reshape(
                    number_samples, X.shape[0], -1)
            loss = self._run(cu, net, X, r, eps)
            grads = [g.clone() for pair in net.grads for g in pair]
            return loss, [g.reshape(p.shape) if p.requires_grad else None for g, p in zip(grads, params)]

        return _FusedELBO.apply(runner, *params)

    def static_evaluation(self, number_samples, empirical_samples, offset_dev):
        from types import SimpleNamespace
        from brancher_b200 import _cuda as cu
        cu.lib()
        if distributed.world_size() != 1 or _INJECTED is not None or not self.static_minibatch():
            return None
        r = cu.sample_range(number_samples, seed=config.seed, offset=config.next_offset(), offset_dev=offset_dev)
        net = self._network(cu)
        net.zero_grads()
        X = self._minibatch(empirical_samples)
        loss = torch.zeros(1, dtype=torch.float64, device=config.device)
        params = self.parameters()
        grads = [g.reshape(-1) if g.is_contiguous() else g for pair in net.grads for g in pair]

        def launch():
            loss.zero_()
            self._run(cu, net, X, r, None, loss=loss)

        return SimpleNamespace(params=params, grads=grads, loss=loss, launch=launch)


def _lower_vae(joint, posterior):
    q_by_name = {v.name: v for v in posterior._flatten()}
    xs = [v for v in joint._flatten() if isinstance(v, RandomVariable) and v.distribution.kind in ("binomial", "bernoulli")]
    if len(xs) != 1:
        raise UnsupportedModelError("vae family: exactly one Binomial / Bernoulli likelihood node expected")
    x = xs[0]
    if x.distribution.kind == "binomial":
        tc = _as_root(x.partial_links["total_count"].expr)
        if tc is None or tc.value.numel() != 1 or float(tc.value.reshape(-1)[0]) != 1.0:
            raise UnsupportedModelError("vae family: Binomial likelihood is lowered only for total_count=1")
    if "logits" not in x.partial_links:
        raise UnsupportedModelError("vae family: the likelihood must be parameterised by logits")
    dec_out = _index_of(x.partial_links["logits"].expr, "mean")
    if dec_out is None or getattr(dec_out, "distribution", None) is None or dec_out.distribution.kind != "deterministic":
        raise UnsupportedModelError("vae family: logits must be DeterministicVariable(decoder(z))['mean']")
    mc = _module_call(dec_out.partial_links["value"].expr)
    z = _var(mc[1]) if mc else None
    if mc is None or z is None or not isinstance(z, RandomVariable) or z.distribution.kind != "normal":
        raise UnsupportedModelError("vae family: the decoder must be a BrancherFunction(nn.Module) applied to a Normal latent")
    decoder = mc[0]
    zl, zs = _as_root(z.partial_links["loc"].expr), (_softplus_root(z.partial_links["scale"].expr) or _as_root(z.partial_links["scale"].expr))
    if zl is None or zs is None or getattr(zl, "learnable", False) or getattr(zs, "learnable", False):
        raise UnsupportedModelError("vae family: the latent prior must have constant parameters")
    sc = torch.nn.functional.softplus(zs.value) if _softplus_root(z.partial_links["scale"].expr) is not None else zs.value
    if float(zl.value.abs().max()) != 0.0 or float((sc - 1.0).abs().max()) > 1e-6:
        raise UnsupportedModelError("vae family: only the standard-normal latent prior N(0, I) is lowered")
    L = int(zl.value.numel())
    # posterior side
    qz, qx = q_by_name.get(z.name), q_by_name.get(x.name)
    if qz is None or qx is None or qz.distribution.kind != "normal" or qx.distribution.kind != "empirical" or not qx.is_observed:
        raise UnsupportedModelError("vae family: the posterior needs an observed EmpiricalVariable %r and a Normal %r" % (x.name, z.name))
    enc_out = _index_of(qz.partial_links["loc"].expr, "mean")
    if enc_out is None or _index_of(qz.partial_links["scale"].expr, "sd") is not enc_out or \
            enc_out.distribution.kind != "deterministic":
        raise UnsupportedModelError("vae family: q(z) must be Normal(encoder_output['mean'], encoder_output['sd'])")
    mc = _module_call(enc_out.partial_links["value"].expr)
    if mc is None or _var(mc[1]) is not qx:
        raise UnsupportedModelError("vae family: the encoder must be a BrancherFunction(nn.Module) applied to the EmpiricalVariable")
    encoder = mc[0]
    if set(v.name for v in _latent_random_variables(joint)) - {z.name, x.name}:
        raise UnsupportedModelError("vae family: unexpected additional latent variables")
    D = int(np.prod(qx.distribution.dataset.shape[1:])) if hasattr(qx.distribution, "dataset") else None
    if D is None:
        lin = [m for m in encoder.modules() if isinstance(m, torch.nn.Linear)]
        D = lin[0].in_features if lin else 0
    enc = _identify_relu_mlp(encoder, D, {"mean": "id", "sd": "softplus+c"}, "encoder")
    dec = _identify_relu_mlp(decoder, L, {"mean": "id"}, "decoder")
    if enc[1]["mean"].out_features != L or dec[1]["mean"].out_features != D:
        raise UnsupportedModelError("vae family: encoder / decoder widths do not match the data (%d) and latent (%d) sizes" % (D, L))
    return VaePlan(joint, posterior, qx, z.name, enc, dec)



def lower(joint, posterior):
    """Pick the kernel family: the dense families (K2 linear, K3 BNN) by pattern, the amortised VAE (K5), else the
    scalar-DAG family (K1)."""
    try:
        return _lower_dense(joint, posterior)
    except UnsupportedModelError as dense_err:
        try:
            return _lower_vae(joint, posterior)
        except UnsupportedModelError as vae_err:
            try:
                return DagPlan(joint, posterior)
            except UnsupportedModelError as dag_err:
                raise UnsupportedModelError("model graph is not recognised by any fused kernel family.\n  dense (K2/K3): %s\n"
                                            "  vae (K5): %s\n  scalar DAG (K1): %s" % (dense_err, vae_err, dag_err)) from None


# ---------------------------------------------------------------------------------------------------
# particle ensembles (SVGD, K4)
# ---------------------------------------------------------------------------------------------------
class _ParticleLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, runner, *params):
        loss, G = runner()
        ctx.G, ctx.shapes = G, [p.shape for p in params]
        return loss.to(torch.float32).reshape(())

    @staticmethod
    def backward(ctx, g):
        return (None,) + tuple(g * ctx.G[i].reshape(sh) for i, sh in enumerate(ctx.shapes))


class ParticlePlan:
    """SVGD over (multi-class) logistic-regression particles: the joint model is the linear family (K2's graph), every
    particle is a ProbabilisticModel holding ONE learnable RootVariable named like the weights latent
    (development_playgrounds/SVGD_logistic_regression.py:34-48).  The same holds for regression particles: the joint model is
    Normal / Cauchy / Laplace(BF.matmul(weights, x), constant scale) (likelihood cu.GAUSSIAN / CAUCHY / LAPLACE, C = 1)."""
    family = "particles (K4)"

    def __init__(self, joint, particles, k, W, x_var, likelihood, C, scale=None):
        """scale: the constant noise scale of a regression likelihood (_constant_scale), None for the logistic ones"""
        from brancher_b200 import _cuda as cu
        self.joint, self.particles, self.k, self.x_var, self.likelihood, self.C = joint, particles, k, x_var, likelihood, C
        self.regression = likelihood in (cu.GAUSSIAN, cu.CAUCHY, cu.LAPLACE)
        if self.regression:
            self.family = "particles (K4, %s likelihood)" % {cu.GAUSSIAN: "Normal", cu.CAUCHY: "Cauchy", cu.LAPLACE: "Laplace"}[likelihood]
        self._scale = scale
        self.prepared_x = None       # fp16-pair form of a fixed observed matrix (regression), rebuilt when the matrix changes
        self.W = W
        lp = W.partial_links
        loc, sc_sp = _as_root(lp["loc"].expr), _softplus_root(lp["scale"].expr)
        sc = sc_sp or _as_root(lp["scale"].expr)
        if loc is None or sc is None:
            raise UnsupportedModelError("particle family: the prior's loc/scale must be constants")
        self.shape = tuple(loc._value.shape[2:])
        full = lambda t: t.detach().to(torch.float32).expand((1, 1) + self.shape).reshape(-1).contiguous()
        self.prior_loc = full(loc.value)
        self.prior_scale = full(torch.nn.functional.softplus(sc.value) if sc_sp is not None else sc.value)
        self.roots = []
        for p in particles:
            roots = [v for v in p._flatten() if isinstance(v, RootVariable) and v.name == W.name]
            if len(roots) != 1 or tuple(roots[0]._value.shape[2:]) != self.shape:
                raise UnsupportedModelError("every particle must hold one root named %r of shape %s" % (W.name, self.shape))
            self.roots.append(roots[0])

    def parameters(self):
        return [r.value for r in self.roots]

    def stacked(self):
        return torch.stack([p.detach().reshape(-1) for p in self.parameters()]).contiguous()

    def noise_scale(self):
        return _noise_scale_tensor(self._scale)

    def observations(self, cu, empirical):
        """(X [N, F], y [N]) of one evaluation, y in the dtype the likelihood's kernels read"""
        X = _data_matrix(empirical[self.x_var], "x")
        yv = empirical[self.k].reshape(-1)
        y = yv.to(torch.int32).contiguous() if self.likelihood == cu.CATEGORICAL else yv.to(torch.float32).contiguous()
        if self.regression and self.prepared_x is None:
            self.prepared_x = cu.PreparedX()
        return X, y

    def loss(self, empirical):
        if config.device.type != "cuda":
            raise RuntimeError("brancher_b200 evaluates particle losses only on CUDA devices (no CPU fallback)")
        from brancher_b200 import _cuda as cu
        cu.lib()

        def runner():
            X, y = self.observations(cu, empirical)
            if self.regression:
                return cu.linreg_particles_loss_grad(X, y, self.likelihood, self.stacked(), self.noise_scale(), self.prior_loc,
                                                     self.prior_scale, prepared=self.prepared_x)
            return cu.linear_particles_loss_grad(X, y, self.likelihood, self.stacked(), self.C, self.prior_loc, self.prior_scale)

        return _ParticleLoss.apply(runner, *self.parameters())


def _lower_regression_particles(joint, particles, k, latents):
    """Particles of Normal / Cauchy / Laplace(loc = BF.matmul(W, x), scale): W the one latent, [1, F] with a Normal prior, x data,
    the scale a constant (a particle holds one root: there is no noise latent to carry)."""
    from brancher_b200 import _cuda as cu
    lik_name = REGRESSION_KINDS[k.distribution.kind]
    what = "particle family: %s likelihood" % lik_name
    loc, scale = k.partial_links["loc"].expr, k.partial_links["scale"].expr
    if not _is_call(loc, "matmul", 2):
        if any(_is_call(a, "matmul", 2) for a, _ in _commutative_add(loc)):
            raise UnsupportedModelError("%s %r: a bias added to BF.matmul(weights, x) is not lowered -- append a column of ones "
                                        "to x instead" % (what, k.name))
        raise UnsupportedModelError("%s %r: loc must be BF.matmul(weights, x)" % (what, k.name))
    W, x = _var(loc.args[0]), _var(loc.args[1])
    if W not in latents or not _is_data(x):
        raise UnsupportedModelError("%s %r: loc must be BF.matmul(weights, x) with weights a latent and x data" % (what, k.name))
    nu = _var(scale)
    if nu is not None and nu in latents:
        raise UnsupportedModelError("%s %r: a %s-distributed noise latent is not lowered -- a particle holds one root, the "
                                    "weights; give the noise scale as a constant" % (what, k.name, nu.distribution.kind))
    const = _constant_scale(scale, what, k)
    if const is None:
        raise UnsupportedModelError("%s %r: the noise scale must be a constant (deterministic or data-dependent scales are not "
                                    "lowered)" % (what, k.name))
    extra = sorted(v.name for v in latents if v is not W)
    if extra:
        raise UnsupportedModelError("%s %r: latent variables other than the weights are not lowered: %s" % (what, k.name, extra))
    if W.distribution.kind != "normal":
        raise UnsupportedModelError("%s %r: only a Normal prior on the weights is lowered (got %s)" % (what, k.name,
                                                                                                      W.distribution.kind))
    shape = tuple(W.partial_links["loc"].expr.var._value.shape[2:]) if _as_root(W.partial_links["loc"].expr) else ()
    if len(shape) != 2 or shape[0] != 1:
        raise UnsupportedModelError("%s %r: weights must have shape [1, F] (multi-output regression is not lowered), got %s"
                                    % (what, k.name, shape))
    if shape[1] > 128:
        raise UnsupportedModelError("%s %r: at most 128 features are lowered, got F = %d" % (what, k.name, shape[1]))
    likelihood = {"normal": cu.GAUSSIAN, "cauchy": cu.CAUCHY, "laplace": cu.LAPLACE}[k.distribution.kind]
    return ParticlePlan(joint, particles, k, W, x, likelihood, 1, scale=const)


def lower_particles(joint, particles):
    from brancher_b200 import _cuda as cu
    latents = _latent_random_variables(joint)
    liks = _observed_likelihood_nodes(joint)
    if len(liks) == 1 and liks[0].distribution.kind in REGRESSION_KINDS:
        return _lower_regression_particles(joint, particles, liks[0], latents)
    if len(liks) != 1 or len(latents) != 1:
        raise UnsupportedModelError("particle family needs one observed likelihood node and one latent weight matrix")
    k, W = liks[0], latents[0]
    kind = k.distribution.kind
    if kind not in ("binomial", "bernoulli", "categorical") or "logits" not in k.partial_links:
        raise UnsupportedModelError("particle family: likelihood %r is not lowered" % kind)
    if kind == "binomial":
        tc = _as_root(k.partial_links["total_count"].expr)
        if tc is None or tc.value.numel() != 1 or float(tc.value.reshape(-1)[0]) != 1.0:
            raise UnsupportedModelError("Binomial likelihood is lowered only for total_count=1")
    logits = k.partial_links["logits"].expr
    if not (_is_call(logits, "matmul", 2) and _var(logits.args[0]) is W and _is_data(_var(logits.args[1]))):
        raise UnsupportedModelError("particle family: logits must be BF.matmul(weights, x)")
    if W.distribution.kind != "normal":
        raise UnsupportedModelError("particle family: only a Normal prior on the weights is lowered")
    shape = tuple(W.partial_links["loc"].expr.var._value.shape[2:]) if _as_root(W.partial_links["loc"].expr) else ()
    if len(shape) != 2:
        raise UnsupportedModelError("particle family: weights must be a [C, F] matrix")
    C = shape[0]
    if kind != "categorical" and C != 1:
        raise UnsupportedModelError("Binomial/Bernoulli logistic regression needs weights of shape [1, F]")
    return ParticlePlan(joint, particles, k, W, _var(logits.args[1]), cu.CATEGORICAL if kind == "categorical" else cu.BERNOULLI, C)


class _WvgdLoss(torch.autograd.Function):
    """params = [theta_0.., loc_0.., rho_0..]; the runner returns the loss and one gradient per parameter."""
    @staticmethod
    def forward(ctx, runner, *params):
        loss, grads = runner()
        ctx.grads = grads
        return loss.to(torch.float32).reshape(())

    @staticmethod
    def backward(ctx, g):
        return (None,) + tuple(g * x for x in ctx.grads)


class WvgdPlan:
    """WVGD over (multi-class) logistic-regression or regression ensembles (development_playgrounds/WVGD_logistic_regression.py:33-58): the
    joint model is the linear family, particle k holds one learnable root named like the weights latent, sampler k one
    learnable Normal of the same name whose loc/scale are roots (scale a scalar or a full tensor)."""
    family = "wvgd (K6)"

    def __init__(self, pplan, samplers):
        self.pplan = pplan
        W_name = pplan.roots[0].name
        if len(samplers) != len(pplan.particles):
            raise UnsupportedModelError("WVGD needs one variational sampler per particle")
        self.loc_roots, self.scale_roots = [], []
        q_names = set()
        for smp in samplers:
            qs = [v for v in smp._flatten() if isinstance(v, RandomVariable) and v.name == W_name]
            if len(qs) != 1 or qs[0].distribution.kind != "normal":
                raise UnsupportedModelError("every WVGD sampler must hold one Normal variable named %r" % W_name)
            lq = qs[0].partial_links
            loc, sc = _as_root(lq["loc"].expr), _softplus_root(lq["scale"].expr)
            if loc is None or sc is None or tuple(loc._value.shape[2:]) != pplan.shape:
                raise UnsupportedModelError("WVGD sampler %r: loc/scale must be learnable roots of the particle's shape" % W_name)
            if sc._value.numel() not in (1, loc._value.numel()):
                raise UnsupportedModelError("WVGD sampler %r: scale must be a scalar or match the weights' shape" % W_name)
            self.loc_roots.append(loc)
            self.scale_roots.append(sc)
            q_names |= {loc.name, sc.name}
        if len({r._value.numel() for r in self.scale_roots}) != 1:
            raise UnsupportedModelError("WVGD samplers must agree on the shape of their scale parameter")
        # tied mode: the prior's auto-named hyper-parameter roots collide with the samplers' (utilities.py:282-309)
        lp = pplan.W.partial_links
        p_loc, p_sc = _as_root(lp["loc"].expr), (_softplus_root(lp["scale"].expr) or _as_root(lp["scale"].expr))
        tied = {p_loc.name in q_names, p_sc.name in q_names}
        if len(tied) != 1:
            raise UnsupportedModelError("WVGD: prior loc/scale roots are tied to the samplers inconsistently")
        self.tied = tied.pop()

    def parameters(self):
        return [r.value for r in self.pplan.roots] + [r.value for r in self.loc_roots] + [r.value for r in self.scale_roots]

    def loss(self, empirical, number_samples, biased, first_column_only):
        if config.device.type != "cuda":
            raise RuntimeError("brancher_b200 evaluates the WVGD loss only on CUDA devices (no CPU fallback)")
        from brancher_b200 import _cuda as cu
        cu.lib()
        pp = self.pplan
        n = len(pp.roots)
        params = self.parameters()
        r = cu.sample_range(number_samples, seed=config.seed, offset=config.next_offset())

        def runner():
            X, y = pp.observations(cu, empirical)
            theta = pp.stacked()
            loc = torch.stack([p.value.detach().reshape(-1) for p in self.loc_roots]).contiguous()
            scalar = self.scale_roots[0]._value.numel() == 1
            rho = torch.stack([p.value.detach().reshape(-1) for p in self.scale_roots]).contiguous()
            rho = rho.reshape(n) if scalar else rho
            eps0 = eps1 = None
            if _INJECTED is not None:          # {"elbo": [n,S,*shape], "particle": [n,S,*shape]}
                cv = lambda a: torch.as_tensor(a, dtype=torch.float32, device=theta.device).reshape(n, number_samples, -1).contiguous()
                eps0, eps1 = cv(_INJECTED["elbo"]), cv(_INJECTED["particle"])
            prior = None if self.tied else (pp.prior_loc, pp.prior_scale)
            loss, dloc, drho, dth, counts = cu.wvgd_loss_grad(X, y, pp.likelihood, pp.C, loc, rho, theta, number_samples, r, eps0, eps1,
                                                              prior=prior, biased=biased, first_column_only=first_column_only,
                                                              noise_scale=pp.noise_scale() if pp.regression else None,
                                                              prepared=pp.prepared_x)
            self.accepted = counts
            drho = drho.sum(1, keepdim=True) if scalar else drho
            grads = [dth[i].reshape(params[i].shape) for i in range(n)]
            grads += [dloc[i].reshape(params[n + i].shape) for i in range(n)]
            grads += [drho[i].reshape(params[2 * n + i].shape) for i in range(n)]
            return loss, grads

        return _WvgdLoss.apply(runner, *params)


def _wvgd_ensemble_weights(self, empirical, number_post_samples, first_column_only, chunk=8192, max_redraws=8):
    """WassersteinVariationalGradientDescent.post_process (inference.py:234-247) on the device: per sampler k the log
    normaliser of the importance weights of its truncated draws,  logZ_k = log sum_{s accepted} exp(log p(z_ks, data) -
    log q_k(z_ks))  (get_importance_weights, variables.py:821-841: unnormalised q log-prob, no division by the count), and
    the ensemble weights softmax_k(logZ_k).  Draws + Voronoi owner: K6a; log-likelihood of every draw: K6b; the masked
    log-sum-exp over [P, S] is a handful of torch reductions.  A sampler without any accepted draw is re-drawn (the
    reference loops until one is accepted, transformations.py:28-43).  Returns (weights [P], logZ [P], counts [P])."""
    from brancher_b200 import _cuda as cu
    cu.lib()
    pp = self.pplan
    n = len(pp.roots)
    dev = config.device
    X, y = pp.observations(cu, empirical)
    sigma = pp.noise_scale() if pp.regression else None
    theta = pp.stacked()
    loc = torch.stack([p.value.detach().reshape(-1) for p in self.loc_roots]).contiguous()
    scalar = self.scale_roots[0]._value.numel() == 1
    rho = torch.stack([p.value.detach().reshape(-1) for p in self.scale_roots]).contiguous()
    rho = rho.reshape(n) if scalar else rho
    d = loc.shape[1]
    F_last = d // pp.C
    injected = None
    if _INJECTED is not None:
        injected = torch.as_tensor(_INJECTED["post"], dtype=torch.float32, device=dev).reshape(n, number_post_samples, d)
    logZ = torch.full((n,), float("-inf"), dtype=torch.float64, device=dev)
    counts = torch.zeros(n, dtype=torch.int64, device=dev)
    ids = torch.arange(n, device=dev, dtype=torch.int32)[:, None]
    sg = torch.nn.functional.softplus(rho).to(torch.float64)
    log_sg_sum = (torch.log(sg) * (d if scalar else 1)).reshape(n, -1).sum(1)          # sum_i log sigma_ki
    done, redraws = 0, 0
    while done < number_post_samples or (injected is None and redraws < max_redraws and bool((counts == 0).any())):
        S = min(chunk, number_post_samples - done) if done < number_post_samples else min(chunk, number_post_samples)
        if done >= number_post_samples:
            redraws += 1
        eps = None if injected is None else injected[:, done:done + S].contiguous()
        r = cu.sample_range(S, seed=config.seed, offset=config.next_offset())
        Z, e, owner = cu.wvgd_sample_assign(loc, rho, theta, S, F_last, r, 0, eps, first_column_only)
        if pp.regression:
            ll, _ = cu.linreg_vectors_loglik_grad(X, y, pp.likelihood, Z.reshape(n * S, d), sigma, False, pp.prepared_x)
        else:
            ll, _ = cu.linear_vectors_loglik_grad(X, y, pp.likelihood, Z.reshape(n * S, d), pp.C, False)
        logw = ll.reshape(n, S)
        if not self.tied:          # tied: the prior's roots take sampler k's values, log p(z) == log q_k(z) and the pair cancels
            c = 0.5 * float(np.log(2 * np.pi))
            logq = (-0.5 * e.to(torch.float64) ** 2).sum(2) - log_sg_sum[:, None] - d * c
            pl, ps = pp.prior_loc.to(torch.float64), pp.prior_scale.to(torch.float64)
            logp = (-0.5 * ((Z.to(torch.float64) - pl) / ps) ** 2 - torch.log(ps) - c).sum(2)
            logw = logw + logp - logq
        mask = owner == ids
        if done >= number_post_samples:                       # re-draw: only for samplers that still have nothing
            mask = mask & (counts == 0)[:, None]
        logw = torch.where(mask, logw, torch.full_like(logw, float("-inf")))
        logZ = torch.logaddexp(logZ, torch.logsumexp(logw, 1))
        counts = counts + mask.sum(1)
        done += S if done < number_post_samples else 0
        if injected is not None and done >= number_post_samples:
            break
    weights = torch.softmax(logZ, 0)
    return weights, logZ, counts


WvgdPlan.ensemble_weights = _wvgd_ensemble_weights


def get_wvgd_plan(joint, particles, samplers):
    key = ("wvgd",) + tuple(id(p) for p in particles) + tuple(id(s) for s in samplers)
    plan = joint._plans.get(key)
    if plan is None:
        plan = WvgdPlan(get_particle_plan(joint, particles), list(samplers))
        joint._plans[key] = plan
    return plan


def get_particle_plan(joint, particles):
    key = ("particles",) + tuple(id(p) for p in particles)
    plan = joint._plans.get(key)
    if plan is None:
        plan = lower_particles(joint, list(particles))
        joint._plans[key] = plan
    return plan


def _observation_signature(joint):
    """which variables are observed (and how): a plan bakes this in, so observe() / unobserve() after the first evaluation
    must not reuse it"""
    return tuple(sorted((v.name, bool(getattr(v, "has_observed_value", False))) for v in joint._flatten() if v.is_observed))


def get_plan(joint, posterior):
    key = (id(posterior), _observation_signature(joint))
    plan = joint._plans.get(key)
    if plan is None or plan.posterior is not posterior:
        plan = lower(joint, posterior)
        joint._plans[key] = plan
    return plan
