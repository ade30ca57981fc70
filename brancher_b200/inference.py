"""Inference driver (mirror of brancher/inference.py:50-151): same signature and side effects.

    inference.perform_inference(joint_model, number_iterations, number_samples, optimizer, lr=...,
                                inference_method=ReverseKL(gradient_estimator=PathwiseDerivativeEstimator))

Each iteration is: loss = inference_method.compute_loss(...) [one fused CUDA ELBO+gradient evaluation],
isfinite check, loss.backward() [hands the kernel's gradients to .grad], optimizer step.

Deliberate deviation: the reference appends the loss twice per iteration with different shapes and
then crashes in np.array(loss_list) under numpy >= 1.24 (inference.py:105,108-109); here
`diagnostics["loss curve"]` holds ONE scalar per iteration.
"""
import warnings
from abc import ABC, abstractmethod

import numpy as np
import torch

from brancher_b200 import gradient_estimators
from brancher_b200.optimizers import ProbabilisticOptimizer


def perform_inference(joint_model, number_iterations, number_samples=1, optimizer="Adam", input_values={},
                      inference_method=None, posterior_model=None, sampler_model=None, pretraining_iterations=0,
                      **opt_params):
    if not inference_method:
        warnings.warn("The inference method was not specified, using the default reverse KL variational inference")
        inference_method = ReverseKL()
    if not posterior_model:
        posterior_model = joint_model.posterior_model
    if not sampler_model:
        sampler_model = getattr(inference_method, "sampler_model", None) or getattr(joint_model, "posterior_sampler", None)

    joint_model.update_observed_submodel()

    optimizers_list = []

    def append_prob_optimizer(model):
        prob_opt = ProbabilisticOptimizer(model, optimizer, **opt_params)
        if prob_opt.optimizer:
            optimizers_list.append(prob_opt)

    append_prob_optimizer(posterior_model)
    if inference_method.learnable_model:
        append_prob_optimizer(joint_model)
    if inference_method.learnable_sampler:
        append_prob_optimizer(sampler_model)

    inference_method.check_model_compatibility(joint_model, posterior_model, sampler_model)

    if _fused_loop(joint_model, posterior_model, number_iterations, number_samples, optimizer, opt_params, inference_method,
                   optimizers_list, input_values, pretraining_iterations):
        inference_method.post_process(joint_model)
        return

    try:
        from tqdm import tqdm
        iterator = tqdm(range(number_iterations))
    except ImportError:   # pragma: no cover
        iterator = range(number_iterations)

    losses = []
    for iteration in iterator:
        loss = inference_method.compute_loss(joint_model, posterior_model, sampler_model, number_samples)
        if torch.isfinite(loss.detach()).all().item():
            for opt in optimizers_list:
                opt.zero_grad()
            loss.backward()
            inference_method.correct_gradient(joint_model, posterior_model, sampler_model, number_samples)
            optimizers_list[0].update()
            if iteration > pretraining_iterations:
                for opt in optimizers_list[1:]:
                    opt.update()
        else:
            warnings.warn("Numerical error, skipping sample")
        losses.append(loss.detach())
    curve = torch.stack(losses).cpu().numpy() if losses else np.zeros((0,))
    joint_model.diagnostics.update({"loss curve": curve})
    inference_method.post_process(joint_model)


_FUSED_SGD = {"lr", "momentum", "weight_decay"}
_FUSED_ADAM = {"lr", "betas", "eps", "weight_decay"}
fused_loop_enabled = True        # set to False to force the step-by-step loop (tests compare the two)
last_loop = None                 # "graph" | "eager": which loop the last perform_inference ran


def _fused_loop(joint_model, posterior_model, number_iterations, number_samples, optimizer, opt_params, inference_method,
                optimizers_list, input_values, pretraining_iterations):
    """The whole iteration -- fused ELBO + gradient evaluation, optimiser step, finiteness check, loss curve, next Philox
    offset -- captured ONCE in a CUDA graph and replayed `number_iterations` times with no host synchronisation in between
    (SURVEY 8(f)1; replaces the loop body brancher/inference.py:95-108 and optimizers.py:69-73).  Used when the iteration is
    static: ReverseKL with the pathwise estimator, a lowered plan with persistent buffers, observations that are fixed
    tensors (no per-iteration minibatch draw), SGD / Adam with plain hyper-parameters, one process.  Returns False when the
    step-by-step loop has to run instead."""
    global last_loop
    last_loop = "eager"
    from brancher_b200 import config, lowering, distributed
    if not fused_loop_enabled or number_iterations <= 0 or config.device.type != "cuda" or distributed.world_size() != 1:
        return False
    # the cyclic garbage collector is held off for the duration of the loop set-up and the replays: a full collection over a
    # large heap (every Brancher variable is a small object graph) costs ~100 ms when it happens to trigger here -- measured as
    # one perform_inference call in five taking 219 ms instead of 104 ms (profiles/tools/api_probe.py)
    import gc
    gc_was_enabled = gc.isenabled()
    gc.disable()
    try:
        return _fused_loop_body(joint_model, posterior_model, number_iterations, number_samples, optimizer, opt_params,
                                inference_method, optimizers_list, input_values, pretraining_iterations)
    finally:
        if gc_was_enabled:
            gc.enable()


def _fused_loop_body(joint_model, posterior_model, number_iterations, number_samples, optimizer, opt_params, inference_method,
                     optimizers_list, input_values, pretraining_iterations):
    global last_loop
    from brancher_b200 import config, lowering, distributed
    if type(inference_method) is not ReverseKL or \
            inference_method.gradient_estimator is not gradient_estimators.PathwiseDerivativeEstimator:
        return False
    if input_values or pretraining_iterations or lowering._INJECTED is not None:
        return False
    if optimizer == "SGD" and set(opt_params) <= _FUSED_SGD and "lr" in opt_params:
        kind = 0
    elif optimizer == "Adam" and set(opt_params) <= _FUSED_ADAM:
        kind = 1
    else:
        return False
    joint_model.update_observed_submodel()
    observed = joint_model.observed_submodel
    if any(getattr(v, "distribution", None) is not None and v.distribution.kind == "empirical" for v in observed._flatten()):
        return False                              # a fresh minibatch is drawn every iteration
    plan = lowering.get_plan(joint_model, posterior_model)
    if not hasattr(plan, "static_evaluation"):
        return False
    from brancher_b200 import _cuda as cu
    empirical = observed._get_sample(1, observed=True, differentiable=False)
    dev = config.device
    offset_dev = torch.zeros(1, dtype=torch.int64, device=dev)
    ev = plan.static_evaluation(number_samples, empirical, offset_dev)
    if ev is None:
        return False
    trainable = [(p, g) for p, g in zip(ev.params, ev.grads) if p.requires_grad]
    # every parameter the step-by-step loop would update must be covered by the plan's gradients
    covered = {id(p) for p, _ in trainable}
    for opt in optimizers_list:
        for group in opt.optimizer.param_groups:
            if any(id(p) not in covered for p in group["params"]):
                return False
    if not trainable or any(not (p.is_contiguous() and p.dtype == torch.float32) for p, _ in trainable):
        return False
    fo = cu.FusedOptimizer([p.detach() for p, _ in trainable], [g for _, g in trainable], kind,
                           lr=opt_params.get("lr", 1e-3), momentum=opt_params.get("momentum", 0.0),
                           weight_decay=opt_params.get("weight_decay", 0.0), betas=opt_params.get("betas", (0.9, 0.999)),
                           eps=opt_params.get("eps", 1e-8), curve_len=number_iterations)

    def iteration():
        ev.launch()
        fo.step(ev.loss, offset_dev)

    # first iteration eagerly on a side stream (lazy initialisation must not happen under capture), the rest from a graph
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        iteration()
    torch.cuda.current_stream(dev).wait_stream(side)
    if number_iterations > 1:
        # capture_begin / capture_end directly: the torch.cuda.graph context manager runs gc.collect() and empties the caching
        # allocator on entry -- tens of milliseconds of host time on a large Python heap, paid by every perform_inference call
        graph = torch.cuda.CUDAGraph()
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            graph.capture_begin()
            try:
                iteration()
            finally:
                graph.capture_end()
        torch.cuda.current_stream(dev).wait_stream(side)
        # the capture itself does not execute: (number_iterations - 1) replays follow the eager first iteration
        for _ in range(number_iterations - 1):
            graph.replay()
    counters = fo.counters.cpu().numpy()                 # the ONE synchronisation of the loop
    curve = fo.curve[:number_iterations].cpu().numpy()
    for _ in range(number_iterations - 1):               # the step-by-step loop would have consumed one offset per iteration
        config.next_offset()
    if counters[2]:
        warnings.warn("Numerical error, skipped %d samples" % int(counters[2]))
    joint_model.diagnostics.update({"loss curve": curve})
    last_loop = "graph"
    return True


class InferenceMethod(ABC):
    learnable_model = False
    needs_sampler = False
    learnable_sampler = False

    @abstractmethod
    def check_model_compatibility(self, joint_model, posterior_model, sampler_model):
        pass

    @abstractmethod
    def compute_loss(self, joint_model, posterior_model, sampler_model, number_samples, input_values={}):
        pass

    def correct_gradient(self, joint_model, posterior_model, sampler_model, number_samples, input_values={}):
        pass

    @abstractmethod
    def post_process(self, joint_model):
        pass


class ReverseKL(InferenceMethod):
    """loss = -ELBO (inference.py:129-151)."""

    def __init__(self, gradient_estimator=gradient_estimators.PathwiseDerivativeEstimator):
        self.learnable_model = True
        self.needs_sampler = False
        self.learnable_sampler = False
        self.gradient_estimator = gradient_estimator

    def check_model_compatibility(self, joint_model, posterior_model, sampler_model):
        from brancher_b200 import lowering
        lowering.get_plan(joint_model, posterior_model)       # raises UnsupportedModelError early

    def compute_loss(self, joint_model, posterior_model, sampler_model, number_samples, input_values={}):
        return -joint_model.estimate_log_model_evidence(number_samples=number_samples, method="ELBO",
                                                        input_values=input_values, for_gradient=True,
                                                        posterior_model=posterior_model,
                                                        gradient_estimator=self.gradient_estimator)

    def post_process(self, joint_model):
        pass


class SteinVariationalGradientDescent(InferenceMethod):
    """SVGD over a list of particle models (inference.py:277-327).  `compute_loss` is ONE fused launch for all particles
    (K4a), `correct_gradient` replaces the reference's four nested Python loops by the tiled pairwise kernel (K4b),
    including its exact-median bandwidth heuristic and its sign convention for the interaction term."""

    def __init__(self):
        self.learnable_model = False
        self.needs_sampler = False
        self.learnable_sampler = False
        self.bandwidth = 0.01          # overwritten by update_bandwidth on every correct_gradient, as in the reference

    def check_model_compatibility(self, joint_model, posterior_model, sampler_model):
        from brancher_b200 import lowering
        lowering.get_particle_plan(joint_model, posterior_model)

    def compute_loss(self, joint_model, posterior_model, sampler_model, number_samples, input_values={}):
        from brancher_b200 import lowering
        plan = lowering.get_particle_plan(joint_model, posterior_model)
        joint_model.update_observed_submodel()
        empirical = joint_model.observed_submodel._get_sample(1, observed=True, differentiable=False)
        return plan.loss(empirical)

    def correct_gradient(self, joint_model, posterior_model, sampler_model, number_samples, input_values={}):
        from brancher_b200 import lowering, _cuda as cu
        plan = lowering.get_particle_plan(joint_model, posterior_model)
        params = plan.parameters()
        theta = plan.stacked()
        grad = torch.stack([p.grad.detach().reshape(-1) for p in params]).contiguous()
        out, bw = cu.svgd_direction(theta, grad)
        self.bandwidth = bw                      # device scalar; float(self.bandwidth) synchronises on demand
        for p, row in zip(params, out):
            p.grad = row.reshape(p.shape).clone()

    def post_process(self, joint_model):
        pass


class MAP(InferenceMethod):
    """Maximum a posteriori (inference.py:251-274): the posterior model holds one learnable RootVariable per latent,
    loss = -log p(data, theta).  The point estimate is a one-particle ensemble of the linear family or of the dense regression
    family at a constant noise scale (K4a: one fused launch for the joint log-probability and its gradient), any scalar model goes
    through the scalar-DAG family (K1)."""

    def __init__(self):
        self.learnable_model = False
        self.needs_sampler = False
        self.learnable_sampler = False

    def _plan(self, joint_model, posterior_model):
        from brancher_b200 import lowering
        try:
            return "particles", lowering.get_particle_plan(joint_model, [posterior_model])
        except lowering.UnsupportedModelError as particle_err:
            try:
                return "dag", lowering.get_plan(joint_model, posterior_model)
            except lowering.UnsupportedModelError as dag_err:
                raise lowering.UnsupportedModelError("MAP: the model is lowered neither as a linear-family point estimate (%s) "
                                                     "nor as a scalar DAG (%s)" % (particle_err, dag_err)) from None

    def check_model_compatibility(self, joint_model, posterior_model, sampler_model):
        from brancher_b200.variables import RootVariable
        assert all(isinstance(var, RootVariable) for var in posterior_model.flatten())
        self._plan(joint_model, posterior_model)

    def compute_loss(self, joint_model, posterior_model, sampler_model, number_samples, input_values={}):
        kind, plan = self._plan(joint_model, posterior_model)
        joint_model.update_observed_submodel()
        empirical = joint_model.observed_submodel._get_sample(1, observed=True, differentiable=False)
        if kind == "particles":
            return plan.loss(empirical)
        return -plan.elbo(1, empirical)          # no q noise, no entropy terms: -ELBO of a point mass is -log p(data, theta)

    def post_process(self, joint_model):
        pass


class WassersteinVariationalGradientDescent(InferenceMethod):
    """WVGD over (sampler, particle) ensembles (inference.py:154-248).  `compute_loss` = sum_k -ELBO(joint, q = sampler k
    truncated to particle k's Voronoi cell) + the importance-weighted squared distance between every particle and its own
    sampler's draws; here it is three fused CUDA stages (K6: sample + Voronoi owner, per-draw log-likelihoods and
    gradients, masked reduction) instead of P^2 Python graph walks per evaluation.

    Same constructor as the reference.  `cost_function` / `deviation_statistics` are not lowered (only the default
    squared-distance cost runs on the GPU); `first_column_only=True` (default) reproduces the reference's numpy cost, which
    for weights of shape [C, F] only sees column 0 (utilities.py:125-126) -- pass False for the full squared distance.
    Deviation: a sampler whose draw has no accepted sample contributes nothing to that term in this evaluation (the
    reference re-draws until one is accepted, transformations.py:33); `accepted` holds the per-sampler counts.
    `post_process` (ensemble weights) re-draws such samplers as the reference does."""

    def __init__(self, variational_samplers, particles, cost_function=None, deviation_statistics=None, biased=False,
                 number_post_samples=20000, gradient_estimator=gradient_estimators.PathwiseDerivativeEstimator,
                 first_column_only=True):
        if cost_function is not None or deviation_statistics is not None:
            raise NotImplementedError("brancher_b200 lowers only the default WVGD cost (squared distance) to CUDA")
        self.gradient_estimator = gradient_estimator
        self.learnable_model = False
        self.needs_sampler = True
        self.learnable_sampler = True
        self.biased = biased
        self.number_post_samples = number_post_samples
        self.first_column_only = first_column_only
        self.particles = list(particles)
        # the reference wraps every sampler with truncate_model (transformations.py:10-69); the truncation rule
        # (argmin_j cost == k) is evaluated by the K6a kernel, so the samplers themselves are kept as they are
        self.sampler_model = list(variational_samplers)
        self.accepted = None
        self.weights = None

    def check_model_compatibility(self, joint_model, posterior_model, sampler_model):
        from collections.abc import Iterable
        from brancher_b200 import lowering
        from brancher_b200.variables import Variable, ProbabilisticModel
        assert isinstance(sampler_model, Iterable) and all(isinstance(s, (Variable, ProbabilisticModel)) for s in sampler_model), \
            "The Wasserstein Variational GD method require a list of variables or probabilistic models as sampler"
        lowering.get_wvgd_plan(joint_model, posterior_model, sampler_model)

    def compute_loss(self, joint_model, posterior_model, sampler_model, number_samples, input_values={}):
        from brancher_b200 import lowering
        plan = lowering.get_wvgd_plan(joint_model, posterior_model, sampler_model)
        joint_model.update_observed_submodel()
        empirical = joint_model.observed_submodel._get_sample(1, observed=True, differentiable=False)
        loss = plan.loss(empirical, number_samples, self.biased, self.first_column_only)
        self.accepted = plan.accepted
        return loss

    def post_process(self, joint_model):
        """Ensemble weights (inference.py:234-247): softmax over samplers of the log normaliser of the importance weights,
        log sum_s exp(log p - log q_k) over `number_post_samples` truncated draws -- evaluated on the device
        (lowering.WvgdPlan.ensemble_weights).  `weights` is a numpy array as in the reference; `log_normalizers` and
        `accepted_post` (accepted draws per sampler) are kept for inspection."""
        from brancher_b200 import lowering
        plan = lowering.get_wvgd_plan(joint_model, self.particles, self.sampler_model)
        joint_model.update_observed_submodel()
        empirical = joint_model.observed_submodel._get_sample(1, observed=True, differentiable=False)
        w, logZ, counts = plan.ensemble_weights(empirical, self.number_post_samples, self.first_column_only)
        self.weights = w.cpu().numpy()
        self.log_normalizers = logZ.cpu().numpy()
        self.accepted_post = counts.cpu().numpy()
