"""ctypes binding of the C-ABI library (include/brancher_cuda.h) -- the `brancher/_cuda` shim the north
star asks for.  PyTorch is only the carrier of device memory and streams here: every compute call
passes raw device pointers + the current CUDA stream to hand-written sm_100a kernels.

There is NO CPU fallback: `lib()` raises if the shared library is missing, and every wrapper raises if
a tensor is not a CUDA tensor.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbrancher_cuda.so")
ABI_VERSION = 6

_lib = None


class BrancherCudaError(RuntimeError):
    pass


class MFVar(ctypes.Structure):
    """struct brn_mf_var"""
    _fields_ = [("mu", ctypes.c_void_p), ("rho", ctypes.c_void_p),
                ("prior_loc", ctypes.c_void_p), ("prior_scale", ctypes.c_void_p),
                ("eps", ctypes.c_void_p), ("dmu", ctypes.c_void_p), ("drho", ctypes.c_void_p),
                ("numel", ctypes.c_int64), ("var_id", ctypes.c_uint32), ("tied", ctypes.c_int32)]


class SampleRange(ctypes.Structure):
    """struct brn_sample_range"""
    _fields_ = [("s0", ctypes.c_int32), ("s_local", ctypes.c_int32), ("s_total", ctypes.c_int32),
                ("_pad", ctypes.c_int32), ("seed", ctypes.c_uint64), ("offset", ctypes.c_uint64),
                ("offset_dev", ctypes.c_void_p)]


VAE_MAX_HIDDEN = 6


class DenseLayer(ctypes.Structure):
    """struct brn_dense_layer"""
    _fields_ = [("W", ctypes.c_void_p), ("b", ctypes.c_void_p), ("dW", ctypes.c_void_p), ("db", ctypes.c_void_p),
                ("n_in", ctypes.c_int32), ("n_out", ctypes.c_int32)]


class VaeModel(ctypes.Structure):
    """struct brn_vae_model"""
    _fields_ = [("D", ctypes.c_int32), ("L", ctypes.c_int32), ("n_enc", ctypes.c_int32), ("n_dec", ctypes.c_int32),
                ("sd_offset", ctypes.c_float), ("_pad", ctypes.c_int32),
                ("enc", DenseLayer * VAE_MAX_HIDDEN), ("enc_mean", DenseLayer), ("enc_sd", DenseLayer),
                ("dec", DenseLayer * VAE_MAX_HIDDEN), ("dec_out", DenseLayer)]


class WvgdArgs(ctypes.Structure):
    """struct brn_wvgd_args"""
    _fields_ = [(n, ctypes.c_void_p) for n in
                ("loc", "rho", "theta", "prior_loc", "prior_scale", "owner0", "owner1", "ll0", "ll1", "G0", "eps0", "eps1",
                 "Z0", "Z1", "dloc", "drho", "dtheta", "counts", "loss")] + \
               [(n, ctypes.c_int32) for n in ("P", "S", "d", "rho_per_elem", "biased", "_pad")]


class OptTensor(ctypes.Structure):
    """struct brn_opt_tensor"""
    _fields_ = [("param", ctypes.c_void_p), ("grad", ctypes.c_void_p), ("m", ctypes.c_void_p), ("v", ctypes.c_void_p)]


class OptHyper(ctypes.Structure):
    """struct brn_opt_hyper"""
    _fields_ = [("kind", ctypes.c_int32), ("lr", ctypes.c_float), ("momentum", ctypes.c_float), ("weight_decay", ctypes.c_float),
                ("beta1", ctypes.c_float), ("beta2", ctypes.c_float), ("eps", ctypes.c_float), ("_pad", ctypes.c_int32)]


# name -> (restype, argtypes): every symbol include/brancher_cuda.h declares
SYMBOLS = {
    "brn_abi_version": (ctypes.c_int, []),
    "brn_last_error": (ctypes.c_char_p, []),
    "brn_last_variant": (ctypes.c_char_p, []),
    "brn_profile_enable": (None, [ctypes.c_int]),
    "brn_profile_collect": (ctypes.c_int, []),
    "brn_profile_num_stages": (ctypes.c_int, []),
    "brn_profile_stage": (ctypes.c_char_p, [ctypes.c_int, ctypes.POINTER(ctypes.c_double),
                                            ctypes.POINTER(ctypes.c_longlong)]),
    "brn_profile_reset": (None, []),
    "brn_launch_count": (ctypes.c_longlong, []),
    "brn_gemm_nt_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 3),
    "brn_gemm_nt_3xtf32": (ctypes.c_int, [ctypes.c_void_p] * 3 + [ctypes.c_int] * 3 +
                           [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "brn_philox_normal_fill": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint32,
                                              ctypes.POINTER(SampleRange), ctypes.c_void_p]),
    "brn_mf_normal_prior_entropy": (ctypes.c_int, [ctypes.POINTER(MFVar), ctypes.c_void_p, ctypes.c_void_p,
                                                   ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_void_p]),
    "brn_bnn_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 5),
    "brn_set_data_ready_event": (None, [ctypes.c_void_p]),
    "brn_minibatch_indices": (ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_void_p,
                                             ctypes.c_void_p, ctypes.c_void_p]),
    "brn_bnn_elbo_fwd_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 4 +
                             [ctypes.POINTER(MFVar), ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_size_t,
                              ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_bnn_predict": (ctypes.c_int, [ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.POINTER(MFVar), ctypes.POINTER(SampleRange),
                                       ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p]),
    "brn_bnn_elbo_fwd_bwd_act": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5 +
                                 [ctypes.POINTER(MFVar), ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_size_t,
                                  ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_bnn_deep_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 3 + [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "brn_bnn_deep_elbo_fwd_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 3 +
                                  [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(MFVar), ctypes.POINTER(SampleRange),
                                   ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_bnn_deep_predict": (ctypes.c_int, [ctypes.c_void_p] + [ctypes.c_int] * 3 +
                             [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(MFVar), ctypes.POINTER(SampleRange),
                              ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_linear_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "brn_linear_elbo_fwd_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                               ctypes.c_int, ctypes.c_int, ctypes.POINTER(MFVar),
                                               ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_size_t,
                                               ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_linear_prepared_x_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int]),
    "brn_linear_prepare_x": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t,
                                            ctypes.c_void_p]),
    "brn_linear_elbo_fwd_bwd_px": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                  ctypes.c_int, ctypes.c_int, ctypes.POINTER(MFVar),
                                                  ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_size_t,
                                                  ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_linreg_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int, ctypes.c_int]),
    "brn_linreg_elbo_fwd_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                               ctypes.POINTER(MFVar), ctypes.POINTER(MFVar), ctypes.c_void_p,
                                               ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int,
                                               ctypes.c_void_p, ctypes.c_void_p]),
    "brn_linreg_elbo_fwd_bwd_lik": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                   ctypes.c_int, ctypes.POINTER(MFVar), ctypes.POINTER(MFVar), ctypes.c_void_p,
                                                   ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int,
                                                   ctypes.c_void_p, ctypes.c_void_p]),
    "brn_linreg_vectors_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int, ctypes.c_int]),
    "brn_linreg_particles_loss_grad": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                      ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                      ctypes.c_size_t, ctypes.c_void_p]),
    "brn_linreg_vectors_loglik_grad": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                      ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "brn_svgd_sharded_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "brn_svgd_sharded_offsets": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int] + [ctypes.POINTER(ctypes.c_size_t)] * 4),
    "brn_svgd_sharded_phase": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5 +
                               [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "brn_dag_elbo_fwd_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                            ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                            ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_linear_particles_loss_grad": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                      ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                      ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "brn_linear_particles_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "brn_vae_workspace_bytes": (ctypes.c_size_t, [ctypes.POINTER(VaeModel), ctypes.c_int, ctypes.c_int]),
    "brn_vae_elbo_fwd_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                            ctypes.POINTER(VaeModel), ctypes.c_void_p, ctypes.c_uint32,
                                            ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int,
                                            ctypes.c_void_p, ctypes.c_void_p]),
    "brn_wvgd_sample_assign": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p] +
                               [ctypes.c_int] * 6 + [ctypes.POINTER(SampleRange), ctypes.c_void_p, ctypes.c_void_p,
                                                     ctypes.c_void_p, ctypes.c_void_p]),
    "brn_linear_vectors_loglik_grad": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                      ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_wvgd_reduce": (ctypes.c_int, [ctypes.POINTER(WvgdArgs), ctypes.c_void_p]),
    "brn_opt_step": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.POINTER(OptHyper),
                                    ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                    ctypes.c_void_p]),
    "brn_allreduce_oneshot": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "brn_svgd_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "brn_svgd_direction": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5 +
                           [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
}


def lib():
    """Load (once) and return the C-ABI library; raise loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BrancherCudaError(
                "%s not found: build it with `python -m brancher_b200._cuda.build` "
                "(brancher_b200 has no CPU fallback for the ELBO hot path)" % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.brn_abi_version() != ABI_VERSION:
            raise BrancherCudaError("ABI mismatch: library %d, binding %d" % (handle.brn_abi_version(), ABI_VERSION))
        _lib = handle
    return _lib


def _check(status, what):
    if status != 0:
        raise BrancherCudaError("%s failed (%d): %s" % (what, status, lib().brn_last_error().decode()))


def profile_enable(on=True):
    lib().brn_profile_enable(int(on))


def profile_reset():
    lib().brn_profile_reset()


def profile_collect():
    """{stage: (total_ms, calls)} accumulated since the last reset (synchronises the recorded events)."""
    _check(lib().brn_profile_collect(), "brn_profile_collect")
    out = {}
    for i in range(lib().brn_profile_num_stages()):
        ms, calls = ctypes.c_double(), ctypes.c_longlong()
        name = lib().brn_profile_stage(i, ctypes.byref(ms), ctypes.byref(calls))
        out[name.decode()] = (ms.value, calls.value)
    return out


def launch_count():
    return lib().brn_launch_count()


def last_variant():
    return lib().brn_last_variant().decode()


def _ptr(t, dtype=torch.float32, what="tensor"):
    if t is None:
        return None
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise BrancherCudaError("%s must be a CUDA tensor (no CPU fallback)" % what)
    if t.dtype != dtype or not t.is_contiguous():
        raise BrancherCudaError("%s must be contiguous %s, got %s contiguous=%s" % (what, dtype, t.dtype, t.is_contiguous()))
    return t.data_ptr()


def _stream(device):
    return torch.cuda.current_stream(device).cuda_stream


_workspaces = {}


def _workspace(device, nbytes):
    """Grow-only scratch buffer per device (kernels are stream-ordered on the current stream)."""
    key = (device.type, device.index)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


class MeanFieldVar:
    """Host-side description of one `brn_mf_var`.  mu/rho are flat views of the `<name>_loc` /
    `<name>_scale` parameters; dmu/drho receive d loss / d param."""

    def __init__(self, mu, rho, var_id, prior_loc=None, prior_scale=None, eps=None, dmu=None, drho=None):
        self.mu = mu.detach().reshape(-1).contiguous()
        self.rho = rho.detach().reshape(-1).contiguous()
        self.numel = self.mu.numel()
        if self.rho.numel() != self.numel:
            raise BrancherCudaError("MeanFieldVar: rho has %d elements, mu has %d" % (self.rho.numel(), self.numel))
        self.var_id = int(var_id)
        self.tied = prior_loc is None
        dev = self.mu.device

        def full(p):
            p = torch.as_tensor(p, dtype=torch.float32, device=dev)
            return p.expand(mu.shape).reshape(-1).contiguous() if p.numel() != self.numel else p.reshape(-1).contiguous()

        self.prior_loc = None if self.tied else full(prior_loc)
        self.prior_scale = None if self.tied else full(prior_scale)
        self.eps = None if eps is None else eps.detach().reshape(-1, self.numel).contiguous()
        # gradient sinks: caller-provided (zeroed) views, e.g. slices of one flat buffer, or fresh zeros
        self.dmu = torch.zeros_like(self.mu) if dmu is None else dmu
        self.drho = torch.zeros_like(self.rho) if drho is None else drho

    def struct(self):
        # validated once per set of tensors: the host-side preamble of a call sits in front of the first launch and is fully
        # exposed whenever the caller synchronises every step (the end-to-end path: ~30 us for the four K3 variables)
        key = tuple(0 if t is None else t.data_ptr() for t in (self.mu, self.rho, self.prior_loc, self.prior_scale, self.eps,
                                                                 self.dmu, self.drho))
        if getattr(self, "_struct_key", None) != key:
            self._struct = MFVar(_ptr(self.mu, what="mu"), _ptr(self.rho, what="rho"),
                                 _ptr(self.prior_loc, what="prior_loc"), _ptr(self.prior_scale, what="prior_scale"),
                                 _ptr(self.eps, what="eps"), _ptr(self.dmu), _ptr(self.drho),
                                 self.numel, self.var_id, int(self.tied))
            self._struct_key = key
        return self._struct


def flat_grad_views(numels, device):
    """One zeroed flat fp32 buffer [dmu_0 | drho_0 | dmu_1 | ...] (each block padded to 4 floats = 16 B) and its
    per-variable (dmu, drho) views: a single memset and a single all-reduce payload instead of 2 per variable.
    The last 4 floats are spare: the multi-GPU reduction carries the fp64 loss there as a (hi, lo) fp32 pair."""
    pad = lambda n: (n + 3) // 4 * 4
    flat = torch.zeros(sum(2 * pad(n) for n in numels) + 4, dtype=torch.float32, device=device)
    views, off = [], 0
    for n in numels:
        views.append((flat[off:off + n], flat[off + pad(n):off + pad(n) + n]))
        off += 2 * pad(n)
    return flat, views


def sample_range(s_total, s0=0, s_local=None, seed=0, offset=0, offset_dev=None):
    """offset_dev: optional int64 CUDA tensor (1 element) whose value is added to `offset` on the device when noise is drawn."""
    s_local = s_total - s0 if s_local is None else s_local
    ptr = None
    if offset_dev is not None:
        if not (offset_dev.is_cuda and offset_dev.dtype == torch.int64 and offset_dev.numel() == 1):
            raise BrancherCudaError("offset_dev must be a 1-element int64 CUDA tensor")
        ptr = offset_dev.data_ptr()
    return SampleRange(int(s0), int(s_local), int(s_total), 0, int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1), ptr)


def _check_eps(v, r):
    if v.eps is not None and v.eps.shape[0] != r.s_local:
        raise BrancherCudaError("eps has %d samples, sample range has %d" % (v.eps.shape[0], r.s_local))


def philox_normal(numel, var_id, r, device):
    """[s_local, numel] standard normals, bit-identical to what the fused kernels generate."""
    out = torch.empty((r.s_local, numel), dtype=torch.float32, device=device)
    _check(lib().brn_philox_normal_fill(_ptr(out), numel, var_id, ctypes.byref(r), _stream(out.device)),
           "brn_philox_normal_fill")
    return out


def mf_normal_prior_entropy(var, r, loss=None):
    """K1a on one MeanFieldVar; accumulates into var.dmu/var.drho; returns the fp64 loss accumulator."""
    dev = var.mu.device
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    _check_eps(var, r)
    st = var.struct()
    _check(lib().brn_mf_normal_prior_entropy(ctypes.byref(st), None, None, ctypes.byref(r),
                                             _ptr(loss, torch.float64), _stream(dev)), "brn_mf_normal_prior_entropy")
    return loss


ACTIVATIONS = {"tanh": 0, "relu": 1, "sigmoid": 2}


def bnn_elbo_fwd_bwd(X, y, vars4, r, with_prior=True, loss=None, data_ready=None, activation="tanh"):
    """K3.  X [B,P] fp32, y [B] int32, vars4 = MeanFieldVar for (weights1 [H,P], b1 [H], weights2 [C,H], b2 [C]).
    data_ready: a torch.cuda.Event recorded on the stream that is still copying X / y to the device; the evaluation waits
    for it only before its first read of the minibatch, so noise generation and weight sampling overlap the copy."""
    dev = X.device
    B, P = X.shape
    H = vars4[1].numel
    C = vars4[3].numel
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    for v in vars4:
        _check_eps(v, r)
    nbytes = lib().brn_bnn_workspace_bytes(B, P, H, C, r.s_local)
    ws = _workspace(dev, nbytes)
    arr = (MFVar * 4)(*[v.struct() for v in vars4])
    if data_ready is not None:
        lib().brn_set_data_ready_event(ctypes.c_void_p(data_ready.cuda_event))
    _check(lib().brn_bnn_elbo_fwd_bwd_act(_ptr(X, what="X"), _ptr(y, torch.int32, "y"), B, P, H, C, ACTIVATIONS[activation], arr,
                                          ctypes.byref(r), ws.data_ptr(), ws.numel(), int(with_prior), _ptr(loss, torch.float64),
                                          _stream(dev)), "brn_bnn_elbo_fwd_bwd")
    return loss


def bnn_predict(X, vars4, r, labels=True, probs=True, activation="tanh"):
    """K3 forward only: posterior-predictive pass for a batch.  Returns (logits [s_local,B,C], labels int32 [s_local,B] or
    None, probs_mean [B,C] or None: this rank's share of the MC average of softmax(logits))."""
    dev = X.device
    B, P = X.shape
    H, C = vars4[1].numel, vars4[3].numel
    nbytes = lib().brn_bnn_workspace_bytes(B, P, H, C, r.s_local)
    ws = _workspace(dev, nbytes)
    arr = (MFVar * 4)(*[v.struct() for v in vars4])
    logits = torch.empty((r.s_local, B, C), dtype=torch.float32, device=dev)
    lab = torch.empty((r.s_local, B), dtype=torch.int32, device=dev) if labels else None
    pm = torch.zeros((B, C), dtype=torch.float32, device=dev) if probs else None
    _check(lib().brn_bnn_predict(_ptr(X, what="X"), B, P, H, C, ACTIVATIONS[activation], arr, ctypes.byref(r), ws.data_ptr(), ws.numel(), _ptr(logits),
                                 _ptr(lab, torch.int32), _ptr(pm), _stream(dev)), "brn_bnn_predict")
    return logits, lab, pm


def _deep_shape(X, vars_, activations):
    """(B, P, H array, act array, C) of a deep BNN: vars_ = MeanFieldVar for (W1, b1, W2, b2, ..., W_out, b_out)."""
    B, P = X.shape
    n_hidden = len(vars_) // 2 - 1
    if len(vars_) % 2 or len(activations) != n_hidden:
        raise BrancherCudaError("deep BNN: %d variables and %d activations do not describe a network" % (len(vars_), len(activations)))
    H = (ctypes.c_int * max(n_hidden, 1))(*[v.numel for v in vars_[1:-2:2]])
    act = (ctypes.c_int * max(n_hidden, 1))(*[ACTIVATIONS[a] for a in activations])
    return B, P, n_hidden, H, act, vars_[-1].numel


def bnn_deep_elbo_fwd_bwd(X, y, vars_, r, activations, with_prior=True, loss=None, data_ready=None):
    """K3 with 2..4 hidden layers.  X [B,P] fp32, y [B] int32, vars_ = MeanFieldVar for (weights1 [H1,P], b1 [H1],
    weights2 [H2,H1], b2 [H2], ..., weights_out [C,H_L], b_out [C]); activations: one of "tanh" / "relu" / "sigmoid" per
    hidden layer.  data_ready as for bnn_elbo_fwd_bwd."""
    dev = X.device
    B, P, n_hidden, H, act, C = _deep_shape(X, vars_, activations)
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    for v in vars_:
        _check_eps(v, r)
    nbytes = lib().brn_bnn_deep_workspace_bytes(B, P, n_hidden, H, C, r.s_local)
    ws = _workspace(dev, nbytes)
    arr = (MFVar * len(vars_))(*[v.struct() for v in vars_])
    if data_ready is not None:
        lib().brn_set_data_ready_event(ctypes.c_void_p(data_ready.cuda_event))
    _check(lib().brn_bnn_deep_elbo_fwd_bwd(_ptr(X, what="X"), _ptr(y, torch.int32, "y"), B, P, n_hidden, H, act, C, arr,
                                           ctypes.byref(r), ws.data_ptr(), ws.numel(), int(with_prior), _ptr(loss, torch.float64),
                                           _stream(dev)), "brn_bnn_deep_elbo_fwd_bwd")
    return loss


def bnn_deep_predict(X, vars_, r, activations, labels=True, probs=True):
    """Posterior-predictive pass of a deep BNN (as bnn_predict): (logits [s_local,B,C], labels int32 [s_local,B] or None,
    probs_mean [B,C] or None)."""
    dev = X.device
    B, P, n_hidden, H, act, C = _deep_shape(X, vars_, activations)
    nbytes = lib().brn_bnn_deep_workspace_bytes(B, P, n_hidden, H, C, r.s_local)
    ws = _workspace(dev, nbytes)
    arr = (MFVar * len(vars_))(*[v.struct() for v in vars_])
    logits = torch.empty((r.s_local, B, C), dtype=torch.float32, device=dev)
    lab = torch.empty((r.s_local, B), dtype=torch.int32, device=dev) if labels else None
    pm = torch.zeros((B, C), dtype=torch.float32, device=dev) if probs else None
    _check(lib().brn_bnn_deep_predict(_ptr(X, what="X"), B, P, n_hidden, H, act, C, arr, ctypes.byref(r), ws.data_ptr(), ws.numel(),
                                      _ptr(logits), _ptr(lab, torch.int32), _ptr(pm), _stream(dev)), "brn_bnn_deep_predict")
    return logits, lab, pm


BERNOULLI, CATEGORICAL, GAUSSIAN = 0, 1, 2
CAUCHY, LAPLACE = 3, 4          # regression likelihoods of linreg_elbo_fwd_bwd (with GAUSSIAN: include/brancher_cuda.h, BRN_LINREG_*)


class PreparedX:
    """The prepared (scaled fp16 pair) form of a fixed data matrix for the one-pass K2 kernel (brn_linear_prepare_x), rebuilt
    only when the matrix changes: a different tensor, or the same tensor after an in-place write (torch's version counter).
    The source tensor is kept referenced, so its memory cannot be handed to another tensor while the prepared form is live."""

    def __init__(self):
        self.buf, self.src, self.version = None, None, None

    def get(self, X, likelihood, C):
        """pointer-carrying uint8 tensor for `px`, or None when this call has no prepared form"""
        N, F = X.shape
        nbytes = lib().brn_linear_prepared_x_bytes(N, F) if (likelihood in (BERNOULLI, GAUSSIAN, CAUCHY, LAPLACE) and C == 1) else 0
        if nbytes == 0 or X.data_ptr() % 16:
            return None
        same = (self.src is not None and self.src.data_ptr() == X.data_ptr() and self.src.shape == X.shape
                and self.src.device == X.device and self.version == X._version)
        if not same:
            if self.buf is None or self.buf.numel() < nbytes or self.buf.device != X.device:
                self.buf = torch.empty(nbytes, dtype=torch.uint8, device=X.device)
            _check(lib().brn_linear_prepare_x(_ptr(X, what="X"), N, F, self.buf.data_ptr(), self.buf.numel(), _stream(X.device)),
                   "brn_linear_prepare_x")
            self.src, self.version = X, X._version
        return self.buf


def linear_elbo_fwd_bwd(X, y, likelihood, w, C, r, with_prior=True, loss=None, prepared=None):
    """K2.  X [N,F] fp32; y [N] fp32 {0,1} (BERNOULLI, C=1) or int32 labels (CATEGORICAL); w MeanFieldVar [C,F].
    prepared: a PreparedX kept by the caller across evaluations of the same data matrix (optional)."""
    dev = X.device
    N, F = X.shape
    if w.numel != C * F:
        raise BrancherCudaError("linear_elbo_fwd_bwd: weights have %d elements, expected C*F = %d*%d" % (w.numel, C, F))
    if y.numel() != N:
        raise BrancherCudaError("linear_elbo_fwd_bwd: y has %d entries for %d rows (labels / targets, not one-hot)" % (y.numel(), N))
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    _check_eps(w, r)
    nbytes = lib().brn_linear_workspace_bytes(N, F, C, r.s_local)
    ws = _workspace(dev, nbytes)
    st = w.struct()
    ydt = torch.float32 if likelihood == BERNOULLI else torch.int32
    px = prepared.get(X, likelihood, C) if (prepared is not None and N > 0) else None
    _check(lib().brn_linear_elbo_fwd_bwd_px(_ptr(X, what="X"), px.data_ptr() if px is not None else None, _ptr(y, ydt, "y"),
                                            likelihood, N, F, C, ctypes.byref(st), ctypes.byref(r), ws.data_ptr(), ws.numel(),
                                            int(with_prior), _ptr(loss, torch.float64), _stream(dev)), "brn_linear_elbo_fwd_bwd_px")
    return loss


def linreg_elbo_fwd_bwd(X, y, w, r, nu=None, noise_scale=None, with_prior=True, loss=None, prepared=None, likelihood=GAUSSIAN):
    """K2g, Bayesian linear regression y ~ Normal(X w, sigma), or the robust Cauchy(X w, sigma) / Laplace(X w, sigma) with
    likelihood=CAUCHY / LAPLACE.  X [N,F] fp32; y [N] fp32; w MeanFieldVar [1,F] (var_id 0).
    Exactly one noise form: nu, a MeanFieldVar of one element read as q = LogNormal(mu, softplus(rho)) with a LogNormal prior
    (var_id 1), or noise_scale, a 1-element fp32 CUDA tensor holding sigma (read on the device at every call).
    prepared: a PreparedX kept by the caller across evaluations of the same data matrix (optional)."""
    dev = X.device
    N, F = X.shape
    if (nu is None) == (noise_scale is None):
        raise BrancherCudaError("linreg_elbo_fwd_bwd: give exactly one of nu and noise_scale")
    if likelihood not in (GAUSSIAN, CAUCHY, LAPLACE):
        raise BrancherCudaError("linreg_elbo_fwd_bwd: unknown likelihood %r (GAUSSIAN, CAUCHY or LAPLACE)" % (likelihood,))
    if w.numel != F:
        raise BrancherCudaError("linreg_elbo_fwd_bwd: weights have %d elements, expected F = %d" % (w.numel, F))
    if y.numel() != N:
        raise BrancherCudaError("linreg_elbo_fwd_bwd: y has %d entries for %d rows" % (y.numel(), N))
    if noise_scale is not None and noise_scale.numel() != 1:
        raise BrancherCudaError("linreg_elbo_fwd_bwd: noise_scale must hold one element")
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    _check_eps(w, r)
    if nu is not None:
        _check_eps(nu, r)
    ws = _workspace(dev, lib().brn_linreg_workspace_bytes(N, F, r.s_local))
    st = w.struct()
    nst = nu.struct() if nu is not None else None
    px = prepared.get(X, likelihood, 1) if (prepared is not None and N > 0) else None
    _check(lib().brn_linreg_elbo_fwd_bwd_lik(_ptr(X, what="X"), px.data_ptr() if px is not None else None, _ptr(y, what="y"),
                                             likelihood, N, F, ctypes.byref(st), ctypes.byref(nst) if nst is not None else None,
                                             _ptr(noise_scale, what="noise_scale"), ctypes.byref(r), ws.data_ptr(), ws.numel(),
                                             int(with_prior), _ptr(loss, torch.float64), _stream(dev)), "brn_linreg_elbo_fwd_bwd")
    return loss


_host_feed = {}


def linear_elbo_fwd_bwd_host(X_host, y_host, likelihood, w, C, r, device, with_prior=True, loss=None, slabs=8):
    """K2 fed from pinned HOST buffers (the minibatch loader's side of the path, distributions.py:410-462): the rows are
    cut into `slabs` slabs and slab i+1 is copied host->device on a side stream while slab i is being evaluated, through
    two device staging buffers.  Every slab call regenerates the same weight samples from the Philox range `r`, the
    gradients and the loss accumulate (+=) across the calls and the prior/entropy terms are counted once, so the result
    equals one call on the whole [N, F] matrix up to fp32 summation order."""
    if not (X_host.is_pinned() and y_host.is_pinned()):
        raise BrancherCudaError("linear_elbo_fwd_bwd_host: X_host and y_host must be pinned host tensors")
    N, F = X_host.shape
    loss = torch.zeros(1, dtype=torch.float64, device=device) if loss is None else loss
    if N == 0:
        return linear_elbo_fwd_bwd(torch.empty((0, F), device=device), torch.empty((0,), dtype=y_host.dtype, device=device),
                                   likelihood, w, C, r, with_prior, loss)
    slabs = max(1, min(int(slabs), (N + 127) // 128))
    rows = ((N + slabs - 1) // slabs + 127) // 128 * 128
    key = (device.type, device.index, rows, F, y_host.dtype)
    st = _host_feed.get(key)
    if st is None:
        st = {"copy": torch.cuda.Stream(device), "X": [torch.empty((rows, F), device=device) for _ in range(2)],
              "y": [torch.empty((rows,), dtype=y_host.dtype, device=device) for _ in range(2)],
              "ready": [torch.cuda.Event() for _ in range(2)], "done": [torch.cuda.Event() for _ in range(2)]}
        _host_feed[key] = st
    main = torch.cuda.current_stream(device)
    st["copy"].wait_stream(main)            # staging buffers may still be read by an earlier evaluation
    i = 0
    for r0 in range(0, N, rows):
        n, b = min(rows, N - r0), i & 1
        with torch.cuda.stream(st["copy"]):
            if i >= 2:
                st["copy"].wait_event(st["done"][b])
            st["X"][b][:n].copy_(X_host[r0:r0 + n], non_blocking=True)
            st["y"][b][:n].copy_(y_host[r0:r0 + n], non_blocking=True)
            st["ready"][b].record(st["copy"])
        main.wait_event(st["ready"][b])
        linear_elbo_fwd_bwd(st["X"][b][:n], st["y"][b][:n], likelihood, w, C, r, with_prior and i == 0, loss)
        st["done"][b].record(main)
        i += 1
    return loss


def minibatch_indices(N, B, device, seed=0, offset=0, return_rounds=False):
    """[B] int64 CUDA tensor of distinct row ids of [0, N), uniformly without replacement, a pure function of
    (N, B, seed, offset) -- the device-side counterpart of np.random.choice(range(N), B, replace=False)."""
    if int(N) <= 0 or int(B) < 0:
        raise BrancherCudaError("minibatch_indices: need N > 0 and B >= 0 (got N=%s B=%s)" % (N, B))
    out = torch.empty((B,), dtype=torch.int64, device=device)
    rounds = torch.zeros(1, dtype=torch.int32, device=device) if return_rounds else None
    _check(lib().brn_minibatch_indices(int(N), int(B), int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1),
                                       _ptr(out, torch.int64, "out"), _ptr(rounds, torch.int32, "rounds"), _stream(device)),
           "brn_minibatch_indices")
    return (out, rounds) if return_rounds else out


def dag_elbo_fwd_bwd(ops, n_ops, n_slots, params, data, n_rows, eps, n_eps, r, loss=None, dparams=None):
    """K1.  ops: uint8 CUDA tensor holding n_ops packed `brn_dag_op` records (24 bytes each); params [n_params] fp32;
    data [n_rows, n_cols] fp32 or None; eps [s_local, n_eps] fp32 or None (Philox).  Returns (loss fp64 [1], dparams)."""
    dev = ops.device
    if ops.dtype != torch.uint8 or ops.numel() != 24 * n_ops:
        raise BrancherCudaError("ops must be a uint8 tensor of %d bytes" % (24 * n_ops))
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    dparams = torch.zeros_like(params) if dparams is None else dparams       # accumulated into (+=): the caller zeroes its own
    n_cols = 0 if data is None else data.shape[1]
    if eps is not None and (eps.shape[0] != r.s_local or eps.shape[1] != n_eps):
        raise BrancherCudaError("eps must be [s_local=%d, n_eps=%d], got %s" % (r.s_local, n_eps, tuple(eps.shape)))
    _check(lib().brn_dag_elbo_fwd_bwd(_ptr(ops, torch.uint8, "ops"), n_ops, n_slots, _ptr(params, what="params"), params.numel(),
                                      _ptr(data, what="data"), n_cols, n_rows, _ptr(eps, what="eps"), n_eps, ctypes.byref(r),
                                      _ptr(dparams), _ptr(loss, torch.float64), _stream(dev)), "brn_dag_elbo_fwd_bwd")
    return loss, dparams


def linear_particles_loss_grad(X, y, likelihood, theta, C, prior_loc=None, prior_scale=None, loss=None):
    """K4a.  theta [n, C*F] particles -> (loss fp64 [1] accumulator, G [n, C*F] = d loss / d theta)."""
    dev = X.device
    N, F = X.shape
    n = theta.shape[0]
    theta = theta.reshape(n, -1)
    if theta.shape[1] != C * F:
        raise BrancherCudaError("linear_particles_loss_grad: particles have %d elements, expected C*F = %d*%d" % (theta.shape[1], C, F))
    if y.numel() != N:
        raise BrancherCudaError("linear_particles_loss_grad: y has %d entries for %d rows" % (y.numel(), N))
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    G = torch.empty_like(theta)
    ydt = torch.float32 if likelihood == BERNOULLI else torch.int32
    nbytes = lib().brn_linear_particles_workspace_bytes(N, F, C, n) if likelihood == BERNOULLI else 0
    ws = _workspace(dev, nbytes) if nbytes else None
    _check(lib().brn_linear_particles_loss_grad(_ptr(X, what="X"), _ptr(y, ydt, "y"), likelihood, N, F, C,
                                                _ptr(theta, what="theta"), n, _ptr(prior_loc, what="prior_loc"),
                                                _ptr(prior_scale, what="prior_scale"), _ptr(G), _ptr(loss, torch.float64),
                                                ws.data_ptr() if ws is not None else None, nbytes,
                                                _stream(dev)), "brn_linear_particles_loss_grad")
    return loss, G


def _regression_args(fn, X, y, likelihood, V, noise_scale):
    N, F = X.shape
    if likelihood not in (GAUSSIAN, CAUCHY, LAPLACE):
        raise BrancherCudaError("%s: unknown likelihood %r (GAUSSIAN, CAUCHY or LAPLACE)" % (fn, likelihood))
    if V.shape[1] != F:
        raise BrancherCudaError("%s: weight vectors have %d elements, expected F = %d" % (fn, V.shape[1], F))
    if y.numel() != N:
        raise BrancherCudaError("%s: y has %d entries for %d rows" % (fn, y.numel(), N))
    if noise_scale is None or noise_scale.numel() != 1:
        raise BrancherCudaError("%s: noise_scale must be a 1-element fp32 CUDA tensor" % fn)


def linreg_particles_loss_grad(X, y, likelihood, theta, noise_scale, prior_loc=None, prior_scale=None, loss=None, prepared=None):
    """K4a for regression particles: y ~ Normal / Cauchy / Laplace(X theta_k, sigma) (likelihood GAUSSIAN / CAUCHY / LAPLACE), theta
    [n, F], noise_scale a 1-element fp32 CUDA tensor holding sigma -> (loss fp64 [1] accumulator, G [n, F] = d loss / d theta) with
    loss += sum_k [-ll_k - log N(theta_k; prior)].  prepared: a PreparedX kept by the caller for a fixed X (optional)."""
    dev = X.device
    N, F = X.shape
    n = theta.shape[0]
    theta = theta.reshape(n, -1) if n else theta.reshape(0, F)
    _regression_args("linreg_particles_loss_grad", X, y, likelihood, theta, noise_scale)
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    G = torch.empty_like(theta)
    ws = _workspace(dev, lib().brn_linreg_vectors_workspace_bytes(N, F, n))
    px = prepared.get(X, likelihood, 1) if (prepared is not None and N > 0) else None
    _check(lib().brn_linreg_particles_loss_grad(_ptr(X, what="X"), px.data_ptr() if px is not None else None, _ptr(y, what="y"),
                                                likelihood, N, F, _ptr(theta, what="theta"), n, _ptr(prior_loc, what="prior_loc"),
                                                _ptr(prior_scale, what="prior_scale"), _ptr(noise_scale, what="noise_scale"), _ptr(G),
                                                _ptr(loss, torch.float64), ws.data_ptr(), ws.numel(), _stream(dev)),
           "brn_linreg_particles_loss_grad")
    return loss, G


def linreg_vectors_loglik_grad(X, y, likelihood, V, noise_scale, want_grad=True, prepared=None):
    """K6b for regression: V [n, F] weight vectors -> (ll fp64 [n], G [n, F] = -d ll / d V or None); arguments as for
    linreg_particles_loss_grad."""
    dev = X.device
    N, F = X.shape
    n = V.shape[0]
    V = V.reshape(n, -1) if n else V.reshape(0, F)
    _regression_args("linreg_vectors_loglik_grad", X, y, likelihood, V, noise_scale)
    ll = torch.empty(n, dtype=torch.float64, device=dev)
    G = torch.empty_like(V) if want_grad else None
    ws = _workspace(dev, lib().brn_linreg_vectors_workspace_bytes(N, F, n))
    px = prepared.get(X, likelihood, 1) if (prepared is not None and N > 0) else None
    _check(lib().brn_linreg_vectors_loglik_grad(_ptr(X, what="X"), px.data_ptr() if px is not None else None, _ptr(y, what="y"),
                                                likelihood, N, F, _ptr(V, what="V"), n, _ptr(noise_scale, what="noise_scale"), _ptr(G),
                                                _ptr(ll, torch.float64), ws.data_ptr(), ws.numel(), _stream(dev)),
           "brn_linreg_vectors_loglik_grad")
    return ll, G


def svgd_direction(theta, grad, row0=0, rows=None, bandwidth=None):
    """K4b.  theta, grad [n, d] (all particles) -> (out [rows, d], bandwidth device float [1]).  bandwidth=None applies
    the reference's median heuristic (inference.py:317-324); pass a device tensor to reuse a fixed bandwidth."""
    n, d = theta.shape
    rows = n - row0 if rows is None else rows
    dev = theta.device
    update = bandwidth is None
    bw = torch.zeros(1, dtype=torch.float32, device=dev) if update else bandwidth
    out = torch.empty((rows, d), dtype=torch.float32, device=dev)
    ws = _workspace(dev, lib().brn_svgd_workspace_bytes(n, d))
    _check(lib().brn_svgd_direction(_ptr(theta, what="theta"), _ptr(grad, what="grad"), n, d, row0, rows, int(update),
                                    _ptr(bw), _ptr(out), ws.data_ptr(), ws.numel(), _stream(dev)), "brn_svgd_direction")
    return out, bw


class ShardedSvgd:
    """K4b for ONE rank's particle rows [row0, row0 + rows) of n (brn_svgd_sharded_phase).  The rank keeps only its rows of
    the distance matrix; between the phases the caller adds `hist` (phases 0-2), then `cnt_le` (SUM) and `next` (MIN) over the
    ranks -- svgd_direction_sharded does that with torch.distributed; the tests drive several instances on one device."""

    def __init__(self, theta, grad, row0, rows, workspace=None):
        n, d = theta.shape
        self.theta, self.grad, self.n, self.d, self.row0, self.rows = theta, grad, n, d, int(row0), int(rows)
        dev = theta.device
        nbytes = lib().brn_svgd_sharded_workspace_bytes(n, d, self.rows)
        if nbytes == 0:
            raise BrancherCudaError("ShardedSvgd: bad shape n=%d d=%d rows=%d" % (n, d, rows))
        self.ws = _workspace(dev, nbytes) if workspace is None else workspace
        offs = [ctypes.c_size_t() for _ in range(4)]
        _check(lib().brn_svgd_sharded_offsets(n, d, self.rows, *[ctypes.byref(o) for o in offs]), "brn_svgd_sharded_offsets")
        h0, hb, c0, x0 = [o.value for o in offs]
        self.hist = self.ws[h0:h0 + hb].view(torch.int32)           # counts < n^2 / 2 < 2^31
        self.cnt_le = self.ws[c0:c0 + 8].view(torch.int64)
        self.next = self.ws[x0:x0 + 4].view(torch.int32)            # bit pattern of a non-negative float: orders like the float
        self.bw = torch.zeros(1, dtype=torch.float32, device=dev)
        self.out = torch.empty((self.rows, d), dtype=torch.float32, device=dev)

    def phase(self, k):
        _check(lib().brn_svgd_sharded_phase(_ptr(self.theta, what="theta"), _ptr(self.grad, what="grad"), self.n, self.d, self.row0,
                                            self.rows, int(k), _ptr(self.bw), _ptr(self.out), self.ws.data_ptr(), self.ws.numel(),
                                            _stream(self.theta.device)), "brn_svgd_sharded_phase")


def svgd_direction_sharded(theta, grad, row0, rows, group=None):
    """K4b with the median selection sharded over the ranks of `group`: theta, grad [n, d] = ALL particles (all-gathered),
    this rank updates rows [row0, row0 + rows).  Five small collectives (3 x 16 KB histogram, 8 + 4 bytes) replace the
    replicated n^2 selection.  Returns (out [rows, d], bandwidth [1]) -- the same numbers as svgd_direction(...)."""
    import torch.distributed as dist
    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    sh = ShardedSvgd(theta, grad, row0, rows)
    for k in range(3):
        sh.phase(k)
        if multi:
            dist.all_reduce(sh.hist, group=group)
    sh.phase(3)
    if multi:
        dist.all_reduce(sh.cnt_le, group=group)
        dist.all_reduce(sh.next, op=dist.ReduceOp.MIN, group=group)
    sh.phase(4)
    return sh.out, sh.bw


def linear_vectors_loglik_grad(X, y, likelihood, V, C, want_grad=True):
    """K6b.  V [n, C*F] weight vectors -> (ll fp64 [n], G [n, C*F] = -d ll / d V or None)."""
    dev = X.device
    N, F = X.shape
    n = V.shape[0]
    V = V.reshape(n, -1)
    ll = torch.empty(n, dtype=torch.float64, device=dev)
    G = torch.empty_like(V) if want_grad else None
    ydt = torch.float32 if likelihood == BERNOULLI else torch.int32
    _check(lib().brn_linear_vectors_loglik_grad(_ptr(X, what="X"), _ptr(y, ydt, "y"), likelihood, N, F, C, _ptr(V, what="V"), n,
                                                _ptr(G), _ptr(ll, torch.float64), _stream(dev)), "brn_linear_vectors_loglik_grad")
    return ll, G


def wvgd_sample_assign(loc, rho, theta, S, F_last, r, draw, eps=None, first_column_only=True):
    """K6a.  loc, theta [P,d]; rho [P] or [P,d]; eps [P,S,d] or None (Philox) -> (Z [P,S,d], eps [P,S,d], owner int32 [P,S])."""
    P, d = loc.shape
    dev = loc.device
    Z = torch.empty((P, S, d), dtype=torch.float32, device=dev)
    eps_out = torch.empty_like(Z) if eps is None else None
    owner = torch.empty((P, S), dtype=torch.int32, device=dev)
    if eps is not None and tuple(eps.shape) != (P, S, d):
        raise BrancherCudaError("eps has shape %s, expected %s" % (tuple(eps.shape), (P, S, d)))
    _check(lib().brn_wvgd_sample_assign(_ptr(loc, what="loc"), _ptr(rho, what="rho"), int(rho.dim() == 2), _ptr(theta, what="theta"),
                                        _ptr(eps, what="eps"), P, S, d, F_last, int(first_column_only), draw, ctypes.byref(r),
                                        _ptr(Z), _ptr(eps_out), _ptr(owner, torch.int32), _stream(dev)), "brn_wvgd_sample_assign")
    return Z, (eps if eps is not None else eps_out), owner


def wvgd_loss_grad(X, y, likelihood, C, loc, rho, theta, S, r, eps0=None, eps1=None, prior=None, biased=False,
                   first_column_only=True, loss=None, noise_scale=None, prepared=None):
    """K6: one WassersteinVariationalGradientDescent.compute_loss + backward (inference.py:203-229) for P (sampler, particle)
    pairs.  loc, theta [P, C*F]; rho [P] or [P, C*F]; prior = (loc [C*F], scale [C*F]) or None (tied).  For the regression
    likelihoods GAUSSIAN / CAUCHY / LAPLACE (C = 1) noise_scale is the 1-element device tensor holding sigma and prepared an
    optional PreparedX, as for linreg_vectors_loglik_grad.
    Returns (loss fp64 [1], dloc [P,d], drho [P,d] per element, dtheta [P,d], counts int32 [P,2])."""
    P, d = loc.shape
    dev = loc.device
    F_last = d // C
    Z0, e0, o0 = wvgd_sample_assign(loc, rho, theta, S, F_last, r, 0, eps0, first_column_only)
    Z1, e1, o1 = wvgd_sample_assign(loc, rho, theta, S, F_last, r, 1, eps1, first_column_only)
    if likelihood in (GAUSSIAN, CAUCHY, LAPLACE):
        ll0, G0 = linreg_vectors_loglik_grad(X, y, likelihood, Z0.reshape(P * S, d), noise_scale, True, prepared)
        ll1, _ = linreg_vectors_loglik_grad(X, y, likelihood, Z1.reshape(P * S, d), noise_scale, False, prepared)
    else:
        ll0, G0 = linear_vectors_loglik_grad(X, y, likelihood, Z0.reshape(P * S, d), C, True)
        ll1, _ = linear_vectors_loglik_grad(X, y, likelihood, Z1.reshape(P * S, d), C, False)
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    dloc, drho, dtheta = torch.empty_like(loc), torch.empty_like(loc), torch.empty_like(loc)
    counts = torch.empty((P, 2), dtype=torch.int32, device=dev)
    a = WvgdArgs()
    a.loc, a.rho, a.theta = _ptr(loc), _ptr(rho), _ptr(theta, what="theta")
    a.prior_loc = None if prior is None else _ptr(prior[0], what="prior_loc")
    a.prior_scale = None if prior is None else _ptr(prior[1], what="prior_scale")
    a.owner0, a.owner1 = _ptr(o0, torch.int32), _ptr(o1, torch.int32)
    a.ll0, a.ll1, a.G0 = _ptr(ll0, torch.float64), _ptr(ll1, torch.float64), _ptr(G0)
    a.eps0, a.eps1, a.Z0, a.Z1 = _ptr(e0), _ptr(e1), _ptr(Z0), _ptr(Z1)
    a.dloc, a.drho, a.dtheta = _ptr(dloc), _ptr(drho), _ptr(dtheta)
    a.counts, a.loss = _ptr(counts, torch.int32), _ptr(loss, torch.float64)
    a.P, a.S, a.d, a.rho_per_elem, a.biased = P, S, d, int(rho.dim() == 2), int(biased)
    _check(lib().brn_wvgd_reduce(ctypes.byref(a), _stream(dev)), "brn_wvgd_reduce")
    return loss, dloc, drho, dtheta, counts


class VaeNet:
    """Host-side description of `brn_vae_model`: lists of (W [n_out,n_in], b [n_out]) CUDA tensors.

    enc = [(W,b), ...] hidden layers, enc_mean / enc_sd = (W,b) heads; dec = [(W,b), ...] hidden layers, dec_out = (W,b).
    Gradients (d loss / d W, d loss / d b) are accumulated into `grads`, a dict with the same structure of zeroed
    tensors (`zero_grads()` makes one flat buffer, so a multi-GPU reduction is a single all-reduce)."""

    def __init__(self, enc, enc_mean, enc_sd, dec, dec_out, sd_offset=0.1):
        c = lambda wb: (wb[0].detach().contiguous(), wb[1].detach().reshape(-1).contiguous())
        self.enc, self.dec = [c(l) for l in enc], [c(l) for l in dec]
        self.enc_mean, self.enc_sd, self.dec_out = c(enc_mean), c(enc_sd), c(dec_out)
        self.sd_offset = float(sd_offset)
        if not (1 <= len(self.enc) <= VAE_MAX_HIDDEN and 1 <= len(self.dec) <= VAE_MAX_HIDDEN):
            raise BrancherCudaError("VAE family: 1..%d hidden layers per network" % VAE_MAX_HIDDEN)
        self.D = self.enc[0][0].shape[1]
        self.L = self.enc_mean[0].shape[0]
        self.flat = None
        self.grads = None

    def layers(self):
        return self.enc + [self.enc_mean, self.enc_sd] + self.dec + [self.dec_out]

    def zero_grads(self):
        dev = self.enc[0][0].device
        pad = lambda n: (n + 3) // 4 * 4
        total = sum(pad(W.numel()) + pad(b.numel()) for W, b in self.layers()) + 4
        if self.flat is None:
            self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
            self.grads, off = [], 0
            for W, b in self.layers():
                gW = self.flat[off:off + W.numel()].view(W.shape); off += pad(W.numel())
                gb = self.flat[off:off + b.numel()]; off += pad(b.numel())
                self.grads.append((gW, gb))
        else:
            self.flat.zero_()
        return self.grads

    def struct(self):
        if self.grads is None:
            self.zero_grads()
        m = VaeModel()
        m.D, m.L, m.n_enc, m.n_dec, m.sd_offset = self.D, self.L, len(self.enc), len(self.dec), self.sd_offset

        def fill(dst, wb, g):
            W, b = wb
            dst.W, dst.b = _ptr(W, what="W"), _ptr(b, what="b")
            dst.dW, dst.db = _ptr(g[0], what="dW"), _ptr(g[1], what="db")
            dst.n_out, dst.n_in = W.shape

        k = 0
        for i, wb in enumerate(self.enc):
            fill(m.enc[i], wb, self.grads[k]); k += 1
        fill(m.enc_mean, self.enc_mean, self.grads[k]); k += 1
        fill(m.enc_sd, self.enc_sd, self.grads[k]); k += 1
        for i, wb in enumerate(self.dec):
            fill(m.dec[i], wb, self.grads[k]); k += 1
        fill(m.dec_out, self.dec_out, self.grads[k])
        return m


def vae_elbo_fwd_bwd(X, net, r, eps=None, var_id=0, row0=0, B_total=None, add_constant=True, loss=None):
    """K5.  X [B,D] fp32 in {0,1}; net: VaeNet (gradients accumulate into net.grads); eps [s_local,B,L] or None (Philox)."""
    dev = X.device
    B, D = X.shape
    if D != net.D:
        raise BrancherCudaError("X has %d columns, the encoder expects %d" % (D, net.D))
    B_total = B if B_total is None else B_total
    loss = torch.zeros(1, dtype=torch.float64, device=dev) if loss is None else loss
    if eps is not None:
        eps = eps.detach().to(torch.float32).contiguous()
        if tuple(eps.shape) != (r.s_local, B, net.L):
            raise BrancherCudaError("eps has shape %s, expected %s" % (tuple(eps.shape), (r.s_local, B, net.L)))
    m = net.struct()
    nbytes = lib().brn_vae_workspace_bytes(ctypes.byref(m), B, r.s_local)
    if nbytes == 0 and r.s_local > 0:
        raise BrancherCudaError("brn_vae_workspace_bytes: %s" % lib().brn_last_error().decode())
    ws = _workspace(dev, nbytes)
    _check(lib().brn_vae_elbo_fwd_bwd(_ptr(X, what="X"), B, int(row0), int(B_total), ctypes.byref(m), _ptr(eps, what="eps"),
                                      int(var_id), ctypes.byref(r), ws.data_ptr(), ws.numel(), int(add_constant),
                                      _ptr(loss, torch.float64), _stream(dev)), "brn_vae_elbo_fwd_bwd")
    return loss


def gemm_nt_3xtf32(A, B):
    """D = A @ B.T on the tcgen05 path (3xTF32); A [M,K], B [N,K] fp32 CUDA tensors."""
    M, K = A.shape
    N = B.shape[0]
    D = torch.empty((M, N), dtype=torch.float32, device=A.device)
    ws = _workspace(A.device, lib().brn_gemm_nt_workspace_bytes(M, N, K))
    _check(lib().brn_gemm_nt_3xtf32(_ptr(A, what="A"), _ptr(B, what="B"), _ptr(D), M, N, K, ws.data_ptr(), ws.numel(),
                                    _stream(A.device)), "brn_gemm_nt_3xtf32")
    return D



SGD, ADAM = 0, 1


class FusedOptimizer:
    """brn_opt_step over a fixed set of (parameter, gradient) tensors: ONE update launch for all of them, the finiteness
    check of the loss, the loss curve and the Philox offset handled on the device (no host synchronisation per iteration).
    params / grads: lists of contiguous fp32 CUDA tensors whose storage stays put (the parameters are updated in place)."""

    def __init__(self, params, grads, kind, lr, momentum=0.0, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8, curve_len=0):
        if not params:
            raise BrancherCudaError("FusedOptimizer: no parameters")
        dev = params[0].device
        self.params, self.grads = list(params), list(grads)
        need_m = kind == ADAM or momentum != 0.0
        self.m = [torch.zeros_like(p) for p in params] if need_m else [None] * len(params)
        self.v = [torch.zeros_like(p) for p in params] if kind == ADAM else [None] * len(params)
        table = (OptTensor * len(params))()
        prefix = [0]
        for i, (p, g) in enumerate(zip(params, grads)):
            if p.numel() != g.numel():
                raise BrancherCudaError("FusedOptimizer: parameter %d and its gradient differ in size" % i)
            table[i] = OptTensor(_ptr(p, what="param"), _ptr(g, what="grad"), _ptr(self.m[i]), _ptr(self.v[i]))
            prefix.append(prefix[-1] + p.numel())
        self.total = prefix[-1]
        self.table = torch.frombuffer(bytearray(bytes(table)), dtype=torch.uint8).to(dev)
        self.prefix = torch.tensor(prefix, dtype=torch.int64).to(dev)
        self.hyper = OptHyper(int(kind), float(lr), float(momentum), float(weight_decay), float(betas[0]), float(betas[1]),
                              float(eps), 0)
        self.counters = torch.zeros(3, dtype=torch.int64, device=dev)       # successful steps, iterations, skipped
        self.curve = torch.zeros(max(int(curve_len), 1), dtype=torch.float32, device=dev)
        self.curve_len = int(curve_len)

    def step(self, loss, offset_dev=None):
        dev = self.table.device
        _check(lib().brn_opt_step(self.table.data_ptr(), self.prefix.data_ptr(), len(self.params), self.total,
                                  ctypes.byref(self.hyper), _ptr(loss, torch.float64, "loss"), self.counters.data_ptr(),
                                  self.curve.data_ptr() if self.curve_len else None, self.curve_len,
                                  None if offset_dev is None else _ptr(offset_dev, torch.int64, "offset_dev"), _stream(dev)),
               "brn_opt_step")
