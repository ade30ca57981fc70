"""GPU parity tests of the C-ABI entry points against the oracle (tests/helpers.check_against_oracle)."""
import numpy as np
import pytest
import torch

from helpers import load_golden, mf_params, check_against_oracle, assert_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cu():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from brancher_b200 import _cuda
    _cuda.lib()
    return _cuda


DEV = "cuda:0"


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.asarray(a), dtype=dtype).to(DEV).contiguous()


def dev_offset(a, dtype=torch.float32):
    """a on the device as a contiguous view whose data starts 4 bytes past an allocation (not 16-byte aligned)"""
    t = dev(a, dtype)
    buf = torch.empty(t.numel() + 1, dtype=dtype, device=DEV)
    out = buf[1:].view(t.shape)
    out.copy_(t)
    assert out.data_ptr() % 16 == 4
    return out


def make_vars(cu, params, eps, names, prior=None, shapes=None):
    out = []
    for i, n in enumerate(names):
        mu, rho = params[n]
        e = None if eps is None else dev(eps[n]).reshape(np.asarray(eps[n]).shape[0], -1)
        pl = ps = None
        if prior is not None:
            pl, ps = np.broadcast_to(prior[n][0], np.shape(mu)), np.broadcast_to(prior[n][1], np.shape(mu))
            pl, ps = dev(pl.copy()), dev(ps.copy())
        out.append(cu.MeanFieldVar(dev(mu), dev(rho), var_id=i, prior_loc=pl, prior_scale=ps, eps=e))
    return out


def grads_of(vars_, names, params):
    g = {}
    for v, n in zip(vars_, names):
        g[n + "_loc"] = v.dmu.cpu().numpy().reshape(np.shape(params[n][0]))
        g[n + "_scale"] = v.drho.cpu().numpy().reshape(np.shape(params[n][1]))
    return g


# ---------------------------------------------------------------------------------------------
def test_philox_normals(cu):
    r = cu.sample_range(64, seed=1234, offset=7)
    z = cu.philox_normal(100003, 3, r, DEV)
    assert z.shape == (64, 100003)
    assert abs(z.mean().item()) < 2e-3 and abs(z.var().item() - 1) < 5e-3
    assert abs((z ** 4).mean().item() - 3) < 5e-2          # kurtosis of a normal
    z2 = cu.philox_normal(100003, 3, r, DEV)
    assert torch.equal(z, z2)                               # counter-based: deterministic
    # shard invariance: samples [16,48) generated alone equal rows 16..47 of the full draw
    part = cu.philox_normal(100003, 3, cu.sample_range(64, s0=16, s_local=32, seed=1234, offset=7), DEV)
    assert torch.equal(part, z[16:48])
    other = cu.philox_normal(100003, 4, r, DEV)
    assert abs(torch.corrcoef(torch.stack([z.flatten(), other.flatten()]))[0, 1].item()) < 1e-3


@pytest.mark.parametrize("tied", [True, False])
@pytest.mark.parametrize("numel,S", [(1, 1), (7, 5), (1000, 33)])
def test_mf_prior_entropy(cu, tied, numel, S):
    from oracle import elbo_oracle as O
    rng = np.random.RandomState(numel + S)
    params = {"w": (rng.randn(numel).astype("f4"), rng.randn(numel).astype("f4"))}
    eps = {"w": rng.randn(S, numel).astype("f4")}
    prior = None if tied else {"w": (rng.randn(numel).astype("f4"), (0.5 + rng.rand(numel)).astype("f4"))}
    o32 = O.mean_field_prior_entropy(params, eps, prior)
    o64 = O.mean_field_prior_entropy(params, eps, prior, dtype=torch.float64)
    (v,) = make_vars(cu, params, eps, ["w"], prior)
    loss = cu.mf_normal_prior_entropy(v, cu.sample_range(S))
    check_against_oracle(loss.item(), grads_of([v], ["w"], params), o32, o64, "mf")


BNN_NAMES = ["weights1", "b1", "weights2", "b2"]


def run_bnn(cu, X, y, params, eps, prior=None, r=None, with_prior=True, activation="tanh"):
    S = next(iter(eps.values())).shape[0] if eps is not None else r.s_local
    vars4 = make_vars(cu, params, eps, BNN_NAMES, prior)
    loss = cu.bnn_elbo_fwd_bwd(dev(X), dev(y, torch.int32), vars4, r or cu.sample_range(S), with_prior=with_prior,
                               activation=activation)
    return loss.item(), grads_of(vars4, BNN_NAMES, params), vars4


@pytest.mark.parametrize("name,act", [("bnn_small", "tanh"), ("bnn_small_wide", "tanh"), ("bnn_relu", "relu"), ("bnn_sigmoid", "sigmoid")])
def test_bnn_golden(cu, name, act):
    """CUDA vs the live reference's own outputs and vs the oracle on the same inputs (hidden activation tanh / relu / sigmoid)."""
    from oracle import elbo_oracle as O
    g = load_golden(name)
    params = mf_params(g, BNN_NAMES)
    X, y = g["raw"]["X"], g["raw"]["y"]
    o32 = O.bnn_elbo(X, y, params, g["eps"], activation=act)
    o64 = O.bnn_elbo(X, y, params, g["eps"], dtype=torch.float64, activation=act)
    loss, grads, _ = run_bnn(cu, X, y, params, g["eps"], activation=act)
    check_against_oracle(loss, grads, o32, o64, name)
    # and directly against the reference's fp32 numbers, with the reference's measured noise as slack
    ref = (float(g["raw"]["loss"]), g["grad"])
    check_against_oracle(loss, grads, ref, o64, name + " (reference)")


def random_bnn(seed, B, P, H, C, S, sigma=0.05, mu_scale=0.3):
    rng = np.random.RandomState(seed)
    shapes = {"weights1": (H, P), "b1": (H, 1), "weights2": (C, H), "b2": (C, 1)}
    X = rng.rand(B, P).astype("f4")
    y = rng.randint(0, C, size=B)
    from oracle.elbo_oracle import softplus_inverse
    params = {n: ((mu_scale * rng.randn(*s) / np.sqrt(s[1])).astype("f4"),
                  softplus_inverse(sigma * (1 + rng.rand(*s))).astype("f4")) for n, s in shapes.items()}
    eps = {n: rng.randn(S, *s).astype("f4") for n, s in shapes.items()}
    return X, y, params, eps, shapes


@pytest.mark.parametrize("B,P,H,C,S", [(1, 1, 1, 1, 1), (5, 3, 2, 2, 3), (130, 37, 21, 5, 4), (257, 100, 33, 10, 3),
                                       (64, 784, 100, 10, 2), (129, 130, 129, 16, 2)])
@pytest.mark.parametrize("tied", [True, False])
def test_bnn_random_shapes(cu, B, P, H, C, S, tied):
    """ragged sizes: B not a multiple of the 128-row tile, H/P not multiples of 4, C up to the maximum."""
    from oracle import elbo_oracle as O
    X, y, params, eps, shapes = random_bnn(B * 7 + H, B, P, H, C, S)
    prior = None if tied else {n: (0.0, 10.0) for n in shapes}
    o32 = O.bnn_elbo(X, y, params, eps, prior)
    o64 = O.bnn_elbo(X, y, params, eps, prior, dtype=torch.float64)
    loss, grads, _ = run_bnn(cu, X, y, params, eps, prior)
    check_against_oracle(loss, grads, o32, o64, "bnn %s" % ((B, P, H, C, S),))


def test_bnn_philox_mode_and_shard_invariance(cu):
    """eps == NULL: the kernel's own Philox normals, exported with brn_philox_normal_fill, fed to the
    oracle; and the sum of two sample shards equals the unsharded evaluation (SURVEY §8e)."""
    from oracle import elbo_oracle as O
    B, P, H, C, S = 96, 50, 12, 4, 10
    X, y, params, _, shapes = random_bnn(5, B, P, H, C, S)
    r = cu.sample_range(S, seed=99, offset=3)
    eps = {n: cu.philox_normal(int(np.prod(shapes[n])), i, r, DEV).cpu().numpy().reshape((S,) + shapes[n])
           for i, n in enumerate(BNN_NAMES)}
    o32 = O.bnn_elbo(X, y, params, eps)
    o64 = O.bnn_elbo(X, y, params, eps, dtype=torch.float64)
    loss, grads, _ = run_bnn(cu, X, y, params, None, r=r)
    check_against_oracle(loss, grads, o32, o64, "bnn philox")
    la, ga, _ = run_bnn(cu, X, y, params, None, r=cu.sample_range(S, s0=0, s_local=4, seed=99, offset=3))
    lb, gb, _ = run_bnn(cu, X, y, params, None, r=cu.sample_range(S, s0=4, s_local=6, seed=99, offset=3))
    assert_close(la + lb, loss, "sharded loss", rtol=1e-6)
    for k in grads:
        assert_close(ga[k] + gb[k], grads[k], "sharded grad " + k, rtol=1e-5, atol=1e-6, scale=np.abs(grads[k]).max())


# ---------------------------------------------------------------------------------------------
def run_linear(cu, X, y, params, eps, lik, C, prior=None, r=None, x_offset=False, y_offset=False):
    """x_offset / y_offset: pass X / y at a 4-byte offset from a 16-byte boundary"""
    S = eps["weights"].shape[0] if eps is not None else r.s_local
    (w,) = make_vars(cu, params, eps, ["weights"], prior)
    yd = (dev_offset if y_offset else dev)(y, torch.float32 if lik == cu.BERNOULLI else torch.int32)
    loss = cu.linear_elbo_fwd_bwd((dev_offset if x_offset else dev)(X), yd, lik, w, C, r or cu.sample_range(S))
    return loss.item(), grads_of([w], ["weights"], params)


@pytest.mark.parametrize("name,tied", [("logreg_tied", True), ("logreg_declared_prior", False)])
def test_logreg_golden(cu, name, tied):
    from oracle import elbo_oracle as O
    g = load_golden(name)
    params = mf_params(g, ["weights"])
    X, y = g["raw"]["X"], g["raw"]["y"]
    prior = None if tied else {"weights": (g["raw"]["prior_loc"], g["raw"]["prior_scale"])}
    o32 = O.logreg_elbo(X, y, params, g["eps"], prior)
    o64 = O.logreg_elbo(X, y, params, g["eps"], prior, dtype=torch.float64)
    loss, grads = run_linear(cu, X, y, params, g["eps"], cu.BERNOULLI, 1, prior)
    check_against_oracle(loss, grads, o32, o64, name)
    check_against_oracle(loss, grads, (float(g["raw"]["loss"]), g["grad"]), o64, name + " (reference)")


def test_softmax_regression_golden(cu):
    from oracle import elbo_oracle as O
    g = load_golden("softmax_reg")
    params = mf_params(g, ["weights"])
    X, y = g["raw"]["X"], g["raw"]["y"]
    o32 = O.logreg_elbo(X, y, params, g["eps"], likelihood="categorical")
    o64 = O.logreg_elbo(X, y, params, g["eps"], likelihood="categorical", dtype=torch.float64)
    loss, grads = run_linear(cu, X, y, params, g["eps"], cu.CATEGORICAL, 3)
    check_against_oracle(loss, grads, o32, o64, "softmax_reg")
    check_against_oracle(loss, grads, (float(g["raw"]["loss"]), g["grad"]), o64, "softmax_reg (reference)")


@pytest.mark.parametrize("N,F,C,S,lik", [(1, 1, 1, 1, "binomial"), (300, 7, 1, 5, "binomial"),
                                         (1000, 128, 1, 130, "binomial"), (5000, 64, 1, 257, "binomial"),
                                         (333, 20, 10, 14, "categorical"), (129, 128, 3, 50, "categorical")])
def test_linear_random_shapes(cu, N, F, C, S, lik):
    from oracle import elbo_oracle as O
    rng = np.random.RandomState(N + F)
    X = rng.randn(N, F).astype("f4")
    y = rng.randint(0, 2 if C == 1 else C, size=N)
    params = {"weights": ((0.3 * rng.randn(C, F)).astype("f4"), (rng.randn(C, F) - 1).astype("f4"))}
    eps = {"weights": rng.randn(S, C, F).astype("f4")}
    prior = {"weights": (0.0, 0.5)}
    o32 = O.logreg_elbo(X, y, params, eps, prior, likelihood=lik)
    o64 = O.logreg_elbo(X, y, params, eps, prior, likelihood=lik, dtype=torch.float64)
    loss, grads = run_linear(cu, X, y, params, eps, cu.BERNOULLI if C == 1 and lik == "binomial" else cu.CATEGORICAL,
                             C, prior)
    check_against_oracle(loss, grads, o32, o64, "linear %s" % ((N, F, C, S, lik),))


@pytest.mark.parametrize("N,F,S,tied", [(1, 4, 1, True), (300, 8, 5, False), (1000, 128, 70, False), (5000, 128, 300, True),
                                         (20000, 64, 130, False)])
@pytest.mark.parametrize("x_offset", [False, True])
def test_linear_tcgen05_variant(cu, monkeypatch, N, F, S, tied, x_offset):
    """K2 on the tensor cores: logits GEMM with the Bernoulli likelihood fused in its epilogue + K-split gradient GEMM; d^T
    crosses HBM as plain fp32 and converter warps split it inside the gradient GEMM.  A 16-byte aligned X is read in place
    by the logits GEMM (its converter warps split it); X at a 4-byte offset is split into a (hi, lo) pair first."""
    from oracle import elbo_oracle as O
    monkeypatch.setenv("BRN_LINEAR_VARIANT", "tcgen05")
    monkeypatch.setenv("BRN_LINEAR_FLASH", "0")           # the staged GEMM pair (the one-pass kernel has its own test below)
    rng = np.random.RandomState(N + F + S)
    X = rng.randn(N, F).astype("f4")
    y = rng.randint(0, 2, size=N)
    params = {"weights": ((0.3 * rng.randn(1, F)).astype("f4"), (rng.randn(1, F) - 1).astype("f4"))}
    eps = {"weights": rng.randn(S, 1, F).astype("f4")}
    prior = None if tied else {"weights": (0.0, 0.5)}
    o32 = O.logreg_elbo(X, y, params, eps, prior, row_chunk=4096)
    o64 = O.logreg_elbo(X, y, params, eps, prior, dtype=torch.float64, row_chunk=4096)
    loss, grads = run_linear(cu, X, y, params, eps, cu.BERNOULLI, 1, prior, x_offset=x_offset)
    assert cu.last_variant() == "tcgen05"
    check_against_oracle(loss, grads, o32, o64, "linear tcgen05 N=%d F=%d S=%d x_offset=%s" % (N, F, S, x_offset))


@pytest.mark.parametrize("N,F,S,tied", [(1, 16, 1, True), (63, 32, 3, False), (64, 16, 128, False), (777, 48, 129, True),
                                         (1000, 128, 70, False), (5000, 128, 300, True), (20000, 64, 130, False),
                                         (130001, 96, 200, False), (9473, 112, 1000, True)])
@pytest.mark.parametrize("mode", ["default", "y_ldg"])
def test_linear_flash_variant(cu, monkeypatch, N, F, S, tied, mode):
    """K2 in one pass over X (linear_flash.cuh): logits MMA -> Bernoulli likelihood -> d tile in tensor memory -> gradient
    MMA, fp16 (hi, lo) operand pairs.  Ragged row blocks, ragged vector tiles, one and two 64-feature boxes, more row
    groups than row blocks.  Modes: the default (16-byte aligned y: the targets ride along with the X block through shared
    memory) and y_ldg (y at a 4-byte offset: targets loaded per lane and broadcast with shuffles)."""
    from oracle import elbo_oracle as O
    monkeypatch.setenv("BRN_LINEAR_VARIANT", "tcgen05")
    rng = np.random.RandomState(N + F + S)
    X = (rng.randn(N, F) * (1 + 3 * rng.rand(1, F))).astype("f4")
    y = rng.randint(0, 2, size=N)
    params = {"weights": ((0.3 * rng.randn(1, F)).astype("f4"), (rng.randn(1, F) - 1).astype("f4"))}
    eps = {"weights": rng.randn(S, 1, F).astype("f4")}
    prior = None if tied else {"weights": (0.0, 0.5)}
    o32 = O.logreg_elbo(X, y, params, eps, prior, row_chunk=4096)
    o64 = O.logreg_elbo(X, y, params, eps, prior, dtype=torch.float64, row_chunk=4096)
    loss, grads = run_linear(cu, X, y, params, eps, cu.BERNOULLI, 1, prior, y_offset=mode == "y_ldg")
    assert cu.last_variant() == "tcgen05-flash"
    check_against_oracle(loss, grads, o32, o64, "linear flash N=%d F=%d S=%d %s" % (N, F, S, mode))


def test_linear_prepared_x(cu, monkeypatch):
    """brn_linear_prepare_x + brn_linear_elbo_fwd_bwd_px: the prepared fp16-pair form of a fixed data matrix gives the same
    numbers as the per-call path, is rebuilt after an in-place write to X (version counter) and for another tensor, and is
    ignored where the one-pass kernel does not apply (categorical likelihood, F not a multiple of 16)."""
    from oracle import elbo_oracle as O
    monkeypatch.setenv("BRN_LINEAR_VARIANT", "tcgen05")
    rng = np.random.RandomState(11)
    N, F, S = 3000, 64, 40
    X = rng.randn(N, F).astype("f4")
    y = rng.randint(0, 2, size=N)
    params = {"weights": ((0.3 * rng.randn(1, F)).astype("f4"), (rng.randn(1, F) - 1).astype("f4"))}
    eps = {"weights": rng.randn(S, 1, F).astype("f4")}
    prior = {"weights": (0.0, 0.5)}
    Xd, yd = dev(X), dev(y.astype("f4"))
    prep = cu.PreparedX()

    def run(Xt):
        (w,) = make_vars(cu, params, eps, ["weights"], prior)
        loss = cu.linear_elbo_fwd_bwd(Xt, yd, cu.BERNOULLI, w, 1, cu.sample_range(S), prepared=prep).item()
        return loss, grads_of([w], ["weights"], params)

    for scale in (1.0, 1.0, 3.0):          # second pass reuses the prepared form; third follows an in-place change of X
        if scale != 1.0:
            Xd.mul_(scale)
        buf_before = prep.buf.data_ptr() if prep.buf is not None else None
        ver_before = prep.version
        loss, grads = run(Xd)
        assert cu.last_variant() == "tcgen05-flash"
        Xs = (X * np.float32(scale)).astype("f4")
        o32 = O.logreg_elbo(Xs, y, params, eps, prior)
        o64 = O.logreg_elbo(Xs, y, params, eps, prior, dtype=torch.float64)
        check_against_oracle(loss, grads, o32, o64, "prepared X (scale %g)" % scale)
        if scale == 1.0 and buf_before is not None:
            assert prep.version == ver_before and prep.buf.data_ptr() == buf_before      # reused, not rebuilt
    X2 = rng.randn(N, F).astype("f4")                                                    # another tensor: rebuilt
    loss, grads = run(dev(X2))
    check_against_oracle(loss, grads, O.logreg_elbo(X2, y, params, eps, prior),
                         O.logreg_elbo(X2, y, params, eps, prior, dtype=torch.float64), "prepared X (new tensor)")
    assert prep.get(dev(rng.randn(50, 20).astype("f4")), cu.BERNOULLI, 1) is None        # F % 16 != 0: no prepared form
    assert prep.get(Xd, cu.CATEGORICAL, 3) is None
    with pytest.raises(cu.BrancherCudaError):
        cu._check(cu.lib().brn_linear_prepare_x(Xd.data_ptr(), N, F, prep.buf.data_ptr(), 16, None), "brn_linear_prepare_x")


@pytest.mark.parametrize("N,F,S,slabs", [(1000, 16, 9, 3), (20000, 128, 96, 4), (700, 8, 5, 50)])
def test_linear_host_fed_pipeline(cu, N, F, S, slabs):
    """linear_elbo_fwd_bwd_host: pinned host rows copied slab by slab on a side stream while the previous slab is being
    evaluated; injected noise, so the result must match the oracle on the whole matrix (ragged last slab, more slabs
    requested than 128-row tiles, both kernel variants)."""
    from oracle import elbo_oracle as O
    rng = np.random.RandomState(N + S)
    X = rng.randn(N, F).astype("f4")
    y = rng.randint(0, 2, size=N).astype("f4")
    params = {"weights": ((0.3 * rng.randn(1, F)).astype("f4"), (rng.randn(1, F) - 1).astype("f4"))}
    eps = {"weights": rng.randn(S, 1, F).astype("f4")}
    prior = {"weights": (0.0, 0.5)}
    o32 = O.logreg_elbo(X, y, params, eps, prior, row_chunk=4096)
    o64 = O.logreg_elbo(X, y, params, eps, prior, dtype=torch.float64, row_chunk=4096)
    (w,) = make_vars(cu, params, eps, ["weights"], prior)
    Xp, yp = torch.tensor(X).pin_memory(), torch.tensor(y).pin_memory()
    for _ in range(2):          # second pass reuses the staging buffers while the first may still be in flight
        w.dmu.zero_(); w.drho.zero_()
        loss = cu.linear_elbo_fwd_bwd_host(Xp, yp, cu.BERNOULLI, w, 1, cu.sample_range(S), torch.device("cuda:0"), slabs=slabs)
        check_against_oracle(loss.item(), grads_of([w], ["weights"], params), o32, o64, "host-fed linear N=%d" % N)
    with pytest.raises(cu.BrancherCudaError):
        cu.linear_elbo_fwd_bwd_host(torch.tensor(X), yp, cu.BERNOULLI, w, 1, cu.sample_range(S), torch.device("cuda:0"))


def test_linear_empty_rows(cu):
    """N = 0: the ELBO is prior + entropy only."""
    from oracle import elbo_oracle as O
    rng = np.random.RandomState(0)
    F, S = 9, 6
    params = {"weights": (rng.randn(1, F).astype("f4"), rng.randn(1, F).astype("f4"))}
    eps = {"weights": rng.randn(S, 1, F).astype("f4")}
    prior = {"weights": (0.0, 0.5)}
    o32 = O.mean_field_prior_entropy(params, eps, prior)
    o64 = O.mean_field_prior_entropy(params, eps, prior, dtype=torch.float64)
    loss, grads = run_linear(cu, np.zeros((0, F), "f4"), np.zeros((0,), "f4"), params, eps, cu.BERNOULLI, 1, prior)
    check_against_oracle(loss, grads, o32, o64, "linear N=0")


# ---------------------------------------------------------------------------------------------
# K3 tcgen05 variant (TMA + 3xTF32 tensor-core GEMMs)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,P,H,C,S", [(128, 32, 100, 10, 2), (64, 784, 100, 10, 2), (300, 100, 104, 4, 3),
                                       (257, 130, 97, 16, 5), (1024, 784, 100, 10, 4), (40, 33, 21, 3, 1),
                                       (130, 37, 5, 2, 4)])
@pytest.mark.parametrize("tied", [True, False])
def test_bnn_tcgen05_variant(cu, monkeypatch, B, P, H, C, S, tied):
    """forward GEMM -> mid kernel on mma.sync 3xTF32 -> backward GEMM -> statistics."""
    from oracle import elbo_oracle as O
    monkeypatch.setenv("BRN_BNN_VARIANT", "tcgen05")
    X, y, params, eps, shapes = random_bnn(B * 3 + H, B, P, H, C, S)
    prior = None if tied else {n: (0.0, 10.0) for n in shapes}
    o32 = O.bnn_elbo(X, y, params, eps, prior)
    o64 = O.bnn_elbo(X, y, params, eps, prior, dtype=torch.float64)
    loss, grads, _ = run_bnn(cu, X, y, params, eps, prior)
    assert cu.last_variant() == "tcgen05"
    check_against_oracle(loss, grads, o32, o64, "bnn tcgen05 %s" % ((B, P, H, C, S),))


def test_bnn_tcgen05_ksplit_tail(cu, monkeypatch):
    """Enough units (7 m-tiles x 22 n-tiles = 154 > 148 CTAs) that the backward GEMM K-splits its 6 tail units over the
    grid and accumulates them with atomics (UnitIter in csrc/umma_gemm.cuh)."""
    from oracle import elbo_oracle as O
    monkeypatch.setenv("BRN_BNN_VARIANT", "tcgen05")
    B, P, H, C, S = 1024, 784, 100, 10, 44
    X, y, params, eps, shapes = random_bnn(77, B, P, H, C, S)
    o32 = O.bnn_elbo(X, y, params, eps, None, sample_chunk=4)
    o64 = O.bnn_elbo(X, y, params, eps, None, dtype=torch.float64, sample_chunk=4)
    loss, grads, _ = run_bnn(cu, X, y, params, eps, None)
    assert cu.last_variant() == "tcgen05"
    check_against_oracle(loss, grads, o32, o64, "bnn tcgen05 k-split tail")


def test_bnn_variants_agree_philox(cu, monkeypatch):
    """Same Philox noise through the SIMT and tcgen05 variants."""
    B, P, H, C, S = 200, 96, 100, 10, 6
    X, y, params, _, shapes = random_bnn(9, B, P, H, C, S)
    r = cu.sample_range(S, seed=5, offset=2)
    out = {}
    for variant in ("simt", "tcgen05"):
        monkeypatch.setenv("BRN_BNN_VARIANT", variant)
        out[variant] = run_bnn(cu, X, y, params, None, r=r)
        assert cu.last_variant() == variant
    assert_close(out["tcgen05"][0], out["simt"][0], "loss", rtol=1e-6)
    for k in out["simt"][1]:
        sc = np.abs(out["simt"][1][k]).max()
        assert_close(out["tcgen05"][1][k], out["simt"][1][k], "grad " + k, rtol=1e-5, atol=2e-6, scale=sc)


@pytest.mark.parametrize("B,P,H,C,S,variant", [(300, 50, 100, 10, 6, "tcgen05"), (77, 33, 21, 4, 5, "simt"), (1024, 784, 100, 10, 8, "tcgen05")])
def test_bnn_predict_matches_forward_oracle(cu, monkeypatch, B, P, H, C, S, variant):
    """brn_bnn_predict (SURVEY 8(f)3): logits of every (posterior sample, row) vs an fp64 forward pass on the re-materialised
    Philox weights; probs = MC mean of the softmax; class draws follow the probabilities (distributional check)."""
    monkeypatch.setenv("BRN_BNN_VARIANT", variant)
    X, y, params, _, shapes = random_bnn(B + H, B, P, H, C, S)
    r = cu.sample_range(S, seed=21, offset=4)
    mv = make_vars(cu, params, None, BNN_NAMES)
    logits, labels, probs = cu.bnn_predict(dev(X), mv, r)
    assert cu.last_variant() == variant
    eps = {n: cu.philox_normal(int(np.prod(shapes[n])), i, r, DEV).cpu().numpy().reshape((S,) + shapes[n]).astype("f8")
           for i, n in enumerate(BNN_NAMES)}
    sp = lambda v: np.log1p(np.exp(v.astype("f8")))
    W = {n: params[n][0].astype("f8")[None] + sp(params[n][1])[None] * eps[n] for n in BNN_NAMES}
    pre = np.einsum("shp,bp->sbh", W["weights1"], X.astype("f8")) + W["b1"][:, None, :, 0]
    a = np.einsum("sch,sbh->sbc", W["weights2"], np.tanh(pre)) + W["b2"][:, None, :, 0]
    assert_close(logits.cpu().numpy(), a, "predict logits", scale=np.abs(a).max())
    e = np.exp(a - a.max(-1, keepdims=True))
    pm = (e / e.sum(-1, keepdims=True)).mean(0)
    assert_close(probs.cpu().numpy(), pm, "predict probs", rtol=1e-5, atol=1e-6)
    lab = labels.cpu().numpy()
    assert lab.shape == (S, B) and lab.min() >= 0 and lab.max() < C
    # class frequencies over all (sample, row) draws vs the mean probability, within 5 sigma
    freq = np.bincount(lab.reshape(-1), minlength=C) / lab.size
    want = (e / e.sum(-1, keepdims=True)).reshape(-1, C).mean(0)
    assert np.all(np.abs(freq - want) <= 5 * np.sqrt(want * (1 - want) / lab.size) + 1e-3), (freq, want)


@pytest.mark.parametrize("act", ["relu", "sigmoid"])
def test_bnn_tcgen05_activations(cu, monkeypatch, act):
    """relu / sigmoid hidden units through the tensor-core variant vs the fp64 oracle.  Relu: the rows whose pre-activations
    come within 1e-5 (relative) of the kink are left out of the statement (see the C5 test)."""
    from oracle import elbo_oracle as O
    monkeypatch.setenv("BRN_BNN_VARIANT", "tcgen05")
    B, P, H, C, S = 200, 64, 100, 7, 4
    X, y, params, eps, shapes = random_bnn(41, B, P, H, C, S)
    if act == "relu":          # keep every pre-activation away from zero: shift the biases by the sign of the pre-activation mean
        W = {n: params[n][0].astype("f8")[None] + np.log1p(np.exp(params[n][1].astype("f8")))[None] * eps[n] for n in BNN_NAMES}
        pre = np.einsum("shp,bp->sbh", W["weights1"], X.astype("f8")) + W["b1"][:, None, :, 0]
        keep = np.abs(pre).min(axis=(0, 2)) > 1e-4
        X, y = X[keep], y[keep]
        assert keep.sum() > B // 2
    o32 = O.bnn_elbo(X, y, params, eps, None, activation=act)
    o64 = O.bnn_elbo(X, y, params, eps, None, dtype=torch.float64, activation=act)
    loss, grads, _ = run_bnn(cu, X, y, params, eps, None, activation=act)
    assert cu.last_variant() == "tcgen05"
    check_against_oracle(loss, grads, o32, o64, "bnn tcgen05 %s" % act)
