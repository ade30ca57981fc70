"""GPU parity of K5 (brn_vae_elbo_fwd_bwd) against the live reference's golden vectors and the oracle."""
import numpy as np
import pytest
import torch

from helpers import load_golden, vae_nets, check_against_oracle, assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def cu():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from brancher_b200 import _cuda
    _cuda.lib()
    return _cuda


def dev(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32).to(DEV).contiguous()


def make_net(cu, enc, dec, sd_offset=0.1):
    pair = lambda W, b: (dev(W), dev(b))
    return cu.VaeNet([pair(W, b) for W, b in zip(enc["W"], enc["b"])], pair(enc["W_mean"], enc["b_mean"]),
                     pair(enc["W_sd"], enc["b_sd"]), [pair(W, b) for W, b in zip(dec["W"], dec["b"])],
                     pair(dec["W_out"], dec["b_out"]), sd_offset=sd_offset)


def grads_of(net):
    """keys as oracle.vae_elbo returns them"""
    g, k = {}, 0
    for i in range(len(net.enc)):
        g["enc.W.%d" % i], g["enc.b.%d" % i] = net.grads[k]; k += 1
    g["enc.W_mean"], g["enc.b_mean"] = net.grads[k]; k += 1
    g["enc.W_sd"], g["enc.b_sd"] = net.grads[k]; k += 1
    for i in range(len(net.dec)):
        g["dec.W.%d" % i], g["dec.b.%d" % i] = net.grads[k]; k += 1
    g["dec.W_out"], g["dec.b_out"] = net.grads[k]
    return {n: t.detach().cpu().numpy().copy() for n, t in g.items()}


def random_vae(seed, B, D, L, h_enc, h_dec, S, scale=1.0):
    rng = np.random.RandomState(seed)
    X = (rng.rand(B, D) < 0.5).astype("float32")

    def mlp(dims):
        Ws = [(scale * rng.randn(b, a) / np.sqrt(a)).astype("float32") for a, b in zip(dims[:-1], dims[1:])]
        bs = [(0.1 * rng.randn(b)).astype("float32") for b in dims[1:]]
        return Ws, bs

    eW, eb = mlp([D] + list(h_enc))
    hW, hb = mlp([h_enc[-1], L, L])
    enc = {"W": eW, "b": eb, "W_mean": hW[0], "b_mean": hb[0],
           "W_sd": (rng.randn(L, h_enc[-1]) / np.sqrt(h_enc[-1])).astype("float32"), "b_sd": (0.1 * rng.randn(L)).astype("float32")}
    dW, db = mlp([L] + list(h_dec) + [D])
    dec = {"W": dW[:-1], "b": db[:-1], "W_out": dW[-1], "b_out": db[-1]}
    eps = rng.randn(S, B, L).astype("float32")
    return X, enc, dec, eps


@pytest.mark.parametrize("name", ["vae_small", "vae_deep"])
def test_vae_matches_reference_golden(cu, name):
    """injected noise: loss and every encoder/decoder gradient of the LIVE reference (tests/golden/make_golden.py: vae)."""
    from oracle import elbo_oracle as O
    g = load_golden(name)
    enc, dec = vae_nets(g)
    eps = g["eps"]["z"]
    S = eps.shape[0]
    net = make_net(cu, enc, dec)
    loss = cu.vae_elbo_fwd_bwd(dev(g["raw"]["X"]), net, cu.sample_range(S), eps=dev(eps)).item()
    o64 = O.vae_elbo(g["raw"]["X"], enc, dec, eps, dtype=torch.float64)
    check_against_oracle(loss, grads_of(net), (float(g["raw"]["loss"]), g["grad"]), o64, name)
    assert cu.last_variant() == "tcgen05"


@pytest.mark.parametrize("shape", [dict(B=300, D=100, L=2, h_enc=(48, 64), h_dec=(64, 48), S=5),
                                   dict(B=130, D=784, L=2, h_enc=(256, 512), h_dec=(512, 256), S=3),
                                   dict(B=77, D=50, L=5, h_enc=(40,), h_dec=(33,), S=4),
                                   dict(B=64, D=36, L=16, h_enc=(24, 24, 24), h_dec=(600, 20, 20), S=2)])
def test_vae_matches_oracle(cu, shape):
    """multi-tile shapes (several M/N tiles, K tails, the example's widths, wide first decoder layer, deep nets)."""
    from oracle import elbo_oracle as O
    X, enc, dec, eps = random_vae(21, **shape)
    net = make_net(cu, enc, dec)
    loss = cu.vae_elbo_fwd_bwd(dev(X), net, cu.sample_range(shape["S"]), eps=dev(eps)).item()
    o32 = O.vae_elbo(X, enc, dec, eps)
    o64 = O.vae_elbo(X, enc, dec, eps, dtype=torch.float64)
    check_against_oracle(loss, grads_of(net), o32, o64, "vae %s" % (shape,))


def test_vae_philox_mode_and_shard_invariance(cu):
    """Philox noise: the kernel's own draws, re-materialised with brn_philox_normal_fill, give the oracle's answer; sharding
    the rows (data-parallel ranks) and the samples leaves the summed partials unchanged."""
    from oracle import elbo_oracle as O
    B, D, L, S = 96, 60, 3, 6
    X, enc, dec, _ = random_vae(22, B, D, L, (32, 40), (40, 32), S)
    r = cu.sample_range(S, seed=11, offset=3)
    net = make_net(cu, enc, dec)
    loss = cu.vae_elbo_fwd_bwd(dev(X), net, r, var_id=5).item()
    eps = cu.philox_normal(B * L, 5, r, DEV).cpu().numpy().reshape(S, B, L)
    o64 = O.vae_elbo(X, enc, dec, eps, dtype=torch.float64)
    o32 = O.vae_elbo(X, enc, dec, eps)
    full = grads_of(net)
    check_against_oracle(loss, full, o32, o64, "vae philox")
    # rows split 40 + 56, samples split 2 + 4: four partial evaluations accumulate into the same buffers
    net2 = make_net(cu, enc, dec)
    acc = torch.zeros(1, dtype=torch.float64, device=DEV)
    Xd = dev(X)
    for row0, nb in ((0, 40), (40, 56)):
        for s0, ns in ((0, 2), (2, 4)):
            cu.vae_elbo_fwd_bwd(Xd[row0:row0 + nb].contiguous(), net2, cu.sample_range(S, s0=s0, s_local=ns, seed=11, offset=3),
                                var_id=5, row0=row0, B_total=B, add_constant=(row0 == 0 and s0 == 0), loss=acc)
    assert_close(acc.item(), loss, "sharded loss", rtol=1e-6, atol=1e-6)
    part = grads_of(net2)
    for k in full:
        assert_close(part[k], full[k], "sharded grad " + k, rtol=1e-5, atol=1e-6, scale=np.abs(full[k]).max())


def test_vae_rejects_bad_arguments(cu):
    X, enc, dec, eps = random_vae(23, 8, 10, 2, (6,), (6,), 2)
    net = make_net(cu, enc, dec)
    with pytest.raises(cu.BrancherCudaError):
        cu.vae_elbo_fwd_bwd(dev(X)[:, :9].contiguous(), net, cu.sample_range(2))
    with pytest.raises(cu.BrancherCudaError):
        cu.vae_elbo_fwd_bwd(dev(X), net, cu.sample_range(2), eps=dev(eps[:1]))
    with pytest.raises(cu.BrancherCudaError):
        cu.vae_elbo_fwd_bwd(dev(X).cpu(), net, cu.sample_range(2))
