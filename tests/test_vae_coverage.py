"""Which branches of K5's host code the GPU case table of tests/test_vae_coverage_cuda.py reaches, and the oracle at its shapes.

The functions below restate the selections vae.cu and umma_gemm.cuh make from the model's shape; each cites the lines it
mirrors.  The table walk fails when an edit of the table leaves a branch unreached, before any GPU time is spent."""
import math

import numpy as np
import pytest
import torch

from test_vae_coverage_cuda import CASES, CASE, CHILD_CASES, CHILD_SETTINGS, TRANSPOSED, case_inputs, tail_split_case

SMS = 148              # B200
VAE_BK = 16            # vae.cu:23, K chunk of every K5 GEMM
UG_BM = 128            # umma_gemm.cuh:21, M tile


def pick_bn(N, ew16=True):
    """N tile of the forward, data-gradient, output and K-major weight-gradient GEMMs (vae.cu:330-335): -128 is the 128-wide
    tile with sixteen epilogue warps"""
    if ew16 and N % 128 == 0:
        return -128
    nt = (N + 207) // 208
    per = (N + nt - 1) // nt
    return 128 if per <= 128 else (176 if per <= 176 else 208)


def wgrad_tile(n_in, tile_env=2):
    """N tile of the MN-major weight-gradient GEMM (vae.cu:801-809; BRN_VAE_WGRAD_TILE, default 2)"""
    if tile_env == 1:
        return 128
    return 256 if tile_env == 2 and n_in % 256 == 0 else 128


def umma_regime(BN, M, N, K, sms, BK=VAE_BK):
    """umma_plan with allow_split (umma_gemm.cuh:479-497): "tail" when the T = U % grid units of a last, at most half full
    round are K-split, "all" when every unit is K-split over sms / U CTAs, otherwise "none"."""
    m_tiles, n_tiles, k_chunks = -(-M // UG_BM), -(-N // BN), -(-K // BK)
    U = m_tiles * n_tiles
    grid = min(U, sms)
    T = U % grid
    if U > grid and T > 0 and 2 * T <= grid and k_chunks >= 2 * (grid // T):
        return "tail"
    if 2 * U <= sms and k_chunks >= 2 * (sms // U):
        return "all"
    return "none"


def simt_lp(L):
    """template LP of vae_dec0_bwd_kernel and vae_heads_bwd_kernel (vae.cu:877-880, 893-896)"""
    return 2 if L <= 2 else 4 if L <= 4 else 8 if L <= 8 else 16


def simt_jpt(h0):
    """template JPT of vae_dec0_bwd_kernel (vae.cu:716-717)"""
    return 2 if h0 <= 512 else 4


def vae_gemms(c, sms=SMS, wgrad_mn=True, ew16=True, tile_env=2):
    """(role, layer, tile, regime) of every GEMM brn_vae_elbo_fwd_bwd launches for case `c`, in launch order.
    Roles: forward (vae.cu:822-825, 844-845), output (:851), data_grad and wgrad (:859-870, 899-905).  The weight gradient is
    the MN-major GEMM on wgrad_tile (:795-809) or, with BRN_VAE_WGRAD_MN=0, the K-major one on pick_bn (:811-815); both
    allow the K split.  The forward, output and data-gradient GEMMs run in mode 2, which never splits."""
    B, D, R = c["B"], c["D"], c["S"] * c["B"]
    he, hd = list(c["h_enc"]), list(c["h_dec"])
    out = []

    def wgrad(name, n_out, n_in, rows):
        tile = wgrad_tile(n_in, tile_env) if wgrad_mn else pick_bn(n_in, ew16)
        out.append(("wgrad", name, tile, umma_regime(abs(tile), n_out, n_in, rows, sms)))

    for i, n in enumerate(he):
        out.append(("forward", "enc.%d" % i, pick_bn(n, ew16), None))
    for i in range(1, len(hd)):
        out.append(("forward", "dec.%d" % i, pick_bn(hd[i], ew16), None))
    out.append(("output", "dec.out", pick_bn(D, ew16), None))
    for i in range(len(hd), 0, -1):
        n_out = D if i == len(hd) else hd[i]
        wgrad("dec.out" if i == len(hd) else "dec.%d" % i, n_out, hd[i - 1], R)
        out.append(("data_grad", "dec.out" if i == len(hd) else "dec.%d" % i, pick_bn(hd[i - 1], ew16), None))
    for i in range(len(he) - 1, -1, -1):
        wgrad("enc.%d" % i, he[i], D if i == 0 else he[i - 1], B)
        if i > 0:
            out.append(("data_grad", "enc.%d" % i, pick_bn(he[i - 1], ew16), None))
    return out


def branches(c, sms=SMS, **kw):
    """the set of branch labels case `c` reaches"""
    got = set()
    for role, _, tile, regime in vae_gemms(c, sms, **kw):
        got.add("%s tile %d" % (role, tile))
        if regime:
            got.add("%s split %s" % (role, regime))
    got |= {"LP %d" % simt_lp(c["L"]), "L %d" % c["L"], "JPT %d" % simt_jpt(c["h_dec"][0]), "h0 %d" % c["h_dec"][0],
            "B %d" % c["B"], "D %d" % c["D"], "encoder depth %d" % len(c["h_enc"]), "decoder depth %d" % len(c["h_dec"])}
    return got


GEMM_TILES = ["%s tile %d" % (role, t) for role in ("forward", "data_grad", "output") for t in (-128, 128, 176, 208)]
REQUIRED = (GEMM_TILES + ["wgrad tile 256", "wgrad tile 128", "wgrad split none", "wgrad split tail", "wgrad split all"] +
            ["LP %d" % lp for lp in (2, 4, 8, 16)] + ["L %d" % L for L in (1, 4, 8, 9, 16)] + ["JPT 2", "JPT 4"] +
            ["h0 %d" % h for h in (512, 513, 1024)] + ["B %d" % b for b in (1, 31, 33, 77)] + ["D %d" % d for d in (1, 5)] +
            ["%s depth %d" % (side, n) for side in ("encoder", "decoder") for n in (1, 6)])


def reached(cases, **kw):
    where = {}
    for c in cases:
        for b in branches(c, **kw):
            where.setdefault(b, []).append(c["name"])
    return where


def test_case_table_reaches_every_branch():
    where = reached(CASES)
    for b in REQUIRED:
        print("%-24s %s" % (b, ", ".join(where.get(b, ["-- NOT REACHED --"]))))
    missing = [b for b in REQUIRED if b not in where]
    assert not missing, missing
    # the all-split regime on an input width that is not a multiple of 256 (the 128-wide MN-major tile)
    assert any(g[2] == 128 and g[3] == "all" for c in CASES for g in vae_gemms(c)), "no K-split-all on the 128 tile"
    assert len(CASES) == len(CASE), "case names must be unique"


def test_transposed_subset_reaches_the_wide_tiles():
    """BRN_VAE_WGRAD_MN=0 runs the K-major weight gradients on pick_bn's tiles: the subset reaches -128, 176 and 208 there and
    in every other GEMM role, L = 16, and a K split"""
    where = reached([CASE[n] for n in TRANSPOSED], wgrad_mn=False)
    need = ["%s tile %d" % (role, t) for role in ("forward", "data_grad", "output", "wgrad") for t in (-128, 176, 208)]
    need += ["L 16", "wgrad split all"]
    missing = [b for b in need if b not in where]
    assert not missing, missing


def test_child_settings_change_the_selection():
    """each function-static setting changes a GEMM the child cases launch, so its child process tests something"""
    cases = [CASE[n] for n in CHILD_CASES]
    base = [g for c in cases for g in vae_gemms(c)]
    for var, value in CHILD_SETTINGS:
        if var == "BRN_VAE_EW16":
            alt = [g for c in cases for g in vae_gemms(c, ew16=False)]
            assert alt != base and -128 not in [g[2] for g in alt]
        elif var == "BRN_VAE_CW":          # the 4-converter-warp variant exists for the -128 tile only (vae.cu:342-347)
            assert any(g[2] == -128 and g[0] != "wgrad" for g in base)
        else:
            alt = [g for c in cases for g in vae_gemms(c, tile_env=int(value))]
            assert any(g[2] == 256 for g in base) and all(g[2] != 256 for g in alt if g[0] == "wgrad")


def test_tail_split_case_reaches_the_tail_regime():
    for sms in (SMS, 132, 160, 170):
        c = tail_split_case(sms)
        assert umma_regime(128, c["D"], c["h_dec"][-1], c["S"] * c["B"], sms) == "tail", sms
        assert c["D"] % 128 != 0
    assert tail_split_case(SMS) == CASE["tail_split"] and CASE["tail_split"]["D"] == 2000


def test_mirror_spot_values():
    """values worked out by hand from vae.cu / umma_gemm.cuh"""
    assert [pick_bn(n) for n in (1, 128, 150, 176, 200, 208, 209, 250, 256, 300, 500, 513, 1000, 2000)] == \
        [128, -128, 176, 176, 208, 208, 128, 128, -128, 176, 176, 176, 208, 208]
    assert [pick_bn(n, ew16=False) for n in (256, 512, 1024)] == [128, 176, 208]
    assert umma_regime(128, 2000, 1200, 400, 148) == "tail"          # U = 160, T = 12, 25 K chunks >= 24
    assert umma_regime(128, 2000, 1200, 368, 148) == "none"          # 23 K chunks
    assert umma_regime(256, 784, 1024, 308, 148) == "all"            # U = 28, 20 K chunks >= 10
    assert umma_regime(128, 784, 300, 16, 148) == "none"
    assert [simt_lp(L) for L in (1, 2, 3, 4, 5, 8, 9, 16)] == [2, 2, 4, 4, 8, 8, 16, 16]
    assert [simt_jpt(h) for h in (1, 512, 513, 1024)] == [2, 2, 4, 4]


# ------------------------------------------------------------------------------------------------
# the reference side at the new shapes
# ------------------------------------------------------------------------------------------------
def saturated_fraction(X, enc, dec, eps, sd_offset=0.1, bound=30.0):
    """fraction of decoder logits with |l| > bound (fp64 forward pass)"""
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float64)
    h = t(X)
    for W, b in zip(enc["W"], enc["b"]):
        h = torch.relu(h @ t(W).T + t(b))
    mean = h @ t(enc["W_mean"]).T + t(enc["b_mean"])
    sd = torch.nn.functional.softplus(h @ t(enc["W_sd"]).T + t(enc["b_sd"])) + sd_offset
    g = mean + t(eps) * sd
    for W, b in zip(dec["W"], dec["b"]):
        g = torch.relu(g @ t(W).T + t(b))
    logits = g @ t(dec["W_out"]).T + t(dec["b_out"])
    return float((logits.abs() > bound).double().mean()), float(logits.abs().max())


def oracle_agrees(X, enc, dec, eps, sd_offset=0.1):
    """fp32 and fp64 evaluations are finite and agree to the fp32 accumulation error"""
    from oracle import elbo_oracle as O
    l32, g32 = O.vae_elbo(X, enc, dec, eps, sd_offset=sd_offset)
    l64, g64 = O.vae_elbo(X, enc, dec, eps, sd_offset=sd_offset, dtype=torch.float64)
    assert math.isfinite(l32) and math.isfinite(l64)
    assert abs(l32 - l64) <= 1e-5 * abs(l64) + 1e-5, (l32, l64)
    for k in g64:
        assert np.isfinite(g32[k]).all() and np.isfinite(g64[k]).all(), k
        sc = max(np.abs(g64[k]).max(), 1e-8)
        assert np.abs(g32[k] - g64[k]).max() <= 1e-4 * sc, (k, np.abs(g32[k] - g64[k]).max() / sc)
    return l64


@pytest.mark.parametrize("name", sorted(CASE))
def test_oracle_fp32_matches_fp64_at_table_shapes(name):
    X, enc, dec, eps, kept = case_inputs(CASE[name])
    assert X.shape[0] == CASE[name]["B"]
    oracle_agrees(X, enc, dec, eps)


@pytest.mark.parametrize("sd_offset", [1e-3, 1.0])
def test_oracle_sd_offset(sd_offset):
    """the GPU sd_offset cases: softplus stays well above the offset, and the offset moves the loss far beyond tolerance"""
    from oracle import elbo_oracle as O
    c = dict(name="sd_offset", B=33, D=50, L=8, h_enc=(64,), h_dec=(64,), S=4, seed=120)
    X, enc, dec, eps, kept = case_inputs(c, sd_offset=sd_offset)
    l = oracle_agrees(X, enc, dec, eps, sd_offset=sd_offset)
    l_default = O.vae_elbo(X, enc, dec, eps, dtype=torch.float64)[0]
    assert abs(l - l_default) > 1e-3 * abs(l)


def test_oracle_saturated_logits():
    c = dict(name="saturated", B=40, D=300, L=2, h_enc=(64,), h_dec=(150,), S=4, seed=121)
    X, enc, dec, eps, kept = case_inputs(c, saturate=True)
    frac, top = saturated_fraction(X, enc, dec, eps)
    assert frac > 0.5 and 60 < top < 120, (frac, top)
    oracle_agrees(X, enc, dec, eps)
