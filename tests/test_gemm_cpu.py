"""CPU tests of the GEMM and LayerNorm oracles (oracle/gemm.py, oracle/layernorm.py): the references against torch and autograd, every
input regime's defining property, and the error models: an fp32 emulation of each kernel stays within half of its bounds, and the same
emulation with one defect each falls far outside them (or, where the regime is exact, leaves the exact result).  Also the host-only
tile-variant query and the C ABI's alignment refusals, which fire before any CUDA call."""
import ctypes

import pytest
import torch

from oracle import gemm as G
from oracle import layernorm as LN

EPIS = list(range(7))


# ------------------------------------------------------------------------------------------ an fp32 restatement of the GEMM kernel
def _rtz32(x):
    """float64 -> fp32 rounded toward zero."""
    f = x.float()
    return torch.where(f.double().abs() > x.abs(), torch.nextafter(f, torch.zeros_like(f)), f)


def _pack_rz(v):
    return (v.float().view(torch.int32) & -65536).view(torch.float32).bfloat16()


def _sigmoid(u):
    """0.5 tanh(0.851 u) + 0.5 in fp32, with tanh off by a relative 2^-13 (a quarter of tanh.approx.f32's documented error)."""
    t = torch.tanh(torch.tensor(0.851, dtype=torch.float32) * u) * (1 - 2.0 ** -13)
    return 0.5 * t + 0.5


def emulate(epi, inp, mutation=None):
    """The kernel's arithmetic: 16-product blocks added into an fp32 accumulator with round-toward-zero, then the epilogue in fp32."""
    a, b = inp["a"].double(), inp["b"].double()
    M, K = a.shape
    acc = torch.zeros(M, b.shape[0], dtype=torch.float32)
    for k0 in range(0, K, 16):
        if mutation == "drop_kstep" and k0 == 16 * (K // 32):
            continue
        acc = _rtz32(acc.double() + a[:, k0:k0 + 16] @ b[:, k0:k0 + 16].t())
    pack = _pack_rz if mutation == "pack_rz" else (lambda t: t.bfloat16())
    v = acc
    bias = inp["bias"].float().roll(-32) if mutation == "bias_chunk" else inp["bias"].float()
    if epi in (G.BIAS_BF16, G.BIAS_RESID_F32, G.BIAS_QGELU_BF16):
        v = v + bias
    if epi == G.F32:
        return {"out": v.bfloat16().float() if mutation == "f32_via_bf16" else v}
    if epi == G.BIAS_RESID_F32:
        r = inp["resid"].float()
        v = v + r
        return {"out": v + r if mutation == "resid_twice" else v}
    if epi == G.PATCH_POS_F32:
        g2 = inp["g2"]
        rows, cls = G.patch_rows(M, g2)
        tok = torch.full((M // g2 * (g2 + 1), v.shape[1]), float("nan"))
        tok[cls] = 7.0
        tok[rows - 1 if mutation == "patch_remap" else rows] = v + inp["pos"].float()[1 + torch.arange(M) % g2]
        return {"out": tok[rows], "cls_intact": bool((tok[cls] == 7.0).all())}
    if epi == G.BIAS_QGELU_BF16:
        return {"aux": pack(v), "out": pack(v * _sigmoid(v))}
    if epi == G.DQGELU_BF16:
        u = inp["aux"].float()
        s = _sigmoid(u)
        g = s if mutation == "dqgelu_sigmoid" else s * torch.addcmul(torch.ones_like(u), 1.702 * u, 1 - s)
        return {"out": pack(v * g)}
    return {"out": pack(v)}


def _judge(epi, inp, mutation=None):
    got = emulate(epi, inp, mutation)
    ref = G.reference(epi, inp)
    r = G.ratios(got, ref)
    if not got.get("cls_intact", True):
        r["cls"] = float("inf")
    return r, (G.inexact(epi, got, ref) if inp["exact"] else 0)


def _shape(regime):
    return (256, 256, 256, 64) if regime == "sweep" else (200, 256, 512, 40)


# ------------------------------------------------------------------------------------------ the reference
def test_reference_matches_torch_and_autograd():
    inp = G.gauss(130, 256, 192, 3, g2=13)
    a, b = inp["a"].double(), inp["b"].double()
    acc = a @ b.t()
    assert torch.equal(G.reference(G.F32, inp)["out"][0], acc)
    torch.testing.assert_close(G.reference(G.BIAS_RESID_F32, inp)["out"][0], acc + inp["bias"].double() + inp["resid"].double(),
                               rtol=1e-15, atol=1e-15)
    patch = G.reference(G.PATCH_POS_F32, inp)["out"][0]
    assert torch.equal(patch[27], acc[27] + inp["pos"].double()[1 + 27 % 13])
    u = (acc + inp["bias"].double()).requires_grad_()
    h = u * torch.sigmoid(1.702 * u)
    ref = G.reference(G.BIAS_QGELU_BF16, inp)
    torch.testing.assert_close(ref["out"][0], h.detach(), rtol=1e-15, atol=1e-15)
    w = inp["aux"].double().requires_grad_()
    (gw,) = torch.autograd.grad((w * torch.sigmoid(1.702 * w)).sum(), w)
    torch.testing.assert_close(G.reference(G.DQGELU_BF16, inp)["out"][0], acc * gw, rtol=1e-13, atol=1e-15)
    # the slope constant of the QuickGELU bound
    x = torch.linspace(-30, 30, 600001, dtype=torch.float64)
    assert G.qgelu_grad(x).abs().max().item() <= G.QGELU_SLOPE


def test_bf16_cell_is_the_rounding_preimage():
    g = torch.Generator().manual_seed(0)
    x = torch.cat([torch.randn(20000, generator=g, dtype=torch.float64) * 10.0 ** torch.randint(-30, 30, (20000,), generator=g),
                   torch.tensor([0.0, -0.0, 1.0, -1.0, 2.0 ** -133, 3e38])])
    x = x.float().double()
    o = x.float().bfloat16()
    lo, hi = G.bf16_cell(o)
    assert ((lo <= x) & (x <= hi)).all()
    # the neighbours' cells do not contain x (except on a shared edge)
    up = (o.view(torch.int16) + 1).view(torch.bfloat16)
    lo2, _ = G.bf16_cell(up[torch.isfinite(up.float()) & (o.float() > 0)])
    assert (lo2 >= x[torch.isfinite(up.float()) & (o.float() > 0)]).all()


@pytest.mark.parametrize("regime", list(G.REGIMES))
def test_regime_inputs(regime):
    """Every generator checks its own property (an AssertionError here is a broken regime) and returns what the kernel reads."""
    M, N, K, g2 = _shape(regime)
    inp = G.make_inputs(regime, M, N, K, 4, g2=g2)
    assert inp["a"].dtype == torch.bfloat16 and inp["a"].shape == (M, K) and inp["b"].shape == (N, K)
    assert inp["bias"].dtype == torch.float32 and inp["bias"].shape == (N,) and inp["pos"].shape == (g2 + 1, N)
    assert inp["resid"].dtype == torch.float32 and inp["aux"].dtype == torch.bfloat16 and inp["aux"].shape == (M, N)
    assert inp["exact"] == (regime in ("exact", "sweep"))
    if inp["exact"]:
        for epi in G.EXACT_OUTPUTS:
            r = G.reference(epi, inp)
            for name in G.EXACT_OUTPUTS[epi]:
                G.rne_bf16(r[name][0])  # asserts that every exactly computable output is an fp32 value


def test_gauss_keeps_the_original_draws():
    g = torch.Generator().manual_seed(1)
    a = (torch.randn(200, 192, generator=g) * 0.5).bfloat16()
    b = (torch.randn(384, 192, generator=g) * (192 ** -0.5)).bfloat16()
    bias = torch.randn(384, generator=g) * 0.1
    inp = G.gauss(200, 384, 192, 1)
    assert torch.equal(inp["a"], a) and torch.equal(inp["b"], b) and torch.equal(inp["bias"], bias)


def test_sweep_reaches_the_quickgelu_tail_and_both_tie_directions():
    inp = G.sweep(256, 256, 256, 1, g2=64)
    u = G.reference(G.BIAS_QGELU_BF16, inp)["aux"][0]
    assert u.min().item() <= -15.9 and u.max().item() >= 15.9 and (u[:, :-G.TIE_COLS].unique().numel() >= 2000)  # every bf16 multiple of 2^-10 in [-16, 16]
    assert inp["aux"].float().min().item() <= -15.9 and inp["aux"].float().max().item() >= 15.9


@pytest.mark.parametrize("regime", list(G.REGIMES))
@pytest.mark.parametrize("epi", EPIS)
def test_emulated_kernel_stays_within_half_the_bounds(epi, regime):
    M, N, K, g2 = _shape(regime)
    r, bad = _judge(epi, G.make_inputs(regime, M, N, K, 5, g2=g2))
    assert max(r.values()) <= 0.5 and bad == 0, (r, bad)


def test_accumulation_bound_at_long_k():
    """The documented ratios of the accumulation bound at K = 4096 (CPU emulation)."""
    inp = G.gauss(64, 128, 4096, 0)
    ref = G.reference(G.F32, inp)
    assert G.ratios(emulate(G.F32, inp), ref)["out"] <= 0.15
    assert G.ratios(emulate(G.F32, inp, "f32_via_bf16"), ref)["out"] > 10
    assert G.ratios(emulate(G.F32, inp, "drop_kstep"), ref)["out"] > 1000


MUTATIONS = [  # (mutation, epilogue, regime)
    ("f32_via_bf16", G.F32, "gauss"),
    ("pack_rz", G.BF16, "exact"), ("pack_rz", G.BIAS_BF16, "sweep"), ("pack_rz", G.BIAS_QGELU_BF16, "gauss"),
    ("drop_kstep", G.F32, "gauss"), ("drop_kstep", G.BF16, "exact"), ("drop_kstep", G.PATCH_POS_F32, "scaled"),
    ("bias_chunk", G.BIAS_BF16, "gauss"), ("bias_chunk", G.BIAS_RESID_F32, "sweep"), ("bias_chunk", G.BIAS_QGELU_BF16, "scaled"),
    ("patch_remap", G.PATCH_POS_F32, "gauss"), ("patch_remap", G.PATCH_POS_F32, "exact"),
    ("dqgelu_sigmoid", G.DQGELU_BF16, "gauss"), ("dqgelu_sigmoid", G.DQGELU_BF16, "sweep"),
    ("resid_twice", G.BIAS_RESID_F32, "gauss"), ("resid_twice", G.BIAS_RESID_F32, "scaled"),
]


@pytest.mark.parametrize("mutation,epi,regime", MUTATIONS, ids=["%s-%s-%s" % (m, G.EPI_NAMES[e], r) for m, e, r in MUTATIONS])
def test_bounds_reject_a_defective_kernel(mutation, epi, regime):
    M, N, K, g2 = _shape(regime)
    inp = G.make_inputs(regime, M, N, K, 6, g2=g2)
    r, bad = _judge(epi, inp, mutation)
    assert max(r.values()) > 10 or bad > 0, (r, bad)


def test_ties_need_round_to_nearest_even():
    """In the sweep's tie columns a pack that rounds halfway cases away from zero is inexact (and invisible to any tolerance)."""
    inp = G.sweep(256, 256, 256, 2, g2=64)
    ref = G.reference(G.BIAS_BF16, inp)
    v = (inp["a"].double() @ inp["b"].double().t() + inp["bias"].double()).float()
    away = (v.view(torch.int32) + 0x8000) & -65536  # round half away from zero on the magnitude bits
    got = {"out": away.view(torch.float32).bfloat16()}
    assert G.ratios(got, ref)["out"] <= 1.0 and G.inexact(G.BIAS_BF16, got, ref) > 0


# ------------------------------------------------------------------------------------------ LayerNorm
def _ln_emulate(x, gamma, beta, mutation=None):
    D = x.shape[1]
    mean = x.sum(-1) / D
    xc = x - mean[:, None]
    if mutation == "one_pass":
        var = (x * x).sum(-1) / D - mean * mean
    else:
        var = (xc * xc).sum(-1) / (D - 1 if mutation == "unbiased" else D)
    rstd = 1.0 / (var.sqrt() + LN.EPS) if mutation == "eps_outside" else torch.rsqrt(var + LN.EPS)
    y = xc * rstd[:, None] * gamma + beta
    return y, mean, rstd


def _ln_bwd_emulate(dy, x, gamma, mean, rstd, prev):
    D = x.shape[1]
    xh = (x - mean[:, None]) * rstd[:, None]
    dh = dy * gamma
    s1 = dh.sum(-1, keepdim=True) / D
    s2 = (dh * xh).sum(-1, keepdim=True) / D
    dx = rstd[:, None] * (dh - s1 - xh * s2)
    return dx + prev if prev is not None else dx


def _ln_case(regime, D, seed=3, M=64):
    g = torch.Generator().manual_seed(seed)
    x = LN.make_x(regime, M, D, seed)
    gamma = 1 + 0.1 * torch.randn(D, generator=g)
    beta = 0.1 * torch.randn(D, generator=g)
    dy = torch.randn(M, D, generator=g)
    prev = torch.randn(M, D, generator=g)
    return x, gamma, beta, dy, prev


def _ln_fwd_ratios(x, gamma, beta, y, mean, rstd):
    ref = LN.layernorm_fwd(x, gamma, beta)
    r = G.ratios({"y": y, "mean": mean, "rstd": rstd}, {k: (v, b, "f32") for k, (v, b) in ref.items()})
    r["y_bf16"] = G.ratios({"y": y.bfloat16()}, {"y": (*ref["y"], "bf16")})["y"]
    return r


def test_layernorm_reference_matches_autograd():
    x, gamma, beta, dy, _ = _ln_case("gauss", 256)
    x64 = x.double().requires_grad_()
    y = torch.nn.functional.layer_norm(x64, (256,), gamma.double(), beta.double(), LN.EPS)
    (gx,) = torch.autograd.grad((y * dy.double()).sum(), x64)
    ref = LN.layernorm_fwd(x, gamma, beta)
    torch.testing.assert_close(ref["y"][0], y.detach(), rtol=1e-12, atol=1e-12)
    dx, _ = LN.layernorm_bwd(dy, x, gamma, ref["mean"][0], ref["rstd"][0])
    torch.testing.assert_close(dx, gx, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("regime", LN.REGIMES)
@pytest.mark.parametrize("D", [128, 512, 768, 1024, 1280])
def test_layernorm_emulation_stays_within_half_the_bounds(regime, D):
    x, gamma, beta, dy, prev = _ln_case(regime, D)
    y, mean, rstd = _ln_emulate(x, gamma, beta)
    r = _ln_fwd_ratios(x, gamma, beta, y, mean, rstd)
    for p in (None, prev):
        dx = _ln_bwd_emulate(dy, x, gamma, mean, rstd, p)
        ref, b = LN.layernorm_bwd(dy, x, gamma, mean, rstd, p)
        r.update({"dx": G.ratios({"d": dx}, {"d": (ref, b, "f32")})["d"], "dx_bf16": G.ratios({"d": dx.bfloat16()}, {"d": (ref, b, "bf16")})["d"]})
        assert max(r.values()) <= 0.5, r


@pytest.mark.parametrize("mutation,regime", [("one_pass", "offset"), ("unbiased", "gauss"), ("unbiased", "spiky"), ("eps_outside", "constant")])
@pytest.mark.parametrize("D", [128, 768, 1280])
def test_layernorm_bounds_reject_a_defective_forward(mutation, regime, D):
    x, gamma, beta, _, _ = _ln_case(regime, D)
    r = _ln_fwd_ratios(x, gamma, beta, *_ln_emulate(x, gamma, beta, mutation))
    assert max(r.values()) > 10, r


# ------------------------------------------------------------------------------------------ host-only C ABI
def test_tile_variant_query_matches_the_documented_choices():
    from clip_diffusion_b200 import _lib

    q = _lib.load().cg_gemm_tile_variant
    assert q(3136, 768, 3072, _lib.EPI_PATCH_POS_F32) == _lib.GEMM_TILE_PAIR_256x256  # ViT-B/32 patch embedding at 64 cutouts
    assert q(16384, 1024, 640, _lib.EPI_PATCH_POS_F32) == _lib.GEMM_TILE_128x256  # ViT-L/14's
    assert q(200, 384, 192, _lib.EPI_F32) == _lib.GEMM_TILE_128x128  # N % 256 != 0
    assert q(16448, 4096, 1024, _lib.EPI_BIAS_QGELU_BF16) != _lib.GEMM_TILE_PAIR_256x256  # QuickGELU epilogues never pair
    assert q(256, 1024, 4096, _lib.EPI_F32) != _lib.GEMM_TILE_PAIR_256x256  # a pair needs more than 256 rows
    assert q(64, 100, 64, _lib.EPI_F32) < 0 and b"bad sizes" in _lib.load().cg_last_error()


def test_alignment_refusals_fire_without_a_gpu():
    from clip_diffusion_b200 import _lib

    lib = _lib.load()
    P = ctypes.c_void_p
    ok = P(1 << 20)

    def gemm(epi, bias=None, aux=None, pos=None, g2=0):
        return lib.cg_gemm_bf16_tn(ok, ok, 256, 256, 64, 64, 64, epi, bias, ok, aux, 256, pos, g2, None)

    for rc in (gemm(_lib.EPI_BIAS_BF16, bias=P((1 << 20) + 4)), gemm(_lib.EPI_BIAS_RESID_F32, bias=ok, aux=P((1 << 20) + 8)),
               gemm(_lib.EPI_DQGELU_BF16, aux=P((1 << 20) + 2)), gemm(_lib.EPI_PATCH_POS_F32, pos=P((1 << 20) + 12), g2=4)):
        assert rc == -1 and b"16-byte aligned" in lib.cg_last_error()
    m = P(1 << 20)
    for args in ((P((1 << 20) + 4), ok, ok, P((1 << 20) + 64), None), (ok, P((1 << 20) + 8), ok, None, ok),
                 (ok, ok, P((1 << 20) + 12), P((1 << 20) + 64), None), (ok, ok, ok, P((1 << 20) + 36), None), (ok, ok, ok, None, P((1 << 20) + 20))):
        x, gamma, beta, y_bf16, y_f32 = args
        assert lib.cg_layernorm_fwd(x, gamma, beta, 8, 128, 128, y_bf16, y_f32, m, m, None) == -1
        assert b"aligned" in lib.cg_last_error()
    for dy, x, dx, dxb in ((P((1 << 20) + 4), ok, ok, None), (ok, P((1 << 20) + 8), ok, None), (ok, ok, P((1 << 20) + 12), None),
                           (ok, ok, ok, P((1 << 20) + 4))):
        assert lib.cg_layernorm_bwd(dy, x, ok, m, m, 8, 128, 128, 0, dx, dxb, None) == -1
        assert b"aligned" in lib.cg_last_error()
    assert lib.cg_layernorm_bwd(ok, ok, P((1 << 20) + 4), m, m, 8, 128, 128, 0, ok, None, None) == -1
