"""Float64 reference of the tcgen05 GEMM and its fused epilogues (csrc/vit_gemm.cu), its error model, input regimes that reach the
epilogues' rounding and addressing, and a harness that runs the kernel in guarded buffers (TEST-ONLY, torch; the reference runs on
whatever device the inputs are on).

The kernel: acc[M, N] = A[M, K] . B[N, K]^T with bf16 A, B and fp32 accumulation, then one of the CG_EPI_* epilogues in fp32 registers
(include/clipguide_b200.h).  The reference is fed exactly what the kernel reads: bf16 A, B and DQGELU's aux, fp32 bias, pos and
residual.  It returns per output the float64 value and the bound b of the fp32 value the kernel computes before any bf16 rounding.

Error model, per element, with Mag = |A| . |B|^T:
    acc                 |acc - ref| <= 2^-18 Mag
                        (CPU emulation, tests/test_gemm_cpu.py: 16-product blocks added into an fp32 accumulator with round-toward-zero,
                        a pessimistic model of the tensor core, stay <= 0.15 of this at K = 4096; a bf16 round trip of the result reaches
                        up to 50x, a dropped 16-wide k-step >= 1700x.  These ratios come from emulation, not from the device.)
    bias / pos          + 2^-23 (Mag + |bias|)              one fp32 addition (2x its rounding error, which absorbs the cross terms)
    bias + residual     + 2 * 2^-23 (Mag + |bias| + |resid|)  two fp32 additions
    QuickGELU h         1.1 b_u + (2^-12 + 2^-20) |u|       u = acc + bias with bound b_u; |d h / d u| <= 1.0998.  The kernel evaluates
                        sigmoid(1.702 u) as 0.5 tanh.approx(0.851 u) + 0.5; the PTX ISA gives tanh.approx.f32 a maximum relative error
                        of about 2^-11, so the sigmoid is off by at most 2^-12 ABSOLUTE.  In the negative tail 0.5 tanh + 0.5 cancels:
                        a bound relative to h would be wrong there, so the term is |u| 2^-12 (2^-20 |u| covers the fp32 roundings).
    QuickGELU' g        (2^-12 + 2^-20)(1 + 1.702 |u|)     |dg/ds| = |1 + 1.702 u (1 - 2 s)| <= 1 + 1.702 |u|;  out = acc g:
                        b = b_acc (|g| + b_g) + |acc| b_g + 2^-23 |acc g|
fp32 outputs must satisfy |out - ref| <= b.  bf16 outputs are an interval check: round-to-nearest-even is monotone, so a correct kernel
gives out in [rne(ref - b), rne(ref + b)], i.e. the distance from ref to the set of reals that round to out is <= b.  That distance over
b is the ratio reported for a bf16 output: 0 when out = rne(ref), and far above 1 for an output rounded toward zero or one ulp off.

Input regimes (each generator asserts its defining property on the values the kernel reads):
    gauss   A = 0.5 N(0,1), B = K^-1/2 N(0,1), bias = 0.1 N(0,1) (the draws of the original tests), residual / pos N(0,1), aux 2 N(0,1)
    exact   small integers: |a|, |b| <= 8, integer bias, residual and pos.  Every partial sum is an integer below 2^24, so F32, RESID and
            PATCH_POS must equal the float64 result bit for bit, and BIAS_BF16, BF16 and QGELU's u its RNE rounding (ties included:
            odd integers above 256 are halfway between two bf16 numbers)
    scaled  rows of A and rows of B times powers of two in 2^-30 .. 2^30 (exact in bf16; the last rows of A and the last column chunk
            of B at the extremes): every row and column is judged at its own scale
    sweep   A = identity (M = K), so acc holds chosen bf16 values exactly: a dense grid of multiples of 2^-10 in [-16, 16] (QGELU's
            pre-activation; DQGELU's aux is swept the same way), +-0, and in the last 32 columns acc + bias exactly halfway between two
            bf16 numbers (ties to even, both directions).  Every sum is exact in fp32, so the exactness checks of `exact` apply.
Operands are NaN-tailed (NaN rows after M in A, after N in B, NaN in columns K .. lda), outputs are guarded (oracle.attention.Guarded)
and, with ldo > N, sentinel bits fill the gap columns and must survive.
"""
import json

import torch

from oracle.attention import Guarded, nan_tailed

# CG_EPI_* of include/clipguide_b200.h
BIAS_BF16, BIAS_RESID_F32, BIAS_QGELU_BF16, DQGELU_BF16, F32, BF16, PATCH_POS_F32 = range(7)
EPI_NAMES = {BIAS_BF16: "BIAS_BF16", BIAS_RESID_F32: "BIAS_RESID_F32", BIAS_QGELU_BF16: "BIAS_QGELU_BF16", DQGELU_BF16: "DQGELU_BF16",
             F32: "F32", BF16: "BF16", PATCH_POS_F32: "PATCH_POS_F32"}
F32_OUT = (BIAS_RESID_F32, F32, PATCH_POS_F32)
VARIANTS = {0: "128x256", 1: "128x128", 2: "pair256x256"}  # CG_GEMM_TILE_*

C_ACC = 2.0 ** -18
C_ADD = 2.0 ** -23
SIG_ABS = 2.0 ** -12   # 0.5 x the relative error 2^-11 of tanh.approx.f32 (|tanh| <= 1)
C_ROUND = 2.0 ** -20
QGELU_SLOPE = 1.1      # max |d/du u sigmoid(1.702 u)| = 1.0998


def sigmoid_1702(u):
    return torch.sigmoid(1.702 * u)


def qgelu(u):
    return u * sigmoid_1702(u)


def qgelu_grad(u):
    s = sigmoid_1702(u)
    return s * (1.0 + 1.702 * u * (1.0 - s))


# ---------------------------------------------------------------------------------------------------------------- reference + bounds
def reference(epi, inp):
    """Float64 results and bounds of one epilogue: {output name: (ref [M, N], bound [M, N], "f32" | "bf16")}.  The patch epilogue's
    output is given in compact [M, N] form (row m lands on token row (m / g2)(g2 + 1) + 1 + m % g2)."""
    a, b = inp["a"].double(), inp["b"].double()
    acc = a @ b.t()
    mag = a.abs() @ b.abs().t()
    b_acc = C_ACC * mag
    if epi == F32:
        return {"out": (acc, b_acc, "f32")}
    if epi == BF16:
        return {"out": (acc, b_acc, "bf16")}
    if epi == DQGELU_BF16:
        u = inp["aux"].double()
        g = qgelu_grad(u)
        b_g = (SIG_ABS + C_ROUND) * (1.0 + 1.702 * u.abs())
        val = acc * g
        return {"out": (val, b_acc * (g.abs() + b_g) + acc.abs() * b_g + C_ADD * val.abs(), "bf16")}
    if epi == PATCH_POS_F32:
        g2 = inp["g2"]
        p = inp["pos"].double()[1:g2 + 1].repeat(a.shape[0] // g2, 1)
        return {"out": (acc + p, b_acc + C_ADD * (mag + p.abs()), "f32")}
    bias = inp["bias"].double()
    if epi == BIAS_RESID_F32:
        r = inp["resid"].double()
        return {"out": (acc + bias + r, b_acc + 2 * C_ADD * (mag + bias.abs() + r.abs()), "f32")}
    u = acc + bias
    b_u = b_acc + C_ADD * (mag + bias.abs())
    if epi == BIAS_BF16:
        return {"out": (u, b_u, "bf16")}
    assert epi == BIAS_QGELU_BF16, epi
    return {"aux": (u, b_u, "bf16"), "out": (qgelu(u), QGELU_SLOPE * b_u + (SIG_ABS + C_ROUND) * u.abs(), "bf16")}


EXACT_OUTPUTS = {F32: ("out",), BIAS_RESID_F32: ("out",), PATCH_POS_F32: ("out",), BIAS_BF16: ("out",), BF16: ("out",),
                 BIAS_QGELU_BF16: ("aux",)}  # the outputs that are a correctly rounded exact sum in the `exact` and `sweep` regimes


def bf16_cell(o):
    """[lo, hi]: the reals that round-to-nearest-even takes to the bf16 values o (closed at both ends; +-0 share one cell)."""
    mag = (o.view(torch.int16).to(torch.int32) & 0x7FFF)
    val = lambda m: m.to(torch.int16).view(torch.bfloat16).double()  # noqa: E731
    v = val(mag)
    up = val(mag + 1) - v
    dn = torch.where(mag > 0, v - val((mag - 1).clamp_min(0)), up)
    neg = o.double() < 0
    lo = torch.where(neg, -v - up / 2, v - dn / 2)
    hi = torch.where(neg, -v + dn / 2, v + up / 2)
    return lo, hi


def rne_bf16(x):
    """RNE of float64 values that fp32 holds exactly (torch rounds float64 -> bf16 through fp32)."""
    assert torch.equal(x.float().double(), x), "rne_bf16: value not exact in fp32"
    return x.float().bfloat16()


def ratios(got, ref):
    """Worst err / bound per output (see the module docstring; inf when an output holds a non-finite value)."""
    out = {}
    for name, (r, bound, kind) in ref.items():
        g = got[name].to(r.device)
        if not torch.isfinite(g).all():
            out[name] = float("inf")
            continue
        if kind == "f32":
            d = (g.double() - r).abs()
        else:
            lo, hi = bf16_cell(g.bfloat16())
            d = (lo - r).clamp_min(0) + (r - hi).clamp_min(0)
        q = torch.where(d == 0, torch.zeros_like(d), d / bound)
        out[name] = q.max().item()
    return out


def inexact(epi, got, ref):
    """Elements of the exactly computable outputs that differ from the correctly rounded exact result (exact / sweep regimes)."""
    n = 0
    for name in EXACT_OUTPUTS.get(epi, ()):
        r, _, kind = ref[name]
        want = r if kind == "f32" else rne_bf16(r).double()
        n += int((got[name].double().to(r.device) != want).sum())
    return n


# ---------------------------------------------------------------------------------------------------------------- input regimes
def _gen(seed, device):
    return torch.Generator(device=device).manual_seed(seed)


def _divisor_g2(M, g2):
    assert g2 > 0 and M % g2 == 0, "patch rows: g2=%d must divide M=%d" % (g2, M)
    return g2


def gauss(M, N, K, seed, g2=1, device="cpu"):
    """The original tests' operands (same generator draws as their _mk on the same device) plus residual, pos and DQGELU's aux."""
    g = _gen(seed, device)
    a = (torch.randn(M, K, device=device, generator=g) * 0.5).bfloat16()
    b = (torch.randn(N, K, device=device, generator=g) * (K ** -0.5)).bfloat16()
    bias = torch.randn(N, device=device, generator=g) * 0.1
    resid = torch.randn(M, N, device=device, generator=g)
    pos = torch.randn(g2 + 1, N, device=device, generator=g)
    aux = (torch.randn(M, N, device=device, generator=g) * 2.0).bfloat16()
    assert a.abs().max().item() > 1.0 and torch.isfinite(a.float()).all()
    return {"a": a, "b": b, "bias": bias, "resid": resid, "pos": pos, "aux": aux, "g2": _divisor_g2(M, g2), "exact": False}


def exact(M, N, K, seed, g2=1, device="cpu"):
    g = _gen(seed, device)
    ri = lambda lo, hi, *shape: torch.randint(lo, hi + 1, shape, device=device, generator=g).float()  # noqa: E731
    a, b = ri(-8, 8, M, K).bfloat16(), ri(-8, 8, N, K).bfloat16()
    bias, resid, pos = ri(-64, 64, N), ri(-1000, 1000, M, N), ri(-100, 100, g2 + 1, N)
    aux = (torch.randn(M, N, device=device, generator=g) * 2.0).bfloat16()
    for t in (a, b, bias, resid, pos):
        assert torch.equal(t.float(), t.float().round())
    assert a.abs().max().item() <= 8 and b.abs().max().item() <= 8
    assert 64 * K + 64 + 1000 + 100 < 2 ** 24, "exact: partial sums may leave the integers fp32 holds"
    return {"a": a, "b": b, "bias": bias, "resid": resid, "pos": pos, "aux": aux, "g2": _divisor_g2(M, g2), "exact": True}


SCALE_LOG2 = 30


def scaled(M, N, K, seed, g2=1, device="cpu"):
    g = _gen(seed, device)
    ea = torch.randint(-SCALE_LOG2, SCALE_LOG2 + 1, (M,), device=device, generator=g)
    eb = torch.randint(-SCALE_LOG2, SCALE_LOG2 + 1, (N,), device=device, generator=g)
    ea[-1], ea[-2 if M > 1 else -1] = -SCALE_LOG2, SCALE_LOG2  # tail-tile rows at both extremes
    eb[-32:] = torch.tensor([SCALE_LOG2, -SCALE_LOG2] * 16, device=device)  # and the last column chunk
    ea[0] = SCALE_LOG2 if M > 2 else ea[0]
    a0 = (torch.randn(M, K, device=device, generator=g) * 0.5).bfloat16()
    b0 = (torch.randn(N, K, device=device, generator=g) * (K ** -0.5)).bfloat16()
    sa, sb = torch.exp2(ea.double()), torch.exp2(eb.double())
    a = (a0.double() * sa[:, None]).bfloat16()
    b = (b0.double() * sb[:, None]).bfloat16()
    assert torch.equal(a.double() / sa[:, None], a0.double()) and torch.equal(b.double() / sb[:, None], b0.double()), "scaled: not exact"
    assert ea.min().item() == -SCALE_LOG2 and ea.max().item() == SCALE_LOG2 and eb.min().item() == -SCALE_LOG2
    bias = (torch.randn(N, device=device, generator=g).double() * 0.1 * sb * 2.0 ** -SCALE_LOG2).float()
    resid = (torch.randn(M, N, device=device, generator=g).double() * sa[:, None] * sb[None, :]).float()
    pos = (torch.randn(g2 + 1, N, device=device, generator=g).double() * sb * 2.0 ** -SCALE_LOG2).float()
    aux = (torch.randn(M, N, device=device, generator=g) * 2.0).bfloat16()
    return {"a": a, "b": b, "bias": bias, "resid": resid, "pos": pos, "aux": aux, "g2": _divisor_g2(M, g2), "exact": False}


TIE_COLS = 32


def _grid(n, device):
    """n multiples of 2^-10 in [-16, 16] from a dense linspace, exactly representable in bf16, with +-0 at the front."""
    x = torch.linspace(-16.0, 16.0, n, dtype=torch.float64, device=device)
    x = (torch.round(x * 1024) / 1024).bfloat16().double()
    x[:2] = torch.tensor([0.0, -0.0], dtype=torch.float64, device=device)
    return x


def sweep(M, N, K, seed, g2=1, device="cpu"):
    assert M == K and N > TIE_COLS, "sweep: A is the identity (M = K)"
    g = _gen(seed, device)
    nt = N - TIE_COLS
    acc = torch.empty(M, N, dtype=torch.float64, device=device)
    acc[:, :nt] = _grid(M * nt, device).view(nt, M).t()  # column-major fill: every row and every column spans the grid
    bias = torch.zeros(N, dtype=torch.float64, device=device)
    k = torch.arange(M, device=device)
    for j in range(TIE_COLS):
        e = j % 6 - 2  # binades 2^-2 .. 2^3
        step = 2.0 ** (e - 7)
        vals = (2.0 ** e + (1 + (k * 37 + j) % 127) * step) * torch.where(k % 2 == 0, 1.0, -1.0).double()
        acc[:, nt + j] = vals
        bias[nt + j] = step / 2
    a = torch.eye(M, K, device=device).bfloat16()
    b = acc.t().contiguous().bfloat16()
    assert torch.equal(b.double().t(), acc), "sweep: acc values not bf16"
    perm = torch.randperm(M * N, device=device, generator=g)
    aux = acc.flatten()[perm].view(M, N).bfloat16()
    q = lambda t: (torch.round(t * 1024) / 1024)  # noqa: E731
    resid = q(torch.rand(M, N, device=device, generator=g, dtype=torch.float64) * 32 - 16).float()
    pos = q(torch.rand(g2 + 1, N, device=device, generator=g, dtype=torch.float64) * 32 - 16).float()
    # properties: identity, exact grid, +-0, and ties to even in both directions in the tie columns
    assert torch.equal(a.double(), torch.eye(M, dtype=torch.float64, device=device))
    assert torch.equal(q(acc), acc) and acc.abs().max().item() <= 16
    zeros = acc[:, :nt] == 0
    assert zeros.any() and torch.signbit(acc[:, :nt][zeros]).any() and (~torch.signbit(acc[:, :nt][zeros])).any()
    t = acc[:, nt:] + bias[nt:]
    lo, hi = bf16_cell(t.float().bfloat16())
    assert torch.equal(t.float().double(), t), "sweep: acc + bias not exact in fp32"
    on_edge = (t == lo) | (t == hi)
    assert on_edge.all(), "sweep: a tie column holds a value that is not halfway between two bf16 numbers"
    rounded = t.float().bfloat16().double()
    assert (rounded > t).any() and (rounded < t).any(), "sweep: ties must round both up and down to even"
    return {"a": a, "b": b, "bias": bias.float(), "resid": resid, "pos": pos, "aux": aux, "g2": _divisor_g2(M, g2), "exact": True}


REGIMES = {"gauss": gauss, "exact": exact, "scaled": scaled, "sweep": sweep}


def make_inputs(regime, M, N, K, seed, g2=1, device="cpu"):
    return REGIMES[regime](M, N, K, seed, g2=g2, device=device)


def sigma_error(inp, got, ref):
    """Largest |h / u - sigmoid(1.702 u)| over u <= -1 of a QGELU result: the sigmoid error the kernel's tanh.approx leaves (bf16
    rounding of h adds at most 2^-9 sigmoid there)."""
    u = ref["aux"][0]
    sel = u <= -1.0
    h = got["out"].double().to(u.device)
    return ((h[sel] / u[sel]) - sigmoid_1702(u[sel])).abs().max().item() if sel.any() else 0.0


# ---------------------------------------------------------------------------------------------------------------- kernel harness
# (needs the built library and a GPU)
def tile_variant(M, N, K, epi):
    from clip_diffusion_b200 import _lib

    v = _lib.load().cg_gemm_tile_variant(M, N, K, epi)
    _lib.check(0 if v >= 0 else v, "cg_gemm_tile_variant")
    return v


_PATCH_CLS = 7.0  # the class-token rows of the patch epilogue's token buffer: never written


class _Out:
    """A guarded [rows, ldo] output whose first element sits `offset` elements into the guarded region: NaN in [:, :N], sentinel bits
    in the gap columns [:, N:ldo] and in the `offset` elements in front."""

    def __init__(self, rows, N, ldo, dtype, offset, cls_rows=None):
        self.g = Guarded((offset + rows * ldo,), dtype)
        self.offset, self.N = offset, N
        bits = self.g.t.view(self.g.bits_dtype)
        bits[:offset] = self.g.pattern
        self.full = self.g.t[offset:].view(rows, ldo)
        self.full.view(self.g.bits_dtype)[:, N:] = self.g.pattern
        self.cls_rows = cls_rows
        if cls_rows is not None:
            self.full[cls_rows, :N] = _PATCH_CLS
        self.t = self.full[:, :N]

    def intact(self):
        bits = self.g.t.view(self.g.bits_dtype)
        ok = self.g.guards_intact() and bool((bits[:self.offset] == self.g.pattern).all())
        ok = ok and bool((self.full.view(self.g.bits_dtype)[:, self.N:] == self.g.pattern).all())
        if self.cls_rows is not None:
            ok = ok and bool((self.full[self.cls_rows, :self.N] == _PATCH_CLS).all())
        return ok


def _operand(x, pad_cols, pad_rows=64):
    """bf16 [R, C] on the GPU inside a NaN-filled [R + pad_rows, C + pad_cols] allocation (NaN columns C .. ld and NaN rows after R)."""
    R, C = x.shape
    buf = torch.full((R + pad_rows, C + pad_cols), float("nan"), dtype=x.dtype, device="cuda")
    buf[:R, :C] = x.to("cuda")
    return buf[:R, :C]


def _aux_input(x, ldo, offset):
    """An input read with out's row stride: [M, N] values inside a NaN-filled [M, ldo] allocation starting `offset` elements in."""
    M, N = x.shape
    buf = torch.full((offset + (M + 1) * ldo,), float("nan"), dtype=x.dtype, device="cuda")
    v = buf[offset:offset + M * ldo].view(M, ldo)
    v[:, :N] = x.to("cuda")
    return v[:, :N]


def patch_rows(M, g2):
    """Token rows the patch epilogue writes (row m -> (m / g2)(g2 + 1) + 1 + m % g2) and the class-token rows it must not touch."""
    m = torch.arange(M)
    rows = (m // g2) * (g2 + 1) + 1 + m % g2
    return rows, torch.arange(M // g2) * (g2 + 1)


def run_kernel(epi, inp, lda_pad=0, ldb_pad=0, ldo_pad=0, offset=0):
    """cg_gemm_bf16_tn (through vit_ops) on NaN-tailed operands into guarded outputs.  Returns ({output: [M, N] tensor}, guards_ok)."""
    from clip_diffusion_b200 import vit_ops

    M, N = inp["a"].shape[0], inp["b"].shape[0]
    ldo = N + ldo_pad
    a, b = _operand(inp["a"], lda_pad), _operand(inp["b"], ldb_pad)
    bias = nan_tailed(inp["bias"].float()) if epi in (BIAS_BF16, BIAS_RESID_F32, BIAS_QGELU_BF16) else None
    pos = nan_tailed(inp["pos"].float().contiguous()) if epi == PATCH_POS_F32 else None
    dtype = torch.float32 if epi in F32_OUT else torch.bfloat16
    g2 = inp["g2"] if epi == PATCH_POS_F32 else 0
    if epi == PATCH_POS_F32:
        rows, cls = patch_rows(M, g2)
        out = _Out(M // g2 * (g2 + 1), N, ldo, dtype, offset, cls.cuda())
    else:
        out = _Out(M, N, ldo, dtype, offset)
    outs = [out]
    aux = None
    if epi == BIAS_RESID_F32:
        aux = _aux_input(inp["resid"].float(), ldo, offset)
    elif epi == DQGELU_BF16:
        aux = _aux_input(inp["aux"], ldo, offset)
    elif epi == BIAS_QGELU_BF16:
        auxo = _Out(M, N, ldo, torch.bfloat16, offset)
        outs.append(auxo)
        aux = auxo.t
    vit_ops.gemm_bf16_tn(a, b, epi, bias=bias, out=out.t, aux=aux, pos=pos, g2=g2)
    torch.cuda.synchronize()
    ok = all(o.intact() for o in outs)
    got = {"out": out.t[rows.cuda()] if epi == PATCH_POS_F32 else out.t}
    if epi == BIAS_QGELU_BF16:
        got["aux"] = outs[1].t
    return {k: v.clone() for k, v in got.items()}, ok


def check_gemm(epi, inp, **layout):
    """Run the kernel and judge it against the reference: {"ratios": worst err / bound per output, "inexact": count (exact regimes),
    "guards": bool, ...}."""
    got, ok = run_kernel(epi, inp, **layout)
    dev_inp = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in inp.items()}
    ref = reference(epi, dev_inp)
    res = {"ratios": ratios(got, ref), "inexact": inexact(epi, got, ref) if inp["exact"] else 0, "guards": ok}
    if epi == BIAS_QGELU_BF16:
        res["sigma_err"] = sigma_error(dev_inp, got, ref)
    return res


def invariance(M, N, K, seed=5):
    """EPI_F32 on a multi-wave shape: a second run is bit-identical, and A rolled by 37 and by 129 rows gives the identically rolled
    output (no dependence on which CTA or wave a row block lands in)."""
    from clip_diffusion_b200 import vit_ops

    inp = gauss(M, N, K, seed, device="cuda")
    a, b = inp["a"], inp["b"]
    o1 = vit_ops.gemm_bf16_tn(a, b, F32)
    o2 = vit_ops.gemm_bf16_tn(a, b, F32)
    ok = torch.equal(o1, o2)
    for s in (37, 129):
        ok = ok and torch.equal(vit_ops.gemm_bf16_tn(a.roll(s, 0).contiguous(), b, F32), o1.roll(s, 0))
    torch.cuda.synchronize()
    return {"M": M, "N": N, "K": K, "variant": tile_variant(M, N, K, F32), "identical": bool(ok)}


def run_matrix(cases, invariance_shapes=()):
    """Run each case {M, N, K, epi, regime, g2, seed, [lda_pad, ldb_pad, ldo_pad, offset]} in this process (the CG_GEMM_* environment
    of this process picks the tile variants) and print one JSON line "GEMM_MATRIX {...}": per case the worst ratios, the inexact
    count, the guard check and the variant it ran on; then the invariance checks."""
    results = []
    for c in cases:
        inp = make_inputs(c["regime"], c["M"], c["N"], c["K"], c["seed"], g2=c.get("g2", 1), device="cuda")
        layout = {k: c[k] for k in ("lda_pad", "ldb_pad", "ldo_pad", "offset") if k in c}
        r = check_gemm(c["epi"], inp, **layout)
        r.update({k: c[k] for k in ("M", "N", "K", "epi", "regime")}, variant=tile_variant(c["M"], c["N"], c["K"], c["epi"]))
        results.append(r)
        del inp
    inv = [invariance(*s) for s in invariance_shapes]
    print("GEMM_MATRIX " + json.dumps({"cases": results, "invariance": inv, "sms": torch.cuda.get_device_properties(0).multi_processor_count}),
          flush=True)
    return results, inv


# ---------------------------------------------------------------------------------------------------------------- the matrix
# (M, N, K, g2): tail classes of every variant and the towers' real shapes.  g2 divides M (the patch epilogue's patches per image).
MATRIX_SHAPES = [
    (50, 256, 64, 25),        # M < 128, K = 64
    (300, 256, 64, 75),       # K = 64 with more than 256 rows (the pair when forced)
    (129, 384, 128, 43),      # M = 1 mod 128, N % 256 != 0 (128 x 128 on every variant), 2 k-blocks
    (383, 512, 320, 383),     # M = 127 mod 128; pair: M mod 256 = 127 (the second CTA of the last tile has no rows); 5 k-blocks
    (385, 256, 448, 77),      # M = 1 mod 128; pair: M mod 256 = 129; 7 k-blocks
    (777, 512, 1024, 37),
    (616, 2048, 512, 77),     # text tower (ViT-B, T = 77, 8 prompts): c_fc
    (616, 512, 2048, 77),     # text tower: c_proj
    (3136, 768, 3072, 49),    # ViT-B/32 patch embedding at 64 cutouts
    (6304, 2304, 768, 197),   # ViT-B/16 at 32 cutouts: QKV
    (6304, 768, 3072, 197),   # ViT-B/16 at 32 cutouts: c_proj
    (16384, 1024, 640, 256),  # ViT-L/14 patch embedding at 64 cutouts
    (16448, 3072, 1024, 257),  # ViT-L/14 at 64 cutouts: QKV
    (16448, 1024, 4096, 257),  # ViT-L/14 at 64 cutouts: c_proj
]
SWEEP_SHAPES = [(256, 256, 256, 64), (640, 512, 640, 160)]  # M = K (A = identity); 640 rows: pair tiles with M mod 256 = 128
NON_SWEEP = ("gauss", "exact", "scaled")
INVARIANCE_SHAPES = [(16448, 1024, 1024)]


def matrix_cases():
    cases = []
    for i, (M, N, K, g2) in enumerate(MATRIX_SHAPES):
        for epi in range(7):
            c = {"M": M, "N": N, "K": K, "g2": g2, "epi": epi, "regime": NON_SWEEP[(i + epi) % 3], "seed": 100 * i + epi}
            if i % 4 == 1:
                c.update(lda_pad=64, ldb_pad=128, ldo_pad=64)  # strided operands and a gap between output rows
            cases.append(c)
    for j, (M, N, K, g2) in enumerate(SWEEP_SHAPES):
        for epi in range(7):
            cases.append({"M": M, "N": N, "K": K, "g2": g2, "epi": epi, "regime": "sweep", "seed": 7 + j, "ldo_pad": 32 * j})
    return cases


def tail_classes(M, N, K, variant, sms):
    """The tail classes a case exercises on its tile variant (geometry only: the variant itself comes from cg_gemm_tile_variant)."""
    pair = variant == 2
    bn = 256 if variant in (0, 2) else 128
    rows = 2 * 128 if pair else 128
    tiles = -(-M // rows) * (N // bn)
    slots = sms // 2 if pair else sms
    kb = K // 64
    cls = set()
    if M < 128:
        cls.add("M<128")
    if M % 128 == 1:
        cls.add("M%128=1")
    if M % 128 == 127:
        cls.add("M%128=127")
    if pair and 1 <= M % 256 <= 128:
        cls.add("M%256 in [1,128]")
    if pair and M % 256 > 128:
        cls.add("M%256 in (128,256)")
    if tiles > 2 * slots:
        cls.add("tiles>2*slots")
    if kb == 1:
        cls.add("K=64")
    if kb % (6 if pair else 4) != 0:
        cls.add("kblocks%ring!=0")
    return cls


REQUIRED_CLASSES = {0: {"M<128", "M%128=1", "M%128=127", "tiles>2*slots", "K=64", "kblocks%ring!=0"},
                    1: {"M<128", "M%128=1", "M%128=127", "tiles>2*slots", "K=64", "kblocks%ring!=0"},
                    2: {"M%128=1", "M%128=127", "M%256 in [1,128]", "M%256 in (128,256)", "tiles>2*slots", "K=64", "kblocks%ring!=0"}}


if __name__ == "__main__":
    run_matrix(matrix_cases(), INVARIANCE_SHAPES)
