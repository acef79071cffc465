"""Float64 reference of the LayerNorm kernels (csrc/vit_misc.cu: cg_layernorm_fwd / cg_layernorm_bwd, eps 1e-5, biased variance, two
passes over the row) with a per-element error bound, and the input regimes the tests use (TEST-ONLY, torch; any device).

Error model of the fp32 kernels, per row of width D, with u = 2^-24 and n = D / 32 + 8 (a lane adds D / 32 values, then five shuffle
levels; any summation order of depth <= n is covered):
    mean    |m - m_ref| <= b_m = n u mean|x|
    var     b_v = 2 n u var + 2 b_m mean|x - m| + b_m^2             (centred second pass around the fp32 mean)
    rstd    |r - r_ref| <= b_r = r (b_v / (2 (var + eps)) + 2^-21)   (rsqrtf: 2 ulp, plus the roundings of q / D + eps)
    y       |y - y_ref| <= |gamma| (b_m r + |x - m| b_r + 2^-22 |xhat|) + 2^-23 (|xhat gamma| + |beta|)
The backward is judged on the mean / rstd the kernel reads (its own forward's): xhat = (x - mean) rstd, dh = dy gamma,
dx = rstd (dh - mean(dh) - xhat mean(dh xhat)) [+ dx_prev]:
    |dx - ref| <= 2 rstd (2^-22 (|dh| + |s1| + |xhat s2|) + n u (mean|dh| + |xhat| mean|dh xhat|)) + 2^-23 (|dx_prev| + |ref|)
bf16 outputs (y_bf16, dx_bf16) are judged like the GEMM's (oracle.gemm.ratios): the distance from the reference to the reals that
round to the output, over the bound.
"""
import torch

EPS = 1e-5
U = 2.0 ** -24


def _n(D):
    return D / 32 + 8


def layernorm_fwd(x, gamma, beta):
    """float64 y, mean, rstd and their bounds {"y", "mean", "rstd"} -> (ref, bound)."""
    x, gamma, beta = x.double(), gamma.double(), beta.double()
    D = x.shape[-1]
    m = x.mean(-1)
    xc = x - m[:, None]
    var = (xc * xc).mean(-1)
    r = torch.rsqrt(var + EPS)
    xhat = xc * r[:, None]
    y = xhat * gamma + beta
    b_m = _n(D) * U * x.abs().mean(-1)
    b_v = 2 * _n(D) * U * var + 2 * b_m * xc.abs().mean(-1) + b_m * b_m
    b_r = r * (b_v / (2 * (var + EPS)) + 2.0 ** -21)
    b_y = gamma.abs() * (b_m[:, None] * r[:, None] + xc.abs() * b_r[:, None] + 2.0 ** -22 * xhat.abs()) + 2.0 ** -23 * (
        (xhat * gamma).abs() + beta.abs())
    return {"y": (y, b_y), "mean": (m, b_m), "rstd": (r, b_r)}


def layernorm_bwd(dy, x, gamma, mean, rstd, dx_prev=None):
    """float64 dx on the given (fp32) mean / rstd, plus the previous gradient when accumulating: (ref, bound)."""
    dy, x, gamma, mean, rstd = dy.double(), x.double(), gamma.double(), mean.double(), rstd.double()
    D = x.shape[-1]
    xhat = (x - mean[:, None]) * rstd[:, None]
    dh = dy * gamma
    s1 = dh.mean(-1, keepdim=True)
    s2 = (dh * xhat).mean(-1, keepdim=True)
    dx = rstd[:, None] * (dh - s1 - xhat * s2)
    b = 2 * rstd[:, None] * (2.0 ** -22 * (dh.abs() + s1.abs() + (xhat * s2).abs())
                             + _n(D) * U * (dh.abs().mean(-1, keepdim=True) + xhat.abs() * (dh * xhat).abs().mean(-1, keepdim=True)))
    if dx_prev is not None:
        dx = dx + dx_prev.double()
        b = b + 2.0 ** -23 * (dx_prev.double().abs() + dx.abs())
    return dx, b


# ---------------------------------------------------------------------------------------------------------------- input regimes
def make_x(regime, M, D, seed):
    """fp32 [M, D] rows: gauss N(0.5, 4) (the original inputs); offset: mean 300, std 1; spiky: 4 channels 100x the rest; constant:
    every row one value (variance 0)."""
    g = torch.Generator().manual_seed(seed)
    if regime == "gauss":
        x = torch.randn(M, D, generator=g) * 2 + 0.5
    elif regime == "offset":
        x = torch.randn(M, D, generator=g) + 300.0
        assert (x.mean(-1) - 300).abs().max() < 1 and (x.std(-1) - 1).abs().max() < 0.3
    elif regime == "spiky":
        x = torch.randn(M, D, generator=g)
        ch = torch.randperm(D, generator=g)[:4]
        x[:, ch] *= 100.0
        assert (x[:, ch].abs().mean() / x.abs().mean()) > 20
    elif regime == "constant":
        x = (torch.randint(-8, 9, (M, 1), generator=g).float() * 0.375).expand(M, D).contiguous()
        assert (x == x[:, :1]).all()
    else:
        raise KeyError(regime)
    return x


REGIMES = ("gauss", "offset", "spiky", "constant")

