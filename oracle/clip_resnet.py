"""Oracle restatement of OpenAI CLIP's ModifiedResNet image tower (TEST-ONLY, CPU torch), and float64 references of the kernels the
B200 tower is built from (csrc/clip_resnet.cu, the ReLU epilogues of csrc/vit_gemm.cu).

The reference gets RN101 from the un-vendored ``clip`` package (clip_diffusion/models.py:76-80 with config.py:41's default names).
This restates OpenAI's clip/model.py from its published architecture, so parity with openai/CLIP itself is UNPINNED (as for
oracle/clip_vit.py):
  stem      3 x (3x3 conv, no bias -> BatchNorm -> ReLU), the first with stride 2, then AvgPool2d(2)
  layers    Bottleneck(inplanes, planes, stride): relu(bn1(conv1 1x1)) -> relu(bn2(conv2 3x3)) -> AvgPool2d(stride) -> bn3(conv3 1x1),
            plus the identity or downsample = AvgPool2d(stride) -> 1x1 conv -> BatchNorm, then ReLU
  attnpool  tokens = [mean over positions, positions] + positional_embedding; multi-head attention of the query row 0 over all
            tokens with separate q / k / v projections, then c_proj; the output is row 0
BatchNorm runs in eval mode.  Parameter names are OpenAI's under ``visual.``, so real checkpoints map 1:1.
"""
from collections import OrderedDict

import torch
from torch import nn
from torch.nn import functional as F

from oracle.gemm import C_ACC, C_ADD

CONFIGS = {
    # name: (input_resolution, layers, width, heads, embed_dim)
    "RN101": (224, (3, 4, 23, 3), 64, 32, 512),
}


class Bottleneck(nn.Module):
    expansion = 4

    def __init__(self, inplanes, planes, stride=1):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu1 = nn.ReLU()
        self.conv2 = nn.Conv2d(planes, planes, 3, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.relu2 = nn.ReLU()
        self.avgpool = nn.AvgPool2d(stride) if stride > 1 else nn.Identity()
        self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.relu3 = nn.ReLU()
        self.downsample = None
        if stride > 1 or inplanes != planes * 4:
            self.downsample = nn.Sequential(OrderedDict([("-1", nn.AvgPool2d(stride)), ("0", nn.Conv2d(inplanes, planes * 4, 1, bias=False)),
                                                         ("1", nn.BatchNorm2d(planes * 4))]))

    def branch(self, x):
        out = self.relu1(self.bn1(self.conv1(x)))
        out = self.relu2(self.bn2(self.conv2(out)))
        return self.bn3(self.conv3(self.avgpool(out)))

    def forward(self, x):
        identity = x if self.downsample is None else self.downsample(x)
        return self.relu3(self.branch(x) + identity)


class AttentionPool2d(nn.Module):
    def __init__(self, spacial_dim, embed_dim, num_heads, output_dim):
        super().__init__()
        self.positional_embedding = nn.Parameter(torch.zeros(spacial_dim ** 2 + 1, embed_dim))
        self.k_proj = nn.Linear(embed_dim, embed_dim)
        self.q_proj = nn.Linear(embed_dim, embed_dim)
        self.v_proj = nn.Linear(embed_dim, embed_dim)
        self.c_proj = nn.Linear(embed_dim, output_dim)
        self.num_heads = num_heads

    def tokens(self, x):
        x = x.flatten(start_dim=2).permute(2, 0, 1)  # NCHW -> (HW)NC
        x = torch.cat([x.mean(dim=0, keepdim=True), x], dim=0)
        return x + self.positional_embedding[:, None, :].to(x.dtype)

    def forward(self, x):
        x = self.tokens(x)
        x, _ = F.multi_head_attention_forward(
            query=x[:1], key=x, value=x, embed_dim_to_check=x.shape[-1], num_heads=self.num_heads, q_proj_weight=self.q_proj.weight,
            k_proj_weight=self.k_proj.weight, v_proj_weight=self.v_proj.weight, in_proj_weight=None,
            in_proj_bias=torch.cat([self.q_proj.bias, self.k_proj.bias, self.v_proj.bias]), bias_k=None, bias_v=None, add_zero_attn=False,
            dropout_p=0.0, out_proj_weight=self.c_proj.weight, out_proj_bias=self.c_proj.bias, use_separate_proj_weight=True,
            training=False, need_weights=False)
        return x.squeeze(0)


class ModifiedResNet(nn.Module):
    def __init__(self, layers, output_dim, heads, input_resolution=224, width=64):
        super().__init__()
        self.output_dim = output_dim
        self.input_resolution = input_resolution
        self.conv1 = nn.Conv2d(3, width // 2, 3, stride=2, padding=1, bias=False)
        self.bn1 = nn.BatchNorm2d(width // 2)
        self.relu1 = nn.ReLU()
        self.conv2 = nn.Conv2d(width // 2, width // 2, 3, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(width // 2)
        self.relu2 = nn.ReLU()
        self.conv3 = nn.Conv2d(width // 2, width, 3, padding=1, bias=False)
        self.bn3 = nn.BatchNorm2d(width)
        self.relu3 = nn.ReLU()
        self.avgpool = nn.AvgPool2d(2)
        self._inplanes = width
        self.layer1 = self._make_layer(width, layers[0])
        self.layer2 = self._make_layer(width * 2, layers[1], stride=2)
        self.layer3 = self._make_layer(width * 4, layers[2], stride=2)
        self.layer4 = self._make_layer(width * 8, layers[3], stride=2)
        self.attnpool = AttentionPool2d(input_resolution // 32, width * 32, heads, output_dim)

    def _make_layer(self, planes, blocks, stride=1):
        layers = [Bottleneck(self._inplanes, planes, stride)]
        self._inplanes = planes * Bottleneck.expansion
        layers += [Bottleneck(self._inplanes, planes) for _ in range(1, blocks)]
        return nn.Sequential(*layers)

    def stem(self, x):
        x = self.relu1(self.bn1(self.conv1(x)))
        x = self.relu2(self.bn2(self.conv2(x)))
        x = self.relu3(self.bn3(self.conv3(x)))
        return self.avgpool(x)

    def stages(self, x):
        """The stem's output and every Bottleneck's output, in order (the activation-statistics tests read them)."""
        outs = [self.stem(x.type(self.conv1.weight.dtype))]
        for layer in (self.layer1, self.layer2, self.layer3, self.layer4):
            for blk in layer:
                outs.append(blk(outs[-1]))
        return outs

    def forward(self, x):
        return self.attnpool(self.stages(x)[-1])


class OracleCLIPResNet(nn.Module):
    """Stands in for the object ``clip.load("RN101")`` returns: ``.visual.input_resolution``, ``.encode_image`` (oracle/cond_fn.py)."""

    def __init__(self, name, state_dict, dtype=torch.float32):
        super().__init__()
        res, layers, width, heads, embed = CONFIGS[name]
        self.visual = ModifiedResNet(layers, embed, heads, res, width)
        self.load_state_dict({k: v.clone() for k, v in state_dict.items() if k.startswith("visual.")}, strict=True)
        self.to(dtype).eval().requires_grad_(False)

    def encode_image(self, image):
        return self.visual(image.to(self.visual.conv1.weight.dtype))


class _FixedReLU(nn.Module):
    """x * mask: a ReLU whose on/off pattern is given (1 where the saved output of another evaluation is > 0)."""

    def __init__(self, mask):
        super().__init__()
        self.mask = mask

    def forward(self, x):
        return x * self.mask.to(x.dtype)


def relu_modules(visual):
    """The ReLUs of a ModifiedResNet in evaluation order: the stem's three, then relu1, relu2, relu3 of every Bottleneck."""
    mods = [(visual, "relu1"), (visual, "relu2"), (visual, "relu3")]
    for layer in (visual.layer1, visual.layer2, visual.layer3, visual.layer4):
        for blk in layer:
            mods += [(blk, "relu1"), (blk, "relu2"), (blk, "relu3")]
    return mods


def fix_relu_masks(oracle, masks):
    """Replace every ReLU of the oracle by the on/off pattern of another evaluation (NCHW bool tensors in relu_modules order).  A
    ReLU network's input gradient is piecewise constant in its masks: a unit whose pre-activation lies within the bf16 rounding of
    zero switches sides between a bf16 and an fp32 evaluation and moves the gradient by its whole contribution (rel-L2 grows as the
    square root of the fraction of switched units).  With the masks fixed, the oracle's gradient is the derivative of the same
    linearisation the tower differentiates, so a gradient check measures the backward's arithmetic."""
    mods = relu_modules(oracle.visual)
    assert len(mods) == len(masks), (len(mods), len(masks))
    for (mod, attr), m in zip(mods, masks):
        setattr(mod, attr, _FixedReLU(m))
    return oracle


# ---------------------------------------------------------------------------------------------------------------- kernel references
def nhwc(x):
    return x.permute(0, 2, 3, 1)


def nchw(x):
    return x.permute(0, 3, 1, 2)


def im2col3x3(x, stride, kpad):
    """x [N, H, W, C] -> [N*Ho*Wo, kpad], column (ky*3 + kx)*C + c, zero padding and zero columns >= 9C: F.unfold reordered."""
    N, H, W, C = x.shape
    cols = F.unfold(nchw(x).double(), 3, padding=1, stride=stride)  # [N, C*9, L], row c*9 + ky*3 + kx
    L = cols.shape[-1]
    cols = cols.view(N, C, 9, L).permute(0, 3, 2, 1).reshape(N * L, 9 * C)
    return F.pad(cols, (0, kpad - 9 * C))


def avgpool2x2(x):
    """[N, H, W, C] -> [N, H/2, W/2, C] in float64, and the bound of an fp32 sum of four values times 0.25."""
    ref = nhwc(F.avg_pool2d(nchw(x).double(), 2))
    return ref, 4 * C_ADD * nhwc(F.avg_pool2d(nchw(x).double().abs(), 2))


def avgpool2x2_bwd(dy, mask=None):
    """dx = 0.25 dy[n, y/2, x/2] * [mask > 0] (exact in float64: a multiplication by a power of two and a select)."""
    dx = 0.25 * dy.double().repeat_interleave(2, 1).repeat_interleave(2, 2)
    if mask is not None:
        dx = torch.where(mask.double() <= 0, torch.zeros_like(dx), dx)
    return dx


def conv3x3s2_dgrad(dy, w, H, W, kpad):
    """Input gradient of a 3x3 stride-2 padding-1 convolution: dy [N, Ho, Wo, Cout], w [Cout, Cin, 3, 3] -> ([N, H*W, kpad], bound):
    float64 values and the bound of the kernel's fp32 sums (at most 4 * Cout products, each adding one rounding)."""
    N, Cin = dy.shape[0], w.shape[1]
    grad = lambda d, k: torch.nn.grad.conv2d_input((N, Cin, H, W), k, nchw(d), stride=2, padding=1)  # noqa: E731
    ref = nhwc(grad(dy.double(), w.double())).reshape(N, H * W, Cin)
    mag = nhwc(grad(dy.double().abs(), w.double().abs())).reshape(N, H * W, Cin)
    terms = 4 * dy.shape[-1]
    return F.pad(ref, (0, kpad - Cin)), F.pad(terms * 2.0 ** -24 * mag, (0, kpad - Cin))


def attnpool_tokens(x, pos):
    """x [N, S, C], pos [S+1, C] -> tokens [N, S+1, C] in float64, and the bound of the kernel's fp32 arithmetic (the mean: S
    additions and a division)."""
    x, pos = x.double(), pos.double()
    mean = x.mean(dim=1, keepdim=True)
    ref = torch.cat([mean, x], dim=1) + pos[None]
    S = x.shape[1]
    bmean = (S + 2) * 2.0 ** -24 * x.abs().mean(dim=1, keepdim=True)
    bound = torch.cat([bmean, torch.zeros_like(x)], dim=1) + C_ADD * ref.abs()
    return ref, bound


def attnpool_tokens_bwd(dtok, x):
    """dtok [N, S+1, C], x [N, S, C] (the masked ReLU output) -> g [N, S, C] = (dtok[:, 1:] + dtok[:, :1] / S) * [x > 0], and the bound
    of the kernel's division and addition."""
    S = x.shape[1]
    d = dtok.double()
    v = d[:, 1:] + d[:, :1] / S
    keep = x.double() > 0
    ref = torch.where(keep, v, torch.zeros_like(v))
    bound = torch.where(keep, C_ADD * (d[:, 1:].abs() + 2 * d[:, :1].abs() / S), torch.zeros_like(v))
    return ref, bound


# the ReLU epilogues of cg_gemm_bf16_tn_relu (CG_EPI_* of include/clipguide_b200.h); not part of oracle.gemm's matrix
BIAS_RELU_BF16, BIAS_RESID_RELU_BF16, DRELU_BF16, RESID_DRELU = 7, 8, 9, 10
RELU_EPI_NAMES = {BIAS_RELU_BF16: "BIAS_RELU_BF16", BIAS_RESID_RELU_BF16: "BIAS_RESID_RELU_BF16", DRELU_BF16: "DRELU_BF16", RESID_DRELU: "RESID_DRELU"}


def relu_reference(epi, inp):
    """Float64 results and bounds of one ReLU epilogue, in oracle.gemm's model ({output: (ref, bound, "f32" | "bf16")}): inputs are
    what the kernel reads -- bf16 a, b, mask and (BIAS_RESID_RELU) resid, fp32 bias and (RESID_DRELU) resid.  ReLU is 1-Lipschitz, so
    it keeps the bound of its argument; a mask is exact (a select), so masked elements are exactly 0."""
    a, b = inp["a"].double(), inp["b"].double()
    acc = a @ b.t()
    mag = a.abs() @ b.abs().t()
    b_acc = C_ACC * mag
    if epi == BIAS_RELU_BF16:
        u = acc + inp["bias"].double()
        return {"out": (u.clamp_min(0), b_acc + C_ADD * (mag + inp["bias"].double().abs()), "bf16")}
    if epi == BIAS_RESID_RELU_BF16:
        bias, r = inp["bias"].double(), inp["resid"].double()
        u = acc + bias + r
        return {"out": (u.clamp_min(0), b_acc + 2 * C_ADD * (mag + bias.abs() + r.abs()), "bf16")}
    mask = inp.get("mask")
    keep = torch.ones_like(acc, dtype=torch.bool) if mask is None else ~(mask.double() <= 0)
    zero = torch.zeros_like(acc)
    if epi == DRELU_BF16:
        return {"out": (torch.where(keep, acc, zero), torch.where(keep, b_acc, zero), "bf16")}
    assert epi == RESID_DRELU, epi
    r = inp["resid"].double()
    v, bound = torch.where(keep, acc + r, zero), torch.where(keep, b_acc + C_ADD * (mag + r.abs()), zero)
    return {"out": (v, bound, "f32"), "out_bf16": (v, bound, "bf16")}


def relu_inputs(regime, M, N, K, seed, device="cpu"):
    """oracle.gemm's `gauss` or `exact` operands plus the ReLU epilogues' inputs: resid as bf16 (for BIAS_RESID_RELU) and fp32
    (RESID_DRELU), and a bf16 mask of saved ReLU outputs with exact +0 and -0, negative and NaN-free positive values."""
    from oracle import gemm

    inp = gemm.make_inputs(regime, M, N, K, seed, device=device)
    g = torch.Generator(device=device).manual_seed(seed + 1)
    m = torch.randn(M, N, device=device, generator=g)
    sel = torch.randint(0, 4, (M, N), device=device, generator=g)
    m = torch.where(sel == 0, torch.zeros_like(m), m)
    m = torch.where(sel == 1, -torch.zeros_like(m), m)
    inp["mask"] = m.bfloat16()
    inp["resid_bf16"] = inp["resid"].bfloat16()
    assert (inp["mask"].float() == 0).any() and (inp["mask"].float() < 0).any() and (inp["mask"].float() > 0).any()
    return inp


def relu_epilogue_inputs(epi, inp, null_mask=False):
    """The inputs one epilogue reads, as relu_reference and the kernel take them."""
    out = {"a": inp["a"], "b": inp["b"]}
    if epi in (BIAS_RELU_BF16, BIAS_RESID_RELU_BF16):
        out["bias"] = inp["bias"]
    if epi == BIAS_RESID_RELU_BF16:
        out["resid"] = inp["resid_bf16"]
    if epi == RESID_DRELU:
        out["resid"] = inp["resid"].float()
    if epi == DRELU_BF16 or (epi == RESID_DRELU and not null_mask):
        out["mask"] = inp["mask"]
    return out


def run_relu_kernel(epi, inp, ldo_pad=0, offset_bytes=0, alias=False):
    """cg_gemm_bf16_tn_relu (through vit_ops) on NaN-tailed operands into guarded outputs (oracle.gemm's harness).  alias: RESID_DRELU
    reads its residual from its own fp32 output.  Returns ({output: [M, N] tensor}, guards_ok)."""
    from clip_diffusion_b200 import vit_ops
    from oracle import gemm
    from oracle.attention import nan_tailed

    M, N = inp["a"].shape[0], inp["b"].shape[0]
    ldo = N + ldo_pad
    a, b = gemm._operand(inp["a"], 0), gemm._operand(inp["b"], 0)
    f32 = epi == RESID_DRELU
    off = lambda dtype: offset_bytes // (4 if dtype == torch.float32 else 2)  # noqa: E731  every array starts offset_bytes in
    out = gemm._Out(M, N, ldo, torch.float32 if f32 else torch.bfloat16, off(torch.float32 if f32 else torch.bfloat16))
    outs = [out]
    kw = {}
    if "bias" in inp:
        kw["bias"] = nan_tailed(inp["bias"].float())
    if "mask" in inp:
        kw["mask"] = gemm._aux_input(inp["mask"], ldo, off(torch.bfloat16))
    if "resid" in inp:
        if alias:
            out.t.copy_(inp["resid"].to("cuda"))
            kw["resid"] = out.t
        else:
            kw["resid"] = gemm._aux_input(inp["resid"], ldo, off(inp["resid"].dtype))
    if f32:
        ob = gemm._Out(M, N, ldo, torch.bfloat16, off(torch.bfloat16))
        outs.append(ob)
        kw["out_bf16"] = ob.t
    vit_ops.gemm_bf16_tn_relu(a, b, epi, out=out.t, **kw)
    torch.cuda.synchronize()
    got = {"out": out.t.clone()}
    if f32:
        got["out_bf16"] = outs[1].t.clone()
    return got, all(o.intact() for o in outs)


def check_relu_gemm(epi, inp, null_mask=False, **layout):
    """Run one ReLU epilogue and judge it: {"ratios", "inexact" (exact regime: outputs that differ from the correctly rounded exact
    result), "guards"}."""
    from oracle import gemm

    e = relu_epilogue_inputs(epi, inp, null_mask)
    got, ok = run_relu_kernel(epi, e, **layout)
    ref = relu_reference(epi, {k: v.cuda() for k, v in e.items()})
    n_inexact = 0
    if inp["exact"]:
        for name, (r, _, kind) in ref.items():
            want = r if kind == "f32" else gemm.rne_bf16(r).double()
            n_inexact += int((got[name].double() != want).sum())
    return {"ratios": gemm.ratios(got, ref), "inexact": n_inexact, "guards": ok}


# (M, N, K): M < 128, M % 128 = 1 and 127, pair tails, K = 64, the tower's layer shapes at 2 cutouts
RELU_SHAPES = [(50, 128, 64), (129, 384, 128), (383, 512, 320), (385, 256, 576), (777, 512, 1024), (6272, 256, 576), (1568, 1024, 256)]


def relu_matrix_cases():
    cases = []
    for i, (M, N, K) in enumerate(RELU_SHAPES):
        for epi in RELU_EPI_NAMES:
            for regime in ("gauss", "exact"):
                c = {"M": M, "N": N, "K": K, "epi": epi, "regime": regime, "seed": 10 * i + epi}
                if i % 2:
                    c["ldo_pad"] = 64
                cases.append(c)
    return cases


def run_relu_matrix(cases):
    """Run every case in this process (the CG_GEMM_* environment picks the tile variant) and print "RELU_MATRIX {...}"."""
    import json

    from oracle import gemm

    results = []
    for c in cases:
        inp = relu_inputs(c["regime"], c["M"], c["N"], c["K"], c["seed"], device="cuda")
        r = check_relu_gemm(c["epi"], inp, **{k: c[k] for k in ("ldo_pad",) if k in c})
        r.update({k: c[k] for k in ("M", "N", "K", "epi", "regime")}, variant=gemm.tile_variant(c["M"], c["N"], c["K"], c["epi"]))
        results.append(r)
    print("RELU_MATRIX " + json.dumps({"cases": results}), flush=True)
    return results
