"""CPU tests of the ModifiedResNet (RN101) tower's host side and its oracle: OpenAI key naming, BatchNorm folding, the attention pool,
signal through the random init, missing checkpoint keys, and the float64 epilogue references against planted kernel mutations."""
import pytest
import torch
from torch.nn import functional as F

from oracle import clip_resnet as OR
from oracle import gemm as G


def _models():
    from clip_diffusion_b200 import models

    return models


def test_oracle_state_dict_matches_random_init_key_for_key():
    models = _models()
    sd = models.random_clip_resnet_state_dict("RN101", seed=1)
    shapes = models.clip_resnet_state_dict_shapes("RN101")
    assert list(sd) == list(shapes)
    assert {k: tuple(v.shape) for k, v in sd.items()} == shapes
    oracle = OR.OracleCLIPResNet("RN101", sd)
    mine = {k: tuple(v.shape) for k, v in oracle.state_dict().items()}
    assert mine == shapes  # OpenAI's names, order and shapes: strict loading of a real checkpoint maps 1:1


def test_batchnorm_folding_equals_conv_plus_eval_batchnorm():
    models = _models()
    g = torch.Generator().manual_seed(3)
    for k, stride in ((1, 1), (3, 1), (3, 2)):
        w = torch.randn(48, 24, k, k, generator=g, dtype=torch.float64)
        bn = torch.nn.BatchNorm2d(48).double().eval()
        bn.weight.data = 1 + 0.3 * torch.randn(48, generator=g, dtype=torch.float64)
        bn.bias.data = 0.2 * torch.randn(48, generator=g, dtype=torch.float64)
        bn.running_mean = 0.5 * torch.randn(48, generator=g, dtype=torch.float64)
        bn.running_var = 0.5 + torch.rand(48, generator=g, dtype=torch.float64)
        x = torch.randn(2, 24, 9, 9, generator=g, dtype=torch.float64)
        ref = bn(F.conv2d(x, w, stride=stride, padding=k // 2))
        wf, bf = models.fold_batchnorm(w, bn.weight, bn.bias, bn.running_mean, bn.running_var)
        got = F.conv2d(x, wf, bf, stride=stride, padding=k // 2)
        assert ((got - ref).norm() / ref.norm()).item() <= 1e-12


def test_attention_pool_equals_a_hand_written_softmax_over_row_0():
    g = torch.Generator().manual_seed(5)
    C, heads, E = 256, 4, 128
    pool = OR.AttentionPool2d(2, C, heads, E).double()
    for p in pool.parameters():
        p.data = 0.1 * torch.randn(p.shape, generator=g, dtype=torch.float64)
    x = torch.randn(3, C, 2, 2, generator=g, dtype=torch.float64)
    got = pool(x)
    tok = torch.cat([x.flatten(2).mean(-1, keepdim=True), x.flatten(2)], -1).transpose(1, 2) + pool.positional_embedding  # [N, T, C]
    q, k, v = pool.q_proj(tok[:, :1]), pool.k_proj(tok), pool.v_proj(tok)
    split = lambda t: t.view(t.shape[0], t.shape[1], heads, C // heads).transpose(1, 2)  # noqa: E731
    p = torch.softmax(split(q) @ split(k).transpose(-1, -2) / (C // heads) ** 0.5, dim=-1)
    ctx = (p @ split(v)).transpose(1, 2).reshape(3, C)
    want = pool.c_proj(ctx)
    assert got.shape == (3, E) and ((got - want).norm() / want.norm()).item() <= 1e-12


def test_random_init_carries_signal_through_every_block():
    """Activation RMS of every stage within [0.1, 10] x the stem's; each Bottleneck's branch >= 5 % of its output's RMS."""
    models = _models()
    oracle = OR.OracleCLIPResNet("RN101", models.random_clip_resnet_state_dict("RN101", seed=1))
    x = torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(0))
    blocks = [b for layer in (oracle.visual.layer1, oracle.visual.layer2, oracle.visual.layer3, oracle.visual.layer4) for b in layer]
    rms = lambda t: t.pow(2).mean().sqrt().item()  # noqa: E731
    with torch.no_grad():
        outs = oracle.visual.stages(x)
        r0 = rms(outs[0])
        assert len(outs) == 1 + 33
        for i, blk in enumerate(blocks):
            assert 0.1 <= rms(outs[i + 1]) / r0 <= 10, (i, rms(outs[i + 1]) / r0)
            assert rms(blk.branch(outs[i])) >= 0.05 * rms(outs[i + 1]), i
        assert torch.isfinite(oracle.visual.attnpool(outs[-1])).all()


def test_checkpoint_with_a_missing_key_raises_keyerror(tmp_path, monkeypatch):
    models = _models()
    sd = models.random_clip_resnet_state_dict("RN101", seed=2)
    del sd["visual.layer3.7.bn2.running_var"]
    torch.save(sd, str(tmp_path / "RN101.pt"))
    monkeypatch.setenv("CLIPGUIDE_B200_WEIGHTS", str(tmp_path))
    with pytest.raises(KeyError):
        models.load_clip_models(["RN101"], "cuda")


def test_resnet_tower_refuses_a_cpu_device():
    models = _models()
    with pytest.raises(ValueError, match="cpu"):
        models.CLIPModelB200("RN101", device="cpu")
    assert "RN101" in models.CLIP_TEXT_CONFIGS


# ------------------------------------------------------------------------------------------------------- planted epilogue mutations
def _emulate(epi, inp, mutation=None):
    """The kernel's arithmetic on the CPU: fp32 accumulator (float64 product rounded once), then the epilogue in fp32.  `mutation`
    plants one defect: a mask test >= 0 instead of > 0, a dropped residual, or a bf16-rounded residual gradient."""
    acc = (inp["a"].double() @ inp["b"].double().t()).float()
    if epi == OR.BIAS_RESID_RELU_BF16:
        v = acc + inp["bias"].float()
        if mutation != "drop_resid":
            v = v + inp["resid"].float()
        return {"out": v.clamp_min(0).bfloat16()}
    v = acc
    if epi == OR.RESID_DRELU and mutation != "drop_resid":
        r = inp["resid"].float()
        v = v + (r.bfloat16().float() if mutation == "bf16_resid" else r)
    m = inp["mask"].float()
    drop = (m < 0) if mutation == "mask_ge0" else (m <= 0)
    v = torch.where(drop, torch.zeros_like(v), v)
    if epi == OR.DRELU_BF16:
        return {"out": v.bfloat16()}
    return {"out": v, "out_bf16": v.bfloat16()}


@pytest.mark.parametrize("epi,mutation", [(OR.DRELU_BF16, "mask_ge0"), (OR.RESID_DRELU, "mask_ge0"), (OR.RESID_DRELU, "drop_resid"),
                                          (OR.RESID_DRELU, "bf16_resid"), (OR.BIAS_RESID_RELU_BF16, "drop_resid")])
def test_epilogue_references_catch_planted_mutations(epi, mutation):
    inp = OR.relu_inputs("gauss", 200, 128, 256, seed=4)
    # saved ReLU outputs at exactly +-0 over positive gradients: a >= 0 mask passes what threshold_backward zeroes
    e = OR.relu_epilogue_inputs(epi, inp)
    ref = OR.relu_reference(epi, e)
    assert max(G.ratios(_emulate(epi, e), ref).values()) <= 1.0
    assert max(G.ratios(_emulate(epi, e, mutation), ref).values()) > 1.0


def test_kernel_references_match_direct_formulas():
    g = torch.Generator().manual_seed(7)
    x = torch.randn(2, 7, 7, 5, generator=g, dtype=torch.float64)
    cols = OR.im2col3x3(x, 2, 64)  # [2*4*4, 64]
    assert cols.shape == (32, 64) and (cols[:, 45:] == 0).all()
    # output (1, 2) of image 1, tap (ky, kx) = (2, 0): input (2*1 + 2 - 1, 2*2 + 0 - 1) = (3, 3)
    assert torch.equal(cols[16 + 1 * 4 + 2, (2 * 3 + 0) * 5: (2 * 3 + 0) * 5 + 5], x[1, 3, 3])
    assert (cols[0, :5] == 0).all()  # output (0, 0), tap (0, 0) lies in the padding
    dy = torch.randn(2, 4, 4, 6, generator=g, dtype=torch.float64)
    w = torch.randn(6, 3, 3, 3, generator=g, dtype=torch.float64)
    dx, _ = OR.conv3x3s2_dgrad(dy, w, 7, 7, 8)
    xx = torch.randn(2, 3, 7, 7, dtype=torch.float64, requires_grad=True)
    (gx,) = torch.autograd.grad(F.conv2d(xx, w, stride=2, padding=1), xx, OR.nchw(dy))
    assert torch.allclose(dx[..., :3], OR.nhwc(gx).reshape(2, 49, 3), atol=1e-12) and (dx[..., 3:] == 0).all()
