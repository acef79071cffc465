"""GPU parity of CLIP's ModifiedResNet tower (RN101) and its kernels against the oracle (oracle/clip_resnet.py): im2col bit for bit,
the pools, the stem's stride-2 dgrad and the attention-pool front end within float64 bounds, the ReLU epilogues on every GEMM tile
variant, the whole tower (tiny and real-size RN101) through forward_patches / backward_patches and embed_image, CUDA-graph replay, the
guidance step against the oracle cond_fn, the default four-tower configuration, and RN101's text tower."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COS_MIN = 0.999
GRAD_REL_MAX = 1e-2
TINY = {"test-rn-a": (64, (1, 1, 1, 1), 8, 4, 128), "test-rn-b": (96, (2, 1, 2, 1), 16, 8, 256)}


def _lib():
    from clip_diffusion_b200 import _lib

    return _lib


def _register():
    from clip_diffusion_b200 import models
    from oracle import clip_resnet as OR

    for name, cfg in TINY.items():
        models.register_clip_resnet_config(name, *cfg)
        OR.CONFIGS[name] = cfg


def _within(got, ref, bound):
    d = (got.double().cpu() - ref.cpu()).abs()
    return bool((d <= bound.cpu()).all())


@pytest.mark.parametrize("C", [3, 32, 64, 256])
@pytest.mark.parametrize("stride", [1, 2])
def test_im2col_is_bit_exact(C, stride):
    from oracle import clip_resnet as OR

    L = _lib()
    N, H = 3, 7
    ldx = (C + 7) // 8 * 8 + 8  # padded rows, NaN in the gap
    g = torch.Generator().manual_seed(C + stride)
    x = torch.randn(N, H, H, C, generator=g).bfloat16()
    buf = torch.full((N * H * H, ldx), float("nan"), dtype=torch.bfloat16, device="cuda")
    buf[:, :C] = x.view(-1, C).cuda()
    kpad = (9 * C + 63) // 64 * 64
    Ho = (H - 1) // stride + 1
    out = torch.full((N * Ho * Ho, kpad), float("nan"), dtype=torch.bfloat16, device="cuda")
    L.call("cg_im2col3x3_nhwc", L.ptr(buf), N, H, H, C, ldx, stride, kpad, L.ptr(out))
    want = OR.im2col3x3(x, stride, kpad)
    assert torch.equal(out.cpu().double(), want)


def test_avgpool_forward_and_backward():
    from oracle import clip_resnet as OR
    from oracle.gemm import bf16_cell

    L = _lib()
    N, H, C = 2, 14, 256
    g = torch.Generator().manual_seed(1)
    x = torch.randn(N, H, H, C, generator=g).bfloat16()
    y = torch.empty(N, H // 2, H // 2, C, dtype=torch.bfloat16, device="cuda")
    xc = x.cuda()  # device copies stay referenced across the calls
    L.call("cg_avgpool2x2_nhwc_fwd", L.ptr(xc), N, H, H, C, L.ptr(y))
    ref, bound = OR.avgpool2x2(x)
    lo, hi = bf16_cell(y.cpu())
    assert bool(((lo - bound <= ref) & (ref <= hi + bound)).all())
    # backward: mask with exact +-0 (threshold_backward zeroes them), fp32 and bf16 dy / dx
    dy = torch.randn(N, H // 2, H // 2, C, generator=g)
    mask = torch.randn(N, H, H, C, generator=g)
    mask[..., ::3] = 0.0
    mask[..., 1::5] = -0.0
    mask = mask.bfloat16()
    mc = mask.cuda()
    for dy_f32 in (1, 0):
        dyv = dy if dy_f32 else dy.bfloat16()
        dyc = dyv.cuda()
        for m in (mask, None):
            for dx_f32 in (1, 0):
                dx = torch.full((N, H, H, C), float("nan"), device="cuda", dtype=torch.float32 if dx_f32 else torch.bfloat16)
                L.call("cg_avgpool2x2_nhwc_bwd", L.ptr(dyc), dy_f32, L.ptr(mc) if m is not None else None, N, H, H, C, L.ptr(dx), dx_f32)
                want = OR.avgpool2x2_bwd(dyv, m)
                want = want if dx_f32 else want.float().bfloat16().double()
                assert torch.equal(dx.cpu().double(), want), (dy_f32, m is None, dx_f32)


def test_stem_stride2_dgrad_within_bound():
    from oracle import clip_resnet as OR

    L = _lib()
    N, H, Cout, ld = 2, 32, 32, 128
    Ho = H // 2
    g = torch.Generator().manual_seed(2)
    dy = torch.randn(N, Ho, Ho, Cout, generator=g).bfloat16()
    buf = torch.full((N * Ho * Ho, ld), float("nan"), dtype=torch.bfloat16, device="cuda")
    buf[:, :Cout] = dy.view(-1, Cout).cuda()
    w = torch.randn(Cout, 3, 3, 3, generator=g)
    dx = torch.full((N, H * H, 8), float("nan"), device="cuda")
    wc = w.cuda()
    L.call("cg_conv3x3s2_dgrad", L.ptr(buf), N, H, H, Cout, ld, L.ptr(wc), 3, 8, L.ptr(dx))
    ref, bound = OR.conv3x3s2_dgrad(dy, w, H, H, 8)
    assert _within(dx, ref, bound) and (dx[..., 3:] == 0).all()


def test_attention_pool_front_end():
    from oracle import clip_resnet as OR
    from oracle.gemm import bf16_cell

    L = _lib()
    N, S, C = 3, 49, 2048
    g = torch.Generator().manual_seed(3)
    x = torch.randn(N, S, C, generator=g).clamp_min(0).bfloat16()  # a ReLU output: exact zeros
    pos = torch.randn(S + 1, C, generator=g)
    tok = torch.empty(N * (S + 1), C, dtype=torch.bfloat16, device="cuda")
    xc, posc = x.cuda(), pos.cuda()
    L.call("cg_resnet_attnpool_fwd", L.ptr(xc), L.ptr(posc), N, S, C, L.ptr(tok))
    ref, bound = OR.attnpool_tokens(x, pos)
    lo, hi = bf16_cell(tok.cpu().view(N, S + 1, C))
    assert bool(((lo - bound <= ref) & (ref <= hi + bound)).all())
    dtok = torch.randn(N * (S + 1), C, generator=g)
    gf = torch.empty(N * S, C, device="cuda")
    gb = torch.empty(N * S, C, dtype=torch.bfloat16, device="cuda")
    dtokc = dtok.cuda()
    L.call("cg_resnet_attnpool_bwd", L.ptr(dtokc), L.ptr(xc), N, S, C, L.ptr(gf), L.ptr(gb))
    ref, bound = OR.attnpool_tokens_bwd(dtok.view(N, S + 1, C), x)
    assert _within(gf.view(N, S, C), ref, bound)
    assert torch.equal(gb.cpu(), gf.cpu().bfloat16()) and (gf.cpu().view(N, S, C)[x == 0] == 0).all()
    dy = torch.randn(N, C, generator=g)
    dctx = torch.full((N * (S + 1), C), float("nan"), dtype=torch.bfloat16, device="cuda")
    dyc = dy.cuda()
    L.call("cg_resnet_attnpool_dctx", L.ptr(dyc), N, S + 1, C, L.ptr(dctx))
    want = torch.zeros(N, S + 1, C, dtype=torch.bfloat16)
    want[:, 0] = dy.bfloat16()
    assert torch.equal(dctx.cpu().view(N, S + 1, C), want)


# ------------------------------------------------------------------------------------------------------- ReLU epilogues
def test_relu_epilogues_alias_null_mask_and_refusals():
    from clip_diffusion_b200 import vit_ops
    from oracle import clip_resnet as OR

    L = _lib()
    inp = OR.relu_inputs("gauss", 300, 256, 192, seed=8, device="cuda")
    for kw in ({"alias": True}, {"null_mask": True}, {"offset_bytes": 16}):
        null = kw.pop("null_mask", False)
        e = OR.relu_epilogue_inputs(OR.RESID_DRELU, inp, null)
        got, ok = OR.run_relu_kernel(OR.RESID_DRELU, e, **kw)
        ref = OR.relu_reference(OR.RESID_DRELU, e)
        from oracle.gemm import ratios

        assert ok and max(ratios(got, ref).values()) <= 1.0, kw
    # cg_gemm_bf16_tn refuses the new ids; the new entry point refuses the old ones and missing inputs
    a, b = inp["a"], inp["b"]
    with pytest.raises(L.ClipGuideError):
        vit_ops.gemm_bf16_tn(a, b, L.EPI_BIAS_RELU_BF16, bias=inp["bias"])
    out = torch.empty(300, 256, dtype=torch.bfloat16, device="cuda")
    for epi, kw in ((L.EPI_BF16, {}), (L.EPI_DRELU_BF16, {}), (L.EPI_BIAS_RESID_RELU_BF16, {"bias": inp["bias"]})):
        with pytest.raises(L.ClipGuideError):
            vit_ops.gemm_bf16_tn_relu(a, b, epi, out=out, **kw)
    assert L.load().cg_gemm_tile_variant(300, 256, 192, L.EPI_RESID_DRELU) in (0, 1, 2)


FORCE = {"auto": {}, "pair256x256": {"CG_GEMM_PAIR": "1"}, "bn128": {"CG_GEMM_PAIR": "0", "CG_GEMM_BN": "128"},
         "bn256": {"CG_GEMM_PAIR": "0", "CG_GEMM_BN": "256"}}
FORCED_VARIANT = {"pair256x256": 2, "bn128": 1, "bn256": 0}


@pytest.mark.parametrize("force", list(FORCE))
def test_relu_epilogues_on_every_tile_variant(force):
    """Epilogues 7-10 x {gauss, exact} over the GEMM's tail classes and the tower's shapes, in a child process whose CG_GEMM_*
    environment forces the tile variant: within oracle.gemm's error model, bit for bit on small integers, NaN-tailed operands, guarded
    outputs with a gap after each row."""
    from oracle import clip_resnet as OR

    code = "import sys; sys.path.insert(0, %r)\nfrom oracle import clip_resnet as R\nR.run_relu_matrix(R.relu_matrix_cases())\n" % ROOT
    env = {k: v for k, v in os.environ.items() if not k.startswith("CG_GEMM_")}
    env.update(FORCE[force])
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    line = [ln for ln in res.stdout.splitlines() if ln.startswith("RELU_MATRIX ")]
    cases = json.loads(line[-1][len("RELU_MATRIX "):])["cases"]
    assert len(cases) == len(OR.relu_matrix_cases())
    bad = [c for c in cases if not c["guards"] or c["inexact"] or max(c["ratios"].values()) > 1.0]
    assert not bad, bad[:4]
    if force in FORCED_VARIANT:
        ran = {c["epi"] for c in cases if c["variant"] == FORCED_VARIANT[force]}
        assert ran == set(OR.RELU_EPI_NAMES), ran


# ------------------------------------------------------------------------------------------------------- the tower
def _images(n, res, seed):
    return torch.randn(n, 3, res, res, generator=torch.Generator().manual_seed(seed))


def _nhwc_patches(img):
    n, _, res, _ = img.shape
    p = torch.zeros(n, res * res, 8)
    p[..., :3] = img.permute(0, 2, 3, 1).reshape(n, res * res, 3)
    return p.bfloat16()


def _oracle_fwd_bwd(ref, img, demb):
    x = img.clone().requires_grad_()
    emb = ref.encode_image(x)
    (dx,) = torch.autograd.grad(emb, x, demb)
    return emb.detach(), dx


def _device_masks(tower, ws, n):
    """The tower's ReLU on/off patterns (saved outputs > 0) as NCHW bool tensors, in oracle.clip_resnet.relu_modules order."""
    h1 = tower.input_resolution // 2

    def nchw(t, h, c):
        return (t[:, :c].float().cpu() > 0).view(n, h, h, c).permute(0, 3, 1, 2)

    masks = [nchw(t, h1, c.cout) for t, c in zip(ws["stem"], tower.stem)]
    for blk, L, (hi, ho) in zip(tower.blocks, ws["blocks"], tower._geometry()):
        masks += [nchw(L["a1"], hi, blk["planes"]), nchw(L["a2"], hi, blk["planes"]), nchw(L["y"], ho, 4 * blk["planes"])]
    return masks


def _check_tower(name, n, seed):
    """Embedding cosine against the oracle; input gradient against the oracle evaluated with the tower's own ReLU masks (see
    oracle.clip_resnet.fix_relu_masks: bf16 and fp32 evaluations switch a few near-zero units, which a ReLU network's gradient does not
    forgive); the gradient of the unmodified oracle is printed."""
    from clip_diffusion_b200 import models
    from oracle import clip_resnet as OR

    sd = models.random_clip_resnet_state_dict(name, seed=seed)
    mine = models.CLIPModelB200(name, sd, "cuda")
    ref = OR.OracleCLIPResNet(name, sd)
    tower = mine.visual.tower
    res = tower.input_resolution
    img = _images(n, res, seed).bfloat16().float()  # the patches the tower reads are bf16: feed the oracle the same image
    demb = torch.randn(n, tower.output_dim, generator=torch.Generator().manual_seed(seed + 1))
    want, dfree = _oracle_fwd_bwd(ref, img, demb)
    emb = tower.forward_patches(_nhwc_patches(img).cuda())
    _, dwant = _oracle_fwd_bwd(OR.fix_relu_masks(OR.OracleCLIPResNet(name, sd), _device_masks(tower, tower._ws[n], n)), img, demb)
    dp = tower.backward_patches(demb.cuda()).cpu()
    assert torch.isfinite(emb).all() and torch.isfinite(dp).all() and (dp[..., 3:] == 0).all()
    cos = torch.nn.functional.cosine_similarity(emb.cpu(), want, dim=-1).min().item()
    dx = dp[..., :3].reshape(n, res, res, 3).permute(0, 3, 1, 2)
    rel = ((dx - dwant).norm() / dwant.norm()).item()
    rel_free = ((dx - dfree).norm() / dfree.norm()).item()
    # embed_image's path: the fused patchify kernel with patch 1, autograd through _EncodeImageFn (same activations, so same masks)
    from clip_diffusion_b200.utils.functional import embed_image

    x = img.cuda().requires_grad_()
    e2 = embed_image(mine, x, clip_normalize=False)
    (dx2,) = torch.autograd.grad(e2, x, demb.cuda())
    cos2 = torch.nn.functional.cosine_similarity(e2.detach().cpu(), want, dim=-1).min().item()
    rel2 = ((dx2.cpu() - dwant).norm() / dwant.norm()).item()
    print("%s n=%d: cos %.6f / %.6f, dgrad rel-L2 %.3e / %.3e (unmasked oracle: %.3e)" % (name, n, cos, cos2, rel, rel2, rel_free))
    assert cos >= COS_MIN and cos2 >= COS_MIN, (cos, cos2)
    assert rel <= GRAD_REL_MAX and rel2 <= GRAD_REL_MAX, (rel, rel2)


@pytest.mark.parametrize("name", list(TINY))
def test_tiny_tower_matches_oracle(name):
    _register()
    _check_tower(name, 3, seed=21)


def test_rn101_matches_oracle():
    torch.set_num_threads(os.cpu_count() or 1)
    _check_tower("RN101", 2, seed=1)


def test_graph_replay_equals_eager_and_stale_backward_raises():
    from clip_diffusion_b200 import models

    _register()
    name = "test-rn-b"
    sd = models.random_clip_resnet_state_dict(name, seed=4)
    graphed, eager = models.ModifiedResNetB200(name, sd, "cuda"), models.ModifiedResNetB200(name, sd, "cuda")
    eager.use_graphs = False
    for n in (2, 5):
        for it in range(5):
            p = _nhwc_patches(_images(n, 96, 100 * n + it)).cuda()
            d = torch.randn(n, 256, generator=torch.Generator().manual_seed(it)).cuda()
            e1, e2 = graphed.forward_patches(p), eager.forward_patches(p)
            g1, g2 = graphed.backward_patches(d).clone(), eager.backward_patches(d).clone()
            assert torch.equal(e1, e2) and torch.equal(g1, g2), (n, it)
        assert graphed._ws[n]["graphs"]["fwd"]["graph"] is not None
    # deterministic: two runs of the same input agree bit for bit (no float atomics)
    p = _nhwc_patches(_images(2, 96, 7)).cuda()
    d = torch.randn(2, 256).cuda()
    a = (eager.forward_patches(p), eager.backward_patches(d).clone())
    b = (eager.forward_patches(p), eager.backward_patches(d).clone())
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    gen = graphed._generation
    graphed.forward_patches(p)
    graphed.forward_patches(p)
    with pytest.raises(RuntimeError, match="stale"):
        graphed.backward_patches(d, generation=gen + 1)


def test_guidance_step_with_a_vit_and_a_resnet_matches_oracle():
    import copy

    from clip_diffusion_b200 import models
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.rng_record import draw_cutout_record
    from clip_diffusion_b200.sample import GuidanceStep
    from clip_diffusion_b200.unet import create_unet
    from oracle import clip_vit
    from oracle.clip_resnet import OracleCLIPResNet
    from oracle.cond_fn import make_conditon_function

    _register()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    vit = "test-tiny/32"
    models.register_clip_config(vit, *clip_vit.CONFIGS[vit])
    g = torch.Generator().manual_seed(11)
    sd_v, sd_r = models.random_clip_state_dict(vit, seed=5), models.random_clip_resnet_state_dict("test-rn-a", seed=6)
    mine = {vit: models.CLIPModelB200(vit, sd_v, "cuda"), "test-rn-a": models.CLIPModelB200("test-rn-a", sd_r, "cuda")}
    ref = {vit: clip_vit.OracleCLIP(vit, state_dict=sd_v), "test-rn-a": OracleCLIPResNet("test-rn-a", sd_r)}
    text = {vit: {"embeddings": torch.randn(1, 64, generator=g), "weights": torch.tensor(1.0)},
            "test-rn-a": {"embeddings": torch.randn(2, 128, generator=g), "weights": torch.tensor([1.0, -0.5])}}
    text_gpu = {k: {kk: vv.cuda() for kk, vv in v.items()} for k, v in text.items()}
    unet_cpu = create_unet(32, seed=2, device="cpu", use_fp16=False)
    unet_gpu = copy.deepcopy(unet_cpu).cuda()
    diffusion = SpacedDiffusion(steps=50)
    x = torch.randn(1, 3, 128, 128, generator=g)
    records = {}

    def record_source(name, b, H, W, cs, n_over, n_inner, power, gray):
        if (name, b) not in records:
            records[(name, b)] = draw_cutout_record(H, W, cs, n_over, n_inner, power, gray,
                                                    generator=torch.Generator().manual_seed(1000 + len(records)), noise="cpu")
        return records[(name, b)]

    class Cfg:
        num_cutout_batches = 2
        num_overview_cuts_schedule = (3,) * 1000
        num_inner_cuts_schedule = (5,) * 1000
        inner_cut_size_power_schedule = (5,) * 1000
        cut_gray_portion_schedule = (0.3,) * 1000
        grad_threshold = 0.05
        clip_guidance_scale = 8000
        denoise_scale = 10000
        aesthetic_scale = 0

    ct = 30
    f = make_conditon_function(diffusion, unet_cpu, ref, text, lambda: ct, Cfg, record_source)
    ref_out = f(x, diffusion.model_timesteps(torch.tensor([ct])))
    step = GuidanceStep(diffusion, unet_gpu, mine, text_gpu, config=Cfg, record_source=record_source)
    step.current_timestep = ct
    out = step.cond_fn(x.cuda(), diffusion.model_timesteps(torch.tensor([ct], device="cuda")))
    rel_gt = ((step.last_grad_tensor.cpu().view_as(f.last_grad_tensor) - f.last_grad_tensor).norm() / f.last_grad_tensor.norm()).item()
    rel = ((out.cpu() - ref_out).norm() / ref_out.norm()).item()
    print("guidance ViT + RN: d(loss)/d(x_in) rel-L2 %.3e, cond_fn rel-L2 %.3e" % (rel_gt, rel))
    assert rel_gt <= GRAD_REL_MAX and rel <= GRAD_REL_MAX, (rel_gt, rel)


def test_default_four_towers_load_and_step_at_512():
    from clip_diffusion_b200.config import Config
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.models import load_clip_models
    from clip_diffusion_b200.sample import GuidanceStep
    from clip_diffusion_b200.unet import create_unet

    models = load_clip_models(Config.chosen_clip_models, allow_random_init=True)
    assert list(models) == list(Config.chosen_clip_models)
    g = torch.Generator().manual_seed(2)
    text = {k: {"embeddings": torch.randn(1, m.visual.output_dim, generator=g).cuda(), "weights": torch.tensor(1.0, device="cuda")}
            for k, m in models.items()}

    class Cfg:
        num_cutout_batches = 1
        num_overview_cuts_schedule = (4,) * 1000
        num_inner_cuts_schedule = (4,) * 1000
        inner_cut_size_power_schedule = (5,) * 1000
        cut_gray_portion_schedule = (0.3,) * 1000
        grad_threshold = 0.05
        clip_guidance_scale = 8000
        denoise_scale = 10000
        aesthetic_scale = 0

    unet = create_unet(512, seed=2, device="cuda", use_fp16=True, channels_last=True)
    diffusion = SpacedDiffusion(steps=50)
    step = GuidanceStep(diffusion, unet, models, text, config=Cfg)
    x = torch.randn(1, 3, 512, 512, generator=g).cuda()
    out = step.ddim_step(x, 30)
    torch.cuda.synchronize()
    assert torch.isfinite(out["sample"]).all()
    assert step.last_grad_tensor.abs().max().item() > 0


def test_rn101_text_tower_matches_oracle():
    from clip_diffusion_b200 import models
    from oracle import clip_text
    from oracle.clip_text import OracleCLIPText, random_prompt_tokens

    clip_text.TEXT_CONFIGS.setdefault("RN101", models.CLIP_TEXT_CONFIGS["RN101"])  # OpenAI's RN101 text tower: the ViT-B shape
    sd = models.random_clip_text_state_dict("RN101", seed=3)
    mine = models.CLIPModelB200("RN101", dict(models.random_clip_resnet_state_dict("RN101", seed=3), **sd), "cuda")
    ref = OracleCLIPText("RN101", state_dict=sd)
    g = torch.Generator().manual_seed(5)
    tokens = random_prompt_tokens([0, 75, 9, 30], 77, g)
    want = ref.encode_text(tokens)
    got = mine.encode_text(tokens.cuda())
    cos = torch.nn.functional.cosine_similarity(got.cpu(), want, dim=-1)
    assert cos.min().item() >= COS_MIN, cos
