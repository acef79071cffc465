"""CPU tests that PIN the oracle (section 8(c)): against the reference's own modules executed in place (build container,
/root/reference present), against the committed golden vectors those modules produced (everywhere), and against
independent implementations for the un-vendored third-party pieces (torch's antialiased bicubic for ResizeRight,
transformers' CLIP for the OpenAI ViT)."""
import os

import pytest
import torch

from clip_diffusion_b200.rng_record import draw_cutout_record
from oracle import cutouts as OC
from oracle import losses as OL
from oracle import ref_stubs
from oracle import resize_right as RR

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
needs_reference = pytest.mark.skipif(not ref_stubs.available(), reason="needs the original clip-diffusion source tree (set CLIPGUIDE_REFERENCE_ROOT); "
                                     "test_golden_* compare with what it produced")


def test_golden_cutouts_bit_exact():
    """oracle.cutouts + our RNG record reproduce, bit for bit, what the reference's Cutouts.forward produced."""
    for item in torch.load(os.path.join(GOLDEN, "cutouts_reference.pt")):
        H, W, cs, no, ni, p, gp, seed = item["args"]
        torch.manual_seed(seed)
        rec = draw_cutout_record(H, W, cs, no, ni, p, gp, noise="cpu")
        out = OC.make_cutouts(item["x"], rec)
        assert out.shape == item["out"].shape
        assert torch.equal(out, item["out"]), "case %s: max diff %g" % (item["args"], (out - item["out"]).abs().max())


def test_golden_losses():
    g = torch.load(os.path.join(GOLDEN, "losses_reference.pt"))
    x = g["x"].clone().requires_grad_()
    tv = OL.total_variational_loss(x)
    assert torch.equal(tv.detach(), g["tv"])
    assert torch.equal(torch.autograd.grad(tv.sum(), x)[0], g["gtv"])
    rg = OL.rgb_range_loss(x)
    assert torch.equal(rg.detach(), g["range"])
    assert torch.equal(torch.autograd.grad(rg.sum(), x)[0], g["grange"])
    e = g["emb"].clone().requires_grad_()
    sp = OL.square_spherical_distance_loss(e, g["txt"])
    assert torch.equal(sp.detach(), g["sph"])
    assert torch.equal(torch.autograd.grad(sp.sum(), e)[0], g["gsph"])
    assert torch.equal(OC.clip_normalize(g["x"][:, :, :8, :8]), g["clip_normalize"])


def test_golden_config_schedules():
    from clip_diffusion_b200.config import Config

    g = torch.load(os.path.join(GOLDEN, "config_reference.pt"))
    assert Config.num_overview_cuts_schedule == g["over"] and Config.num_inner_cuts_schedule == g["inner"]
    assert Config.inner_cut_size_power_schedule == g["power"] and Config.cut_gray_portion_schedule == g["gray"]
    assert (Config.grad_threshold, Config.clip_guidance_scale, Config.denoise_scale, Config.num_cutout_batches) == (
        g["grad_threshold"], g["clip_guidance_scale"], g["denoise_scale"], g["num_cutout_batches"])
    Config.update(width=700, height=500, clip_guidance_scale=5)
    assert (Config.width, Config.height, Config.clip_guidance_scale, Config.denoise_scale) == (640, 448, 5, 10000)
    Config.update()
    assert (Config.width, Config.height, Config.clip_guidance_scale) == (768, 512, 8000)
    with pytest.raises(TypeError):
        Config.update(bogus=1)


@needs_reference
@pytest.mark.parametrize("case", [(256, 256, 224, 4, 4, 5, 0.3, 0), (128, 192, 64, 12, 4, 5, 0.3, 1), (192, 128, 96, 0, 5, 5, 0.0, 3), (160, 160, 64, 3, 0, 5, 0.3, 5),
                                  (96, 96, 64, 16, 16, 5, 0.3, 4), (64, 64, 64, 2, 2, 5, 1.0, 6)])
def test_reference_in_place_cutouts(case):
    """The reference's own cutouts.py run unmodified (stub imports) == oracle on the record drawn from the same seed."""
    cut, _, _, _ = ref_stubs.install()
    H, W, cs, no, ni, p, gp, seed = case
    x = torch.tanh(torch.randn(1, 3, H, W, generator=torch.Generator().manual_seed(seed))) * 1.1
    torch.manual_seed(seed)
    ref = cut.make_cutouts(x, cs, no, ni, p, gp)
    after_ref = torch.rand(1)
    torch.manual_seed(seed)
    rec = draw_cutout_record(H, W, cs, no, ni, p, gp, noise="cpu")
    after_rec = torch.rand(1)
    assert torch.equal(after_ref, after_rec), "RNG record consumed a different number of draws than the reference"
    assert torch.equal(OC.make_cutouts(x, rec), ref)
    # quirks (SURVEY App. C): inner cut 0 is always gray; > 4 overview cuts are identical plain copies
    if ni > 0:
        assert rec.flags[no] & 1
    if no > 4:
        assert all(f == rec.flags[0] for f in rec.flags[:no])


@needs_reference
def test_reference_in_place_losses():
    _, los, fun, _ = ref_stubs.install()
    x = torch.randn(2, 3, 33, 47) * 1.3
    assert torch.equal(los.total_variational_loss(x), OL.total_variational_loss(x))
    assert torch.equal(los.rgb_range_loss(x), OL.rgb_range_loss(x))
    a, b = torch.randn(5, 1, 32), torch.randn(1, 3, 32)
    assert torch.equal(los.square_spherical_distance_loss(a, b), OL.square_spherical_distance_loss(a, b))
    pred = OL.LinearAestheticPredictor(32)
    assert torch.equal(los.aesthetic_loss(pred, a[:, 0]), OL.aesthetic_loss(pred, a[:, 0]))
    assert torch.equal(fun.CLIP_NORMALIZE(x.abs()), OC.clip_normalize(x.abs()))


# ---- ResizeRight restatement: independent cross-checks (the real package is not available: parity unpinned) -------------
@pytest.mark.parametrize("size,cs", [(512, 224), (300, 224), (97, 64), (768, 336), (1280, 224), (128, 224), (256, 336), (64, 224)])
def test_resize_matches_torch_antialiased_bicubic_in_the_interior(size, cs):
    """Down- AND up-sampling (the min_size = min(W, H, cut_size) branch of cutouts.py:52 upsamples images smaller than the CLIP
    resolution): torch's antialiased bicubic uses the same Keys a = -0.5 kernel, stretched only when downsampling."""
    x = torch.rand(1, 3, size, size, generator=torch.Generator().manual_seed(size))
    mine = RR.resize(x, out_shape=[1, 3, cs, cs])
    ref = torch.nn.functional.interpolate(x, size=(cs, cs), mode="bicubic", antialias=True, align_corners=False)
    m = max(4, int(2 * max(cs / size, 1.0) + 2))  # borders differ by design: ResizeRight zero-pads and keeps the padded taps in the normalisation
    assert (mine[..., m:-m, m:-m] - ref[..., m:-m, m:-m]).abs().max().item() < 5e-5


def test_resize_identity_partition_of_unity_and_border_darkening():
    x = torch.rand(1, 3, 64, 64)
    assert torch.equal(RR.resize(x, out_shape=[1, 3, 64, 64]), x)
    ones = torch.ones(1, 1, 100, 100)
    out = RR.resize(ones, out_shape=[1, 1, 40, 40])
    assert (out[..., 3:-3, 3:-3] - 1).abs().max().item() < 1e-6  # weights sum to one
    assert out[0, 0, 0, 0].item() < 0.9  # zero padding darkens the border
    left, w = RR.dim_tables(100, 40)
    assert w.shape == (40, 10) and (w.sum(1) - 1).abs().max().item() < 1e-6 and int(left[0]) < 0


# ---- OpenAI ViT restatement vs transformers' CLIP --------------------------------------------------------------------
def test_oracle_vit_matches_hf_clip():
    from transformers import CLIPVisionConfig, CLIPVisionModelWithProjection

    from oracle.clip_vit import CONFIGS, OracleCLIP, random_state_dict

    name = "test-small/16"
    res, patch, width, layers, heads, embed = CONFIGS[name]
    sd = random_state_dict(name)
    m = OracleCLIP(name, state_dict=sd)
    hf = CLIPVisionModelWithProjection(CLIPVisionConfig(hidden_size=width, intermediate_size=4 * width, projection_dim=embed, num_hidden_layers=layers,
                                                        num_attention_heads=heads, image_size=res, patch_size=patch, hidden_act="quick_gelu",
                                                        attention_dropout=0.0)).eval()
    hs = {"vision_model.embeddings.class_embedding": sd["visual.class_embedding"],
          "vision_model.embeddings.patch_embedding.weight": sd["visual.conv1.weight"],
          "vision_model.embeddings.position_embedding.weight": sd["visual.positional_embedding"],
          "vision_model.pre_layrnorm.weight": sd["visual.ln_pre.weight"], "vision_model.pre_layrnorm.bias": sd["visual.ln_pre.bias"],
          "vision_model.post_layernorm.weight": sd["visual.ln_post.weight"], "vision_model.post_layernorm.bias": sd["visual.ln_post.bias"],
          "visual_projection.weight": sd["visual.proj"].t()}
    for i in range(layers):
        p, q = "visual.transformer.resblocks.%d." % i, "vision_model.encoder.layers.%d." % i
        w, b = sd[p + "attn.in_proj_weight"], sd[p + "attn.in_proj_bias"]
        for j, n in enumerate("qkv"):
            hs[q + "self_attn.%s_proj.weight" % n] = w[j * width:(j + 1) * width]
            hs[q + "self_attn.%s_proj.bias" % n] = b[j * width:(j + 1) * width]
        for a, c in (("self_attn.out_proj", "attn.out_proj"), ("layer_norm1", "ln_1"), ("layer_norm2", "ln_2"), ("mlp.fc1", "mlp.c_fc"), ("mlp.fc2", "mlp.c_proj")):
            hs[q + a + ".weight"], hs[q + a + ".bias"] = sd[p + c + ".weight"], sd[p + c + ".bias"]
    missing = hf.load_state_dict(hs, strict=False)
    assert not missing.unexpected_keys and all("position_ids" in k for k in missing.missing_keys)
    x = torch.randn(2, 3, res, res)
    with torch.no_grad():
        assert (m.encode_image(x) - hf(pixel_values=x).image_embeds).abs().max().item() < 1e-5


def test_product_and_oracle_share_state_dict_layout():
    from clip_diffusion_b200 import models
    from oracle.clip_vit import OracleCLIP, random_state_dict

    for name in ("ViT-B/32",):
        a, b = models.random_clip_state_dict(name), random_state_dict(name)
        assert a.keys() == b.keys() and all(a[k].shape == b[k].shape for k in a)
    models.register_clip_config("test-tiny/32", 64, 32, 128, 2, 2, 64)
    OracleCLIP("test-tiny/32", state_dict=models.random_clip_state_dict("test-tiny/32"))
