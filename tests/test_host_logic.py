"""CPU tests of the host logic: C-ABI library loads and exports every declared symbol, struct layouts, RNG-record
slicing, shard ranges, diffusion schedule, UNet shapes/parameter counts, loud failure without CUDA."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_in_the_header_at_abi_v5():
    """Every declared entry point is exported and bound, at ABI version 5 (v5 added cg_gemm_tile_variant)."""
    from clip_diffusion_b200 import _lib

    header = open(os.path.join(ROOT, "include", "clipguide_b200.h")).read()
    declared = set(re.findall(r"\b(cg_[a-z0-9_]+)\s*\(", header))
    declared -= {"cg_cut_t", "cg_aug_t"}
    assert len(declared) >= 24
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), "libclipguide_b200.so does not export %s" % name
    assert declared == set(_lib.exported_symbols()), declared ^ set(_lib.exported_symbols())
    assert _lib.load().cg_abi_version() == 5
    assert _lib.load()._cg_missing == []


def test_struct_layouts_match_the_header():
    from clip_diffusion_b200 import _lib

    assert ctypes.sizeof(_lib.CgCut) == 16
    assert ctypes.sizeof(_lib.CgAug) == 184
    assert _lib.CgAug.noise_seed.offset == 120 and _lib.CgAug.input01.offset == 140
    assert _lib.CgAug.noise_mode.offset == 144 and _lib.CgAug.noise_offset.offset == 152 and _lib.CgAug.noise_total.offset == 176


def test_ops_refuse_cpu_tensors_and_bad_arguments_without_a_gpu():
    from clip_diffusion_b200 import _lib, losses
    from clip_diffusion_b200.cutouts import make_cutouts

    with pytest.raises(_lib.ClipGuideError):
        losses.total_variational_loss(torch.zeros(1, 3, 8, 8))
    with pytest.raises(_lib.ClipGuideError):
        make_cutouts(torch.zeros(1, 3, 64, 64), 32, 1, 1, 5, 0.3)
    lib = _lib.load()
    # argument validation happens before any CUDA call
    assert lib.cg_tv_loss_fwd_bwd(None, 1, 3, 8, 8, 1.0, 0, None, None, None) == -1
    assert b"bad arguments" in lib.cg_last_error()
    assert lib.cg_gemm_bf16_tn(ctypes.c_void_p(16), ctypes.c_void_p(16), 8, 100, 64, 64, 64, 4, None, ctypes.c_void_p(16), None, 128, None, 0, None) == -1
    assert b"multiple of 128" in lib.cg_last_error()
    assert lib.cg_cutouts_workspace_bytes(0, 224, 512) == 0 and lib.cg_cutouts_workspace_bytes(16, 224, 512) > 16 * 3 * 224 * 224 * 4 * 3


def test_record_slices_and_shard_ranges():
    from clip_diffusion_b200.rng_record import draw_cutout_record
    from clip_diffusion_b200.sample import shard_range

    g = torch.Generator().manual_seed(3)
    rec = draw_cutout_record(512, 768, 224, 5, 11, 5, 0.3, generator=g, noise="cpu")
    assert rec.num_cuts == 16 and rec.size[:5] == [768] * 5 and rec.y0[0] == -128 and rec.x0[0] == 0
    assert all(224 <= s <= 512 for s in rec.size[5:])
    assert all(0 <= x <= 768 - s and 0 <= y <= 512 - s for x, y, s in zip(rec.x0[5:], rec.y0[5:], rec.size[5:]))
    for world in (1, 2, 3, 8, 16, 20):
        spans = [shard_range(16, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == 16 and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1
        joined = []
        for a, b in spans:
            s = rec.slice(a, b)
            assert s.first_index() == a and (s.flip, s.angle, s.perm, s.hue) == (rec.flip, rec.angle, rec.perm, rec.hue)
            assert s.noise[0].shape[0] == b - a
            joined += s.size
        assert joined == rec.size
    m = rec.inverse_affine_matrix()
    from torchvision.transforms.functional import _get_inverse_affine_matrix

    assert m == _get_inverse_affine_matrix([0.0, 0.0], rec.angle, [float(rec.tx), float(rec.ty)], 1.0, [0.0, 0.0])


def test_pack_record_affine_inverse():
    from clip_diffusion_b200.cutouts import pack_record
    from clip_diffusion_b200.rng_record import draw_cutout_record

    rec = draw_cutout_record(256, 256, 224, 2, 2, 5, 0.3, generator=torch.Generator().manual_seed(1), noise="device")
    cuts, aug = pack_record(rec, normalize=True)
    a = torch.tensor(list(aug.theta), dtype=torch.float64).view(2, 3)
    f = torch.tensor(list(aug.theta_fwd), dtype=torch.float64).view(2, 3)
    A = torch.cat([a, torch.tensor([[0, 0, 1.0]], dtype=torch.float64)])
    F = torch.cat([f, torch.tensor([[0, 0, 1.0]], dtype=torch.float64)])
    assert (A @ F - torch.eye(3, dtype=torch.float64)).abs().max().item() < 1e-5
    assert cuts[0].size == 256 and aug.normalize == 1 and abs(aug.noise_std - 0.01) < 1e-9


def test_diffusion_schedule_and_unet():
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.unet import UNetModel, create_unet

    d = SpacedDiffusion(steps=250)
    assert d.num_timesteps == 250 and d.timestep_map[0] == 0 and d.timestep_map[-1] == 996
    assert float(d.model_timesteps(torch.tensor([249]))) == 996.0
    assert abs(d.alphas_cumprod[-1] - 4.2e-5) < 2e-5
    m = create_unet(32, device="cpu", use_fp16=False)
    x = torch.randn(1, 3, 32, 32, requires_grad=True)
    out = d.p_mean_variance(m, x, torch.tensor([100]), clip_denoised=False)
    assert out["pred_xstart"].shape == x.shape
    (g,) = torch.autograd.grad(out["pred_xstart"].sum(), x)
    assert torch.isfinite(g).all()
    # sampler step with a dummy cond_fn: receives the ORIGINAL timestep (sample.py:157-159 relies on it)
    seen = []
    d.ddim_sample(m, x.detach(), torch.tensor([100]), cond_fn=lambda xx, t, **kw: seen.append(float(t)) or torch.zeros_like(xx))
    assert seen == [400.0]
    with torch.device("meta"):
        n512 = sum(p.numel() for p in UNetModel(512, use_fp16=False).parameters())
        n256 = sum(p.numel() for p in UNetModel(256, use_fp16=False).parameters())
    assert abs(n512 / 1e6 - 558.0) < 0.1 and abs(n256 / 1e6 - 552.8) < 0.1  # SURVEY.md App. A.3 parameter counts


def test_groupnorm_workspace_query_is_host_only_and_sane():
    """cg_groupnorm_nhwc_workspace_bytes needs no GPU: chunk partials (float2 per channel and chunk) + two coefficient rows."""
    from clip_diffusion_b200 import _lib

    lib = _lib.load()
    assert lib.cg_groupnorm_nhwc_workspace_bytes(1, 64, 12) == 0 and lib.cg_groupnorm_nhwc_workspace_bytes(0, 64, 16) == 0  # C % 8, N < 1
    small, big = lib.cg_groupnorm_nhwc_workspace_bytes(1, 64, 1024), lib.cg_groupnorm_nhwc_workspace_bytes(1, 512 * 512, 128)
    assert small >= 2 * 1024 * 4 + 1024 * 8 and big >= 2 * 128 * 4 + 128 * 8
    assert big <= 16 << 20  # bounded: ~8 chunks per SM at most
    assert lib.cg_groupnorm_nhwc_workspace_bytes(2, 4096, 256) % 16 == 0


def test_groupnorm_chunk_geometry_covers_every_row_once():
    """Launch geometry of csrc/unet_norm.cu (host-only query): threads = octets x row lanes <= 256, the row chunks tile [0, HW)
    without gap or overlap, chunks are whole unrolled iterations when the map is large, and the workspace holds all partials."""
    import ctypes as C

    from clip_diffusion_b200 import _lib

    lib = _lib.load()
    out = (C.c_int * 5)()
    shapes = [(1, 512 * 512, 128), (1, 512 * 512, 256), (1, 768 * 768, 128), (1, 256 * 256, 512), (1, 64, 1024), (1, 256, 2048), (2, 63, 32),
              (3, 33 * 31, 256), (1, 24 * 40, 384), (1, 1, 8), (7, 4096, 1536), (1, 96 * 96, 768), (64, 16, 64)]
    for n, hw, c in shapes:
        assert lib.cg_groupnorm_nhwc_geometry(n, hw, c, out) == 0
        cvecs, rpi, threads, chunks, rpc = list(out)
        assert cvecs == c // 8 and rpi >= 1 and threads == cvecs * rpi and threads <= 256
        assert chunks >= 1 and rpc >= 1 and chunks * rpc >= hw and (chunks - 1) * rpc < hw  # exact tiling of the rows
        if hw >= 64 * rpi * 4:
            assert rpc % (rpi * 4) == 0  # whole unrolled iterations per chunk
            assert chunks * n <= 8 * 148 + n  # ~8 CTAs per SM
        assert lib.cg_groupnorm_nhwc_workspace_bytes(n, hw, c) >= n * chunks * c * 8 + 2 * n * c * 4
    assert lib.cg_groupnorm_nhwc_geometry(1, 64, 12, out) != 0 and lib.cg_groupnorm_nhwc_geometry(1, 64, 4096, out) != 0


def test_nhwc_unet_is_never_built_or_run_without_its_kernels():
    """channels_last=True means the sm_100a kernels: refused on the CPU / in fp32, and an NHWC GroupNorm32 fed anything else raises."""
    from clip_diffusion_b200.unet import GroupNorm32, create_unet

    with pytest.raises(ValueError):
        create_unet(32, device="cpu", use_fp16=False, channels_last=True)
    gn = GroupNorm32(4, 16)
    gn.nhwc = True
    with pytest.raises(RuntimeError):
        gn(torch.zeros(1, 16, 4, 4))


def test_group_norm32_stock_path_spells_the_resblock_arithmetic():
    """GroupNorm32(x, scale_shift, silu) on the CPU / fp32 path == silu(GN(x) * (1 + scale) + shift) (guided-diffusion ResBlock)."""
    from torch.nn import functional as Fn

    from clip_diffusion_b200.unet import GroupNorm32

    g = torch.Generator().manual_seed(0)
    gn = GroupNorm32(4, 16)
    with torch.no_grad():
        gn.weight.copy_(torch.randn(16, generator=g))
        gn.bias.copy_(torch.randn(16, generator=g))
    x = torch.randn(2, 16, 5, 7, generator=g)
    ss = torch.randn(2, 32, generator=g)
    want = Fn.group_norm(x, 4, gn.weight, gn.bias, gn.eps)
    assert torch.allclose(gn(x), want, atol=1e-6)
    want = Fn.silu(want * (1 + ss[:, :16, None, None]) + ss[:, 16:, None, None])
    assert torch.allclose(gn(x, scale_shift=ss, silu=True), want, atol=1e-6)


def test_ms_ssim_oracle_properties():
    """oracle.ms_ssim (restated pytorch_msssim.MS_SSIM, parity unpinned): identity, symmetry, monotone in noise, differentiable; the
    product's structural_dissimilarity_loss is CUDA-only and refuses CPU tensors."""
    from clip_diffusion_b200 import _lib
    from clip_diffusion_b200.losses import structural_dissimilarity_loss
    from oracle.ms_ssim import ms_ssim
    from oracle.ms_ssim import structural_dissimilarity_loss as oracle_loss

    g = torch.Generator().manual_seed(0)
    x = torch.rand(1, 3, 192, 192, generator=g, dtype=torch.float64)
    y = torch.rand(1, 3, 192, 192, generator=g, dtype=torch.float64)
    assert abs(ms_ssim(x, x).item() - 1.0) < 1e-9
    vals = [ms_ssim(x, (x + s * torch.randn(x.shape, generator=g, dtype=torch.float64)).clamp(0, 1)).item() for s in (0.02, 0.1, 0.3)]
    assert vals[0] > vals[1] > vals[2] > 0
    assert abs(ms_ssim(x, y).item() - ms_ssim(y, x).item()) < 1e-9
    xx = (x * 2 - 1).requires_grad_()
    loss = oracle_loss(xx, y * 2 - 1)
    (gx,) = torch.autograd.grad(loss, xx)
    assert 0 < loss.item() < 1 and torch.isfinite(gx).all() and gx.abs().max().item() > 0
    with pytest.raises(ValueError):
        ms_ssim(x[..., :100, :100], y[..., :100, :100])
    with pytest.raises(_lib.ClipGuideError):
        structural_dissimilarity_loss(x.float(), y.float())

def test_guided_diffusion_checkpoint_key_mapping_covers_the_whole_unet():
    """ADVICE r1: the reference loads a guided-diffusion checkpoint with model.load_state_dict (models.py:118-124); the key
    mapping must cover every parameter of this UNet, follow guided-diffusion's naming and round-trip the tensors."""
    from clip_diffusion_b200.unet import create_unet, guided_diffusion_key, load_guided_diffusion_state_dict

    m = create_unet(64, seed=2, device="cpu", use_fp16=False)
    own = m.state_dict()
    gd = {guided_diffusion_key(k): torch.randn(v.shape, generator=torch.Generator().manual_seed(i)) for i, (k, v) in enumerate(own.items())}
    assert len(gd) == len(own), "two parameters map to the same guided-diffusion key"
    # guided-diffusion naming landmarks (SURVEY.md App. A.3)
    for key in ("time_embed.0.weight", "time_embed.2.bias", "input_blocks.0.0.weight", "input_blocks.1.0.in_layers.0.weight",
                "input_blocks.1.0.in_layers.2.weight", "input_blocks.1.0.emb_layers.1.weight", "input_blocks.1.0.out_layers.0.bias",
                "input_blocks.1.0.out_layers.3.weight", "middle_block.1.norm.weight", "middle_block.1.qkv.weight", "middle_block.1.proj_out.weight",
                "middle_block.0.in_layers.2.bias", "out.0.weight", "out.2.weight"):
        assert key in gd, key
    assert any(k.endswith("skip_connection.weight") for k in gd)
    assert not any(".layers." in k or ".in_norm." in k or ".emb." in k for k in gd)
    load_guided_diffusion_state_dict(m, gd)
    for k, v in m.state_dict().items():
        assert torch.equal(v, gd[guided_diffusion_key(k)]), k
    bad = dict(gd)
    bad.pop("out.2.weight")
    with pytest.raises(KeyError):
        load_guided_diffusion_state_dict(m, bad)
    bad = dict(gd)
    bad["out.2.weight"] = torch.zeros(1)
    with pytest.raises(ValueError):
        load_guided_diffusion_state_dict(m, bad)


def test_unet_weight_caches_are_invalidated_by_load_state_dict():
    from clip_diffusion_b200.unet import ResBlock, create_unet

    m = create_unet(32, seed=2, device="cpu", use_fp16=False)
    m._emb_cat = ("stale",)
    blocks = [b for b in m.modules() if isinstance(b, ResBlock)]
    blocks[0]._fused_bias = ("stale",)
    m.load_state_dict(m.state_dict())
    assert m._emb_cat is None and blocks[0]._fused_bias is None
    m._emb_cat = ("stale",)
    m.float()
    assert m._emb_cat is None


def test_missing_clip_weights_are_an_error_unless_random_init_is_requested(tmp_path, monkeypatch):
    from clip_diffusion_b200 import models

    monkeypatch.delenv("CLIPGUIDE_B200_WEIGHTS", raising=False)
    with pytest.raises(FileNotFoundError):
        models.load_clip_models(["ViT-B/32"], "cpu")
    monkeypatch.setenv("CLIPGUIDE_B200_WEIGHTS", str(tmp_path))
    with pytest.raises(FileNotFoundError):
        models.load_clip_models(["ViT-B/32"], "cpu")
    torch.save({"visual.conv1.weight": torch.zeros(1)}, str(tmp_path / "ViT-B_32.pt"))
    with pytest.raises(KeyError):
        models.load_clip_models(["ViT-B/32"], "cpu")
    with pytest.raises(ValueError):
        models.load_clip_models(["RN101"], "cpu", allow_random_init=True)
    assert set(models.random_clip_state_dict_keys("ViT-B/32")) == set(models.random_clip_state_dict("ViT-B/32"))
