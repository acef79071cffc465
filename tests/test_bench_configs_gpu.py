"""GPU parity on the configurations bench.py actually runs (VERDICT r1 item 1): the CUDA path there is the fp16 NHWC
CUDA-graphed UNet + a full-size bf16 CLIP tower, not the fp32 stock UNet + toy towers of test_cond_fn_gpu.py.

  * c2       512x512 UNet (fp16, channels_last, fused GroupNorm kernels, CUDA graphs) + ViT-B/16, 16 + 16 cutouts:
             one guided DDIM step (GuidanceStep.ddim_step, the call bench.py times) against the fp32 CPU oracle
             (oracle/cond_fn.py = sample.py:134-238 on the fp32 UNet) driven through the same sampler update.
  * c3-style two towers + tv + range loss (rgb_range_loss is dead code in the reference, losses.py:31-35; opt-in).
  * NCCL     the sharded step on 2 real GPUs (2 processes, one all-reduce) equals the single-GPU step; skipped below 2 GPUs.

Tolerances.  The tower alone meets north_star's bf16 bound (rel-L2 <= 1e-2, tests/test_vit_gpu.py).  With the fp16 UNet in
front of and behind it the comparison against an fp32 UNet also carries the fp16 rounding of the trunk: epsilon <= 1e-2 and
d(eps)/dx <= 2e-2 in tests/test_unet_gpu.py at small sizes.  Stated fp16 tolerances here: d(loss)/d(x_in) <= 3e-2, guidance
gradient (after the UNet VJP) <= 6e-2, DDIM sample <= 2e-2 relative L2.
"""
import copy
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL_GRAD_XIN_FP16 = 3e-2
TOL_GUIDANCE_FP16 = 6e-2
TOL_SAMPLE_FP16 = 2e-2


class _Cfg:
    num_cutout_batches = 1
    inner_cut_size_power_schedule = (5,) * 1000
    cut_gray_portion_schedule = (0.3,) * 1000
    grad_threshold = 0.05
    clip_guidance_scale = 8000
    denoise_scale = 10000
    aesthetic_scale = 0


def _cfg(n_over, n_inner):
    class C(_Cfg):
        num_overview_cuts_schedule = (n_over,) * 1000
        num_inner_cuts_schedule = (n_inner,) * 1000

    return C


def _rel(a, b):
    return ((a - b).norm() / b.norm()).item()


def _records():
    from clip_diffusion_b200.rng_record import draw_cutout_record

    recs = {}

    def record_source(nm, b, H, W, cs, n_over, n_inner, power, gray):
        if (nm, b) not in recs:
            recs[(nm, b)] = draw_cutout_record(H, W, cs, n_over, n_inner, power, gray, generator=torch.Generator().manual_seed(7 + len(recs)), noise="cpu")
        return recs[(nm, b)]

    return record_source


def test_c2_ddim_step_with_graphed_nhwc_fp16_unet_matches_oracle():
    """BASELINE configs[1] as bench.py runs it (fp16 NHWC UNet on csrc/unet_norm.cu + cuDNN, captured in CUDA graphs, shared
    grad-enabled forward, dynamic-thresholding kernel) vs the reference path restated on the CPU in fp32."""
    from clip_diffusion_b200 import models
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.sample import GuidanceStep, make_denoised_function
    from clip_diffusion_b200.unet import create_unet, graph_unet
    from oracle.clip_vit import OracleCLIP
    from oracle.cond_fn import make_conditon_function

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_num_threads(os.cpu_count() or 1)
    size, name, cfg = 512, "ViT-B/16", _cfg(16, 16)
    sd = models.random_clip_state_dict(name, seed=1)
    mine = {name: models.CLIPModelB200(name, sd, "cuda")}
    ref = {name: OracleCLIP(name, state_dict=sd)}
    g = torch.Generator().manual_seed(0)
    text = {name: {"embeddings": torch.randn(1, 512, generator=g), "weights": torch.tensor(1.0)}}
    text_gpu = {name: {k: v.cuda() for k, v in text[name].items()}}
    unet_cpu = create_unet(size, seed=2, device="cpu", use_fp16=False)
    unet_gpu = create_unet(size, seed=2, device="cuda", use_fp16=True, channels_last=True)  # same seed => same weights (convs rounded to fp16)
    unet_gpu = graph_unet(unet_gpu, size, size, "cuda")
    diffusion = SpacedDiffusion(steps=250)
    x = torch.randn(1, 3, size, size, generator=g)
    record_source = _records()
    ct = 120
    state = {"ct": ct}

    def denoised_fn_cpu(x_start):  # sample.py:116-132
        thr = torch.quantile(x_start.reshape(x_start.shape[0], -1).abs(), 0.995, dim=-1).clamp(min=1.0).view(-1, 1, 1, 1)
        return x_start.clamp(min=-thr, max=thr) / thr

    oracle_fn = make_conditon_function(diffusion, unet_cpu, ref, text, lambda: state["ct"], cfg, record_source)
    noise = torch.randn(1, 3, size, size, generator=g)
    t = torch.full((1,), ct, dtype=torch.long)
    expected = diffusion.ddim_sample(unet_cpu, x, t, clip_denoised=False, denoised_fn=denoised_fn_cpu, cond_fn=oracle_fn, model_kwargs={}, eta=0.8, noise=noise)
    exp_guidance = oracle_fn(x, diffusion.model_timesteps(t))

    step = GuidanceStep(diffusion, unet_gpu, mine, text_gpu, config=cfg, record_source=record_source)
    step.current_timestep = ct
    got_guidance = step.cond_fn(x.cuda(), diffusion.model_timesteps(t.cuda()))
    rel_gt = _rel(step.last_grad_tensor.cpu().view_as(oracle_fn.last_grad_tensor), oracle_fn.last_grad_tensor)
    rel_guid = _rel(got_guidance.cpu(), exp_guidance)
    got = step.ddim_step(x.cuda(), ct, eta=0.8, denoised_fn=make_denoised_function(0.995), noise=noise.cuda())
    print("c2 fp16-NHWC-graphed: d(loss)/d(x_in) rel-L2 %.3e, guidance rel-L2 %.3e" % (rel_gt, rel_guid))
    assert rel_gt <= TOL_GRAD_XIN_FP16, rel_gt
    assert rel_guid <= TOL_GUIDANCE_FP16, rel_guid
    rel_s = _rel(got["sample"].cpu().float(), expected["sample"])
    rel_p = _rel(got["pred_xstart"].cpu().float(), expected["pred_xstart"])
    print("c2 fp16-NHWC-graphed: DDIM sample rel-L2 %.3e, pred_xstart rel-L2 %.3e" % (rel_s, rel_p))
    assert rel_s <= TOL_SAMPLE_FP16 and rel_p <= TOL_SAMPLE_FP16, (rel_s, rel_p)


def test_c3_style_two_towers_with_range_loss_matches_oracle():
    """configs[2] flavour at a size the CPU oracle finishes in seconds: two real towers (ViT-B/32 + ViT-B/16), tv + range loss,
    fp32 UNet (so the bound is north_star's bf16 tolerance, 1e-2)."""
    from clip_diffusion_b200 import models
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.sample import GuidanceStep
    from clip_diffusion_b200.unet import create_unet
    from oracle.clip_vit import OracleCLIP
    from oracle.cond_fn import make_conditon_function

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = _cfg(3, 5)
    mine, ref, text = {}, {}, {}
    g = torch.Generator().manual_seed(3)
    for i, name in enumerate(("ViT-B/32", "ViT-B/16")):
        sd = models.random_clip_state_dict(name, seed=1 + i)
        mine[name] = models.CLIPModelB200(name, sd, "cuda")
        ref[name] = OracleCLIP(name, state_dict=sd)
        text[name] = {"embeddings": torch.randn(1, 512, generator=g), "weights": torch.tensor(1.0)}
    text_gpu = {k: {kk: vv.cuda() for kk, vv in v.items()} for k, v in text.items()}
    unet_cpu = create_unet(32, seed=2, device="cpu", use_fp16=False)
    unet_gpu = copy.deepcopy(unet_cpu).cuda()
    diffusion = SpacedDiffusion(steps=50)
    x = torch.randn(1, 3, 256, 256, generator=g) * 1.5  # |x| > 1 in places: the range loss is active
    record_source = _records()
    ct = 20
    oracle_fn = make_conditon_function(diffusion, unet_cpu, ref, text, lambda: ct, cfg, record_source, range_scale=150.0)
    expected = oracle_fn(x, diffusion.model_timesteps(torch.tensor([ct])))
    step = GuidanceStep(diffusion, unet_gpu, mine, text_gpu, config=cfg, record_source=record_source, range_scale=150.0)
    step.current_timestep = ct
    got = step.cond_fn(x.cuda(), diffusion.model_timesteps(torch.tensor([ct], device="cuda")))
    rel_gt = _rel(step.last_grad_tensor.cpu().view_as(oracle_fn.last_grad_tensor), oracle_fn.last_grad_tensor)
    rel = _rel(got.cpu(), expected)
    print("c3-style: d(loss)/d(x_in) rel-L2 %.3e, guidance rel-L2 %.3e" % (rel_gt, rel))
    assert rel_gt <= 1e-2 and rel <= 1e-2, (rel_gt, rel)
    # the range term really contributed
    step0 = GuidanceStep(diffusion, unet_gpu, mine, text_gpu, config=cfg, record_source=record_source, range_scale=0.0)
    step0.current_timestep = ct
    step0.cond_fn(x.cuda(), diffusion.model_timesteps(torch.tensor([ct], device="cuda")))
    assert (step0.last_grad_tensor - step.last_grad_tensor).abs().max().item() > 0


def _nccl_worker(rank, world, port, out_path):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from clip_diffusion_b200 import models
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.sample import GuidanceStep
    from clip_diffusion_b200.unet import create_unet

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = _cfg(5, 6)  # 11 cutouts: an uneven 6 + 5 split
    name = "ViT-B/32"
    mine = {name: models.CLIPModelB200(name, models.random_clip_state_dict(name, seed=1), "cuda")}
    g = torch.Generator().manual_seed(0)
    text = {name: {"embeddings": torch.randn(1, 512, generator=g).cuda(), "weights": torch.tensor(1.0).cuda()}}
    unet = create_unet(32, seed=2, device="cuda", use_fp16=False)
    diffusion = SpacedDiffusion(steps=50)
    x = torch.randn(1, 3, 256, 256, generator=g).cuda()
    ct = 25
    t = diffusion.model_timesteps(torch.tensor([ct], device="cuda"))
    sharded = GuidanceStep(diffusion, unet, mine, text, config=cfg, record_source=_records(), rank=rank, world_size=world)
    sharded.current_timestep = ct
    out = sharded.cond_fn(x, t)
    torch.cuda.synchronize()
    # every rank must hold the same reduced gradient
    gathered = [torch.empty_like(out) for _ in range(world)]
    dist.all_gather(gathered, out.contiguous())
    # identical up to the run-to-run noise of the replicated fp32 UNet VJP (cuDNN algorithms with atomics): the reduced d(loss)/d(x_in)
    # itself is bit-identical on every rank
    same = all(((gathered[0] - o).norm() / gathered[0].norm()).item() <= 1e-5 for o in gathered)
    gt = [torch.empty_like(sharded.last_grad_tensor) for _ in range(world)]
    dist.all_gather(gt, sharded.last_grad_tensor.contiguous())
    same = same and all(torch.equal(gt[0], o) for o in gt)
    if rank == 0:
        single = GuidanceStep(diffusion, unet, mine, text, config=cfg, record_source=_records())
        single.current_timestep = ct
        ref = single.cond_fn(x, t)
        torch.save({"rel": _rel(out, ref), "rel_gt": _rel(sharded.last_grad_tensor, single.last_grad_tensor), "same": same,
                    "processed": sharded.cutouts_processed}, out_path)
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_step_over_nccl_equals_single_gpu(tmp_path):
    """north_star (4) on real devices: 2 processes, each with its slice of the cutouts, ONE NCCL all-reduce of the image gradient."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    out = str(tmp_path / "nccl.pt")
    port = 29750 + (os.getpid() % 200)
    mp.spawn(_nccl_worker, args=(2, port, out), nprocs=2, join=True)
    res = torch.load(out)
    print("NCCL 2-rank: guidance rel-L2 %.3e, d(loss)/d(x_in) rel-L2 %.3e" % (res["rel"], res["rel_gt"]))
    assert res["same"], "ranks disagree after the all-reduce"
    assert res["processed"] == 6
    assert res["rel_gt"] <= 2e-3 and res["rel"] <= 2e-3, res
