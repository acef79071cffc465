"""Timings of CLIP's RN101 image tower (ModifiedResNetB200) on the sm_100a kernels, with CUDA events after warm-up:
  * forward + input gradient (forward_patches + backward_patches, graph-replayed) at N = 16 and 64 cutouts, median of 20 calls;
  * per kernel family, from per-call CUDA events of one eager pass at N = 64 (_lib.PROFILE, as bench.py does): GEMM TFLOP/s and
    im2col / pool GB/s (algorithmic bytes: what each kernel must read and write once) against the sustained peaks;
  * the stock-PyTorch arm: the oracle module (oracle/clip_resnet.py) on the GPU in bf16, channels_last, cuDNN, gradient to the input only;
  * one guided DDIM step at 512x512 with the default four towers (Config.chosen_clip_models) and with the three ViTs only.
Random weights (seeded): throughput does not depend on the values.  The GPU name, power limit and max SM clock are printed in the same
run, and the output is also written to profiles/r03_resnet_bench.txt.
Usage (GPU machine):  python tools/bench_resnet.py"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch

from bench_text import device_line, timeit
from clip_diffusion_b200 import _lib, models

OUT = os.path.join(ROOT, "profiles", "r03_resnet_bench.txt")
LINES = []


def say(s):
    print(s, flush=True)
    LINES.append(s)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1367.9), d.get("hbm_gbs", 6555.0)
    return 1367.9, 6555.0  # the sustained bf16 rate and HBM bandwidth measured on the B200 (MEASURED_PEAKS.json of the measuring runs)


FAMILY = {"cg_gemm_bf16_tn": "gemm", "cg_gemm_bf16_tn_relu": "gemm", "cg_im2col3x3_nhwc": "im2col", "cg_avgpool2x2_nhwc_fwd": "avgpool",
          "cg_avgpool2x2_nhwc_bwd": "avgpool", "cg_attention_fwd": "attention", "cg_attention_bwd": "attention",
          "cg_conv3x3s2_dgrad": "stem dgrad", "cg_resnet_attnpool_fwd": "attnpool", "cg_resnet_attnpool_bwd": "attnpool",
          "cg_resnet_attnpool_dctx": "attnpool", "cg_vit_proj_bwd": "attnpool"}


def work(name, a):
    """(FLOPs, algorithmic bytes) of one call from its arguments."""
    if name.startswith("cg_gemm"):
        return 2.0 * a[2] * a[3] * a[4], 0.0
    if name == "cg_im2col3x3_nhwc":
        n, h, w, c, stride, kpad = a[1], a[2], a[3], a[4], a[6], a[7]
        ho, wo = (h - 1) // stride + 1, (w - 1) // stride + 1
        return 0.0, 2.0 * (n * h * w * c + n * ho * wo * kpad)
    if name == "cg_avgpool2x2_nhwc_fwd":
        n, h, w, c = a[1], a[2], a[3], a[4]
        return 0.0, 2.0 * n * h * w * c * 1.25
    if name == "cg_avgpool2x2_nhwc_bwd":
        dy_f32, mask, n, h, w, c, dx_f32 = a[1], a[2], a[3], a[4], a[5], a[6], a[8]
        e = n * h * w * c
        return 0.0, e / 4 * (4 if dy_f32 else 2) + e * (4 if dx_f32 else 2) + (2 * e if mask is not None else 0)
    return 0.0, 0.0


def main():
    assert torch.cuda.is_available(), "bench_resnet.py measures the GPU: no CPU fallback"
    torch.backends.cudnn.benchmark = True
    say(device_line())
    tflops_peak, gbs_peak = peaks()
    name = "RN101"
    sd = models.random_clip_resnet_state_dict(name, seed=1)
    tower = models.ModifiedResNetB200(name, sd, "cuda")
    from oracle.clip_resnet import OracleCLIPResNet

    stock = OracleCLIPResNet(name, sd).to(device="cuda", dtype=torch.bfloat16).to(memory_format=torch.channels_last)
    g = torch.Generator().manual_seed(0)
    for n in (16, 64):
        patches = torch.zeros(n, 224 * 224, 8)
        patches[..., :3] = torch.randn(n, 224 * 224, 3, generator=g)
        patches = patches.bfloat16().cuda()
        demb = torch.randn(n, 512, generator=g).cuda()

        def ours():
            tower.forward_patches(patches)
            tower.backward_patches(demb)

        us = timeit(ours)
        img = patches[..., :3].float().view(n, 224, 224, 3).permute(0, 3, 1, 2).bfloat16().contiguous(memory_format=torch.channels_last)

        def ref():
            x = img.detach().requires_grad_()
            e = stock.encode_image(x)
            torch.autograd.grad(e, x, demb.bfloat16())

        us_ref = timeit(ref)
        fl = tower.flops_fwd_bwd(n)
        say("RN101 forward + input gradient  N = %2d   ours %9.1f us (%6.1f TFLOP/s algorithmic)   stock PyTorch bf16 cuDNN %9.1f us   "
            "stock / ours %.2fx" % (n, us, fl / us / 1e6, us_ref, us_ref / us))
    # per-family time of one eager pass at N = 64 (per-call events: includes each call's launch gap)
    _lib.PROFILE, _lib.PROFILE_NAMES = [], tuple(FAMILY)
    tower.forward_patches(patches)
    tower.backward_patches(demb)
    torch.cuda.synchronize()
    prof, _lib.PROFILE = _lib.PROFILE, None
    fam = {}
    for nm, args, e0, e1 in prof:
        f = fam.setdefault(FAMILY[nm], [0.0, 0.0, 0.0, 0])
        fl, by = work(nm, args)
        f[0] += e0.elapsed_time(e1) * 1e3
        f[1] += fl
        f[2] += by
        f[3] += 1
    total = sum(f[0] for f in fam.values())
    say("per family, one eager pass at N = 64 (sum of per-call CUDA-event times %.1f us; peaks %.1f TFLOP/s bf16, %.0f GB/s HBM, "
        "sustained, measured on the B200):" % (total, tflops_peak, gbs_peak))
    for k, (us, fl, by, calls) in sorted(fam.items(), key=lambda kv: -kv[1][0]):
        rate = ""
        if fl:
            rate = "%7.1f TFLOP/s  %5.1f %% of peak" % (fl / us / 1e6, 100 * fl / us / 1e6 / tflops_peak)
        elif by:
            rate = "%7.0f GB/s     %5.1f %% of peak" % (by / us / 1e3, 100 * by / us / 1e3 / gbs_peak)
        say("  %-10s %4d calls %10.1f us  %5.1f %% of the pass   %s" % (k, calls, us, 100 * us / total, rate))
    del tower, stock
    torch.cuda.empty_cache()
    step_lines()
    say(device_line())
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as f:
        f.write("\n".join(LINES) + "\n")


def step_lines():
    """One guided DDIM step at 512x512 (fp16 NHWC UNet, Config's cut schedule at diffusion step 500), four towers vs the three ViTs."""
    from clip_diffusion_b200.config import Config
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.sample import GuidanceStep
    from clip_diffusion_b200.unet import create_unet

    unet = create_unet(512, seed=2, device="cuda", use_fp16=True, channels_last=True)
    diffusion = SpacedDiffusion(steps=250)
    all_models = models.load_clip_models(Config.chosen_clip_models, allow_random_init=True)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 3, 512, 512, generator=g).cuda()
    for names in (Config.chosen_clip_models, tuple(n for n in Config.chosen_clip_models if n != "RN101")):
        clip = {k: all_models[k] for k in names}
        text = {k: {"embeddings": torch.randn(1, m.visual.output_dim, generator=g).cuda(), "weights": torch.tensor(1.0, device="cuda")}
                for k, m in clip.items()}
        step = GuidanceStep(diffusion, unet, clip, text, config=Config)
        ms = timeit(lambda: step.ddim_step(x, 125), iters=5, warmup=2) / 1e3
        say("guided DDIM step 512x512, towers %s, %d cutouts per tower and batch x %d batches: %.1f ms/step"
            % ("+".join(names), Config.num_overview_cuts_schedule[500] + Config.num_inner_cuts_schedule[500], Config.num_cutout_batches, ms))


if __name__ == "__main__":
    main()
