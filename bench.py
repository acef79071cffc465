#!/usr/bin/env python
"""Guidance-step benchmark (contract in the task statement; numbers explained in DESIGN.md section "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|target|c3|c1] [--dump-outputs DIR]

A "step" is ONE full CLIP-guided DDIM sampling step on synthetic inputs: the sampler's no-grad UNet forward, the
guidance function (UNet forward with grad -> fused cutouts -> CLIP ViT fwd -> spherical loss+grad -> ViT dgrad ->
cutout backward -> TV -> all-reduce -> UNet VJP -> RMS clamp) and the DDIM update.  Default workload = north_star's
Target: 512x512 uncond guided-diffusion UNet (fp16, random init) + ViT-L/14, 32 overview + 32 inner cutouts, DDIM-250
schedule (`--workload c2` = BASELINE.json configs[1]).  `value` is cutouts/s = steps/s x cutouts per step (steps/s is
reported beside it as `steps_per_s`).  For N > 1 the cutout batch of every step is sharded across ranks (one NCCL all-reduce
of the [3,512,512] fp32 image gradient per step, UNet replicated); --scaling strong (default, configs[2] / north_star (4))
splits the workload's 64 cutouts over the ranks -- the SAME job on more GPUs; --scaling weak keeps the workload's cutouts PER
RANK (N x cutouts per step).  The strong-scaling line also carries the weak number as the secondary field `weak`.

--impl reference times the CPU restatement of the reference path (oracle/, fp32, all host threads) on the same
workload; see cpu_baseline in the JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (image size, clip models, overview cuts, inner cuts, cutout batches, ddim steps, description)
    "c1": (256, ("ViT-B/32",), 12, 4, 1, 250, "256x256 UNet(256 cfg) + ViT-B/32, 12+4 cutouts"),
    "c2": (512, ("ViT-B/16",), 16, 16, 1, 250, "512x512 uncond guided-diffusion UNet + ViT-B/16, 16 overview + 16 inner cutouts, DDIM-250"),
    "c3": (512, ("ViT-B/32", "ViT-B/16", "ViT-L/14"), 32, 32, 1, 250, "512x512 UNet + ViT-B/32+B/16+L/14 ensemble, 64 cutouts per model, tv+range"),
    "target": (512, ("ViT-L/14",), 32, 32, 1, 250, "512x512 UNet + ViT-L/14, 64 cutouts (north_star target)"),
    "c4": (512, ("ViT-B/32", "ViT-B/16", "ViT-L/14"), 8, 8, 1, 250, "512x512 UNet + B/32+B/16+L/14 with aesthetic-predictor loss (aesthetic_scale 500) and a synthetic init image "
           "(MS-SSIM dissimilarity term, MS_SSIM_scale 1000; the LPIPS VGG network is un-vendored and left out), 16 cutouts per model"),
    "c5": (768, ("ViT-L/14@336px",), 64, 64, 1, 250, "768x768 UNet + ViT-L/14@336px, 128 cutouts (cutout-scaling sweep, smallest point)"),
    "c5-512": (768, ("ViT-L/14@336px",), 256, 256, 1, 250, "768x768 UNet + ViT-L/14@336px, 512 cutouts (cutout-scaling sweep, largest point; shard over 8 GPUs)"),
    "clip-only": (512, ("ViT-L/14",), 32, 32, 1, 250, "ViT-L/14, 64 cutouts, guidance gradient only (no UNet)"),
}


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=8)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="target", choices=sorted(WORKLOADS))
    p.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                   help="N>1: strong (default) = the workload's cutouts are split over the ranks (same job, more GPUs); "
                        "weak = every rank keeps the workload's cutouts (N x cutouts per step)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-graphs", action="store_true", help="do not capture the replicated UNet forward/backward into CUDA graphs")
    p.add_argument("--two-forwards", action="store_true", help="evaluate the UNet separately for the sampler and for cond_fn like the reference does")
    p.add_argument("--unet-layout", default="nhwc", choices=["nhwc", "nchw"],
                   help="nhwc (default): channels_last trunk + fused GroupNorm/scale-shift/SiLU kernels (csrc/unet_norm.cu); nchw: stock torch ops")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what the last timed step returned (sample, pred_xstart) to DIR/<name>.npy as float32; "
                        "the inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def dump_outputs(directory, arrays):
    """DIR/<name>.npy, float32, for every tensor of ``arrays`` (each one is [1, 3, size, size]: at most 7 MB per array)."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


class Cfg:
    """Config of the benchmarked step (read at call time by the guidance function, like clip_diffusion.config.Config)."""
    grad_threshold = 0.05
    clip_guidance_scale = 8000
    denoise_scale = 10000
    aesthetic_scale = 0


def make_cfg(n_over, n_inner, batches):
    class C(Cfg):
        num_cutout_batches = batches
        num_overview_cuts_schedule = (n_over,) * 1000
        num_inner_cuts_schedule = (n_inner,) * 1000
        inner_cut_size_power_schedule = (5,) * 1000
        cut_gray_portion_schedule = (0.3,) * 1000
    return C


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:  # reap it: the benchmark must not leave nvidia-smi behind
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
                self.proc.wait()
            self.proc = None

    def summary(self, t0, t1, t_end=None):
        self.stop()
        rows = ([r for ts, r in self.rows if t0 <= ts <= t1 and len(r) >= 7] or [r for ts, r in self.rows if t0 <= ts <= (t_end or t1) and len(r) >= 7]
                or [r for _, r in self.rows[-3:] if len(r) >= 7])
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in rows)
        reasons = [n for i, n in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap"))
                   if any(r[i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons, "samples": len(rows)}


def unet_norm_roofline(dev, hbm_peak):
    """Second roofline object: the HBM-bound op that dominates the replicated UNet's non-conv time (csrc/unet_norm.cu), timed live with
    CUDA events on the launching stream at the level-0 shape of the 512x512 UNet, L2 flushed (512 MB memset) between iterations.
    Algorithmic bytes: forward reads x twice and writes y (3 passes), backward reads (dy, x) twice and writes dx (5 passes)."""
    from clip_diffusion_b200.unet_ops import group_norm_nhwc

    shape = (1, 128, 512, 512)
    x = torch.randn(shape, device=dev).half().contiguous(memory_format=torch.channels_last).requires_grad_()
    gamma, beta = torch.ones(shape[1], device=dev), torch.zeros(shape[1], device=dev)
    ss = torch.zeros(1, 2 * shape[1], device=dev)
    dy = torch.randn(shape, device=dev).half().contiguous(memory_format=torch.channels_last)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    nb = x.numel() * 2
    ts = []
    for it in range(8):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        y = group_norm_nhwc(x, gamma, beta, 32, 1e-5, scale_shift=ss, silu=True)
        torch.autograd.grad(y, x, dy)
        e1.record()
        torch.cuda.synchronize()
        if it >= 3:
            ts.append(e0.elapsed_time(e1))
    ms = sorted(ts)[len(ts) // 2]
    achieved = 8 * nb / (ms / 1e3) / 1e9
    return {"bound": "hbm", "kernel": "cg_groupnorm_nhwc_fwd + _bwd (GroupNorm32+scale-shift+SiLU, 3 + 3 kernels) on [1,512,512,128] fp16 NHWC",
            "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "algorithmic_bytes": 8 * nb, "ms": ms,
            "note": "op-level (includes the two tiny finalize kernels and host launch gaps); per-kernel numbers in profiles/r01_unet_kernel_rooflines.txt"}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def scaled_cuts(wl, world, scaling):
    """(overview, inner) cutouts of one (model, batch): the workload's counts, times the world size under weak scaling."""
    n_over, n_inner = WORKLOADS[wl][2], WORKLOADS[wl][3]
    mult = world if (scaling == "weak" and world > 1) else 1
    return n_over * mult, n_inner * mult


METRIC = "CLIP-guided cutouts/s fwd+bwd inside full guidance steps (= steps/s x cutouts per step) @%dx%d"


def build_cpu_reference(wl, seed=0, world=1, scaling="weak"):
    """The CPU restatement of the reference path (oracle/): same workload, fp32, torch CPU ops."""
    from clip_diffusion_b200.diffusion import SpacedDiffusion  # sampler host logic (numpy + torch ops), not a kernel
    from clip_diffusion_b200.models import random_clip_state_dict
    from clip_diffusion_b200.rng_record import draw_cutout_record
    from clip_diffusion_b200.unet import create_unet
    from oracle.clip_vit import OracleCLIP
    from oracle.cond_fn import make_conditon_function

    size, names, _, _, batches, ddim, _ = WORKLOADS[wl]
    n_over, n_inner = scaled_cuts(wl, world, scaling)
    cfg = make_cfg(n_over, n_inner, batches)
    unet = create_unet(size if size in (256, 512) else 512, seed=2, device="cpu", use_fp16=False)
    diffusion = SpacedDiffusion(steps=ddim)
    g = torch.Generator().manual_seed(seed)
    clip, text = {}, {}
    for i, name in enumerate(names):
        clip[name] = OracleCLIP(name, state_dict=random_clip_state_dict(name, seed=1 + i))
        text[name] = {"embeddings": torch.randn(1, clip[name].visual.output_dim, generator=g), "weights": torch.tensor(1.0)}
    state = {"ct": ddim - 1}

    def record_source(name, b, H, W, cs, no, ni, p, gp):
        return draw_cutout_record(H, W, cs, no, ni, p, gp, noise="cpu")

    cond_fn = make_conditon_function(diffusion, unet, clip, text, lambda: state["ct"], cfg, record_source)
    x = torch.randn(1, 3, size, size, generator=g)

    def denoised_fn(x_start):  # sample.py:116-132
        thr = torch.quantile(x_start.reshape(x_start.shape[0], -1).abs(), 0.995, dim=-1).clamp(min=1.0).view(-1, 1, 1, 1)
        return x_start.clamp(min=-thr, max=thr) / thr

    def step(x, i):
        state["ct"] = i
        t = torch.full((1,), i, dtype=torch.long)
        return diffusion.ddim_sample(unet, x, t, clip_denoised=False, denoised_fn=denoised_fn, cond_fn=cond_fn, model_kwargs={}, eta=0.8)

    return step, x, ddim, (n_over + n_inner) * batches * len(names)


def workload_config(wl, world, scaling):
    """The `config` object of the JSON line: the WORKLOAD only, identical in both arms (b200 and --impl reference); everything
    about how this implementation runs it goes to `impl_details`."""
    size, names, _, _, batches, ddim, desc = WORKLOADS[wl]
    n_over, n_inner = scaled_cuts(wl, world, scaling)
    return {"workload": desc, "image": "%dx%d" % (size, size), "clip_models": list(names), "overview_cuts": n_over, "inner_cuts": n_inner,
            "cutout_batches": batches, "cutouts_per_step": (n_over + n_inner) * batches * len(names), "ddim_steps": ddim, "eta": 0.8,
            "dynamic_thresholding": 0.995, "n_gpus": world, "scaling": scaling if world > 1 else "n/a (1 GPU)"}


def run_reference(args, rank):
    if rank != 0:
        return
    wl = args.workload
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(1234)
    step, x, ddim, cuts = build_cpu_reference(wl, world=args.gpus, scaling=args.scaling)
    i = ddim - 1
    x = step(x, i)["sample"]  # warm-up
    k = args.steps
    t0 = time.time()
    for j in range(k):
        i = i - 1 if i > 0 else ddim - 1
        out = step(x, i)
        x = out["sample"]
    dt = (time.time() - t0) / k
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sample": out["sample"], "pred_xstart": out["pred_xstart"]})
    val = 1.0 / dt
    sample = "%d full guidance step(s) after 1 warm-up step" % k
    line = {
        "impl": "reference", "metric": METRIC % (WORKLOADS[wl][0], WORKLOADS[wl][0]), "value": cuts * val, "unit": "cutouts/s", "n_gpus": args.gpus, "steps": k,
        "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl, args.gpus, args.scaling),
        "cpu_baseline": {"value": cuts * val, "unit": "cutouts/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": cuts * val, "unit": "cutouts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "steps_per_s": val,
    }
    print(json.dumps(line), flush=True)


PROFILED = ("cg_gemm_bf16_tn", "cg_attention_fwd", "cg_attention_bwd", "cg_cutouts_fwd", "cg_cutouts_bwd", "cg_layernorm_fwd", "cg_layernorm_bwd",
            "cg_tv_loss_fwd_bwd", "cg_range_loss_fwd_bwd", "cg_image_losses_fwd_bwd", "cg_spherical_loss_fwd_bwd")


def kernel_rooflines(prof, step_ms, tf_peak, hbm_peak, peak_src, traffic):
    """Per-kernel-family rooflines from the profiled pass: algorithmic work (SURVEY section 8(d)) of every launch of the timed
    region / sum of their CUDA-event durations on the launching stream."""
    fam = {}

    def add(key, work, ms):
        f = fam.setdefault(key, [0.0, 0.0, 0])
        f[0] += work
        f[1] += ms
        f[2] += 1

    for name, a, e0, e1 in prof:
        ms = e0.elapsed_time(e1)
        if name == "cg_gemm_bf16_tn":
            add("gemm", 2.0 * a[2] * a[3] * a[4], ms)
        elif name == "cg_attention_fwd":  # (qkv, Nimg, T, heads, ...): QK^T + PV
            add("attn_fwd", 4.0 * a[1] * a[3] * a[2] * a[2] * 64, ms)
        elif name == "cg_attention_bwd":  # (qkv, ctx, dctx, lse, Nimg, T, heads, ...): dV, dP, dQ, dK (recomputing S is not counted)
            add("attn_bwd", 8.0 * a[4] * a[6] * a[5] * a[5] * 64, ms)
        elif name == "cg_cutouts_fwd":    # (x, H, W, cuts, n, cs, aug, noise, out, fmt, patch, kpad, ws): read the image once, write bf16 patches
            g2 = (a[5] // a[10]) ** 2 if a[10] else 0
            add("cutouts_fwd", 12.0 * a[1] * a[2] + (a[4] * g2 * a[11] * 2.0 if a[10] else a[4] * 3.0 * a[5] * a[5] * 4), ms)
        elif name == "cg_cutouts_bwd":    # (dout, H, W, n, cs, fmt, patch, kpad, ...): read fp32 patch gradients, write the image gradient
            g2 = (a[4] // a[6]) ** 2 if a[6] else 0
            add("cutouts_bwd", 12.0 * a[1] * a[2] + (a[3] * g2 * a[7] * 4.0 if a[6] else a[3] * 3.0 * a[4] * a[4] * 4), ms)
        elif name == "cg_layernorm_fwd":  # (x, g, b, M, D, ...): fp32 in, bf16 out
            add("layernorm_fwd", 6.0 * a[3] * a[4], ms)
        elif name == "cg_layernorm_bwd":  # reads dy, x, dx (fp32), writes dx (fp32) + bf16 copy
            add("layernorm_bwd", 18.0 * a[5] * a[6], ms)
        elif name in ("cg_tv_loss_fwd_bwd", "cg_range_loss_fwd_bwd", "cg_image_losses_fwd_bwd"):  # (x, B, C, H, W, ...): read + write the image
            add("image_losses", 8.0 * a[1] * a[2] * a[3] * a[4], ms)
    out = {}
    steps_in_prof = max(1, sum(1 for n, *_ in prof if n in ("cg_tv_loss_fwd_bwd", "cg_image_losses_fwd_bwd")))
    for key, (work, ms, cnt) in fam.items():
        if ms <= 0:
            continue
        tensor = key in ("gemm", "attn_fwd", "attn_bwd")
        achieved = work / (ms / 1e3) / (1e12 if tensor else 1e9)
        peak = tf_peak if tensor else hbm_peak
        out[key] = {"bound": "tensor" if tensor else "hbm", "achieved": achieved, "peak": peak, "unit": "TFLOP/s" if tensor else "GB/s",
                    "frac": achieved / peak, "launches": cnt, "ms_per_step": ms / steps_in_prof,
                    "share_of_step": (ms / steps_in_prof) / step_ms if step_ms > 0 else None,
                    ("algorithmic_flops_per_launch" if tensor else "algorithmic_bytes_per_launch"): work / cnt}
    g = out.get("gemm", {"achieved": 0.0, "frac": 0.0, "launches": 0, "share_of_step": None})
    roof = {"bound": "tensor", "kernel": "gemm_bf16_tn_kernel (tcgen05/TMEM/TMA, all ViT GEMMs)", "achieved": g["achieved"], "peak": tf_peak, "unit": "TFLOP/s",
            "frac": g["frac"], "traffic": traffic, "algorithmic_flops_per_launch": g.get("algorithmic_flops_per_launch"), "peak_source": peak_src,
            "launches": g["launches"], "share_of_step": g["share_of_step"]}
    return roof, out


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist

    from clip_diffusion_b200 import _lib
    from clip_diffusion_b200.diffusion import SpacedDiffusion
    from clip_diffusion_b200.models import load_clip_models
    from clip_diffusion_b200.sample import GuidanceStep, make_denoised_function
    from clip_diffusion_b200.unet import create_unet, graph_unet
    from clip_diffusion_b200.utils.functional import set_seed

    # (the image exports NCCL_DEBUG=VERSION: NCCL prints its one-line version banner on rank 0's stdout before the JSON line; it is
    # left alone -- the JSON line is always the LAST line of stdout)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    torch.backends.cudnn.benchmark = os.environ.get("CG_CUDNN_BENCHMARK", "1") == "1"  # let cuDNN pick conv algorithms for the static UNet shapes
    _lib.check(_lib.load().cg_check_device(), "cg_check_device")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    size, names, _, _, batches, ddim, desc = WORKLOADS[args.workload]
    set_seed(1234)
    clip_only = args.workload == "clip-only"
    unet = None if clip_only else create_unet(size if size in (256, 512) else 512, seed=2, device=dev, use_fp16=True, channels_last=args.unet_layout == "nhwc")
    diffusion = SpacedDiffusion(steps=ddim)
    unet_graphed = False
    if unet is not None and not args.no_graphs and not args.two_forwards:
        # The replicated UNet is ~7k tiny stock-PyTorch launches per step and the step was launch-bound on the host
        # (profiles/r01_*): capture its forward and backward once into CUDA graphs (static shapes, batch 1).
        unet = graph_unet(unet, size, size, dev)
        unet_graphed = True
    clip_models = load_clip_models(names, dev, allow_random_init=True)
    g = torch.Generator().manual_seed(0)
    text = {n: {"embeddings": torch.randn(1, m.visual.output_dim, generator=g).to(dev), "weights": torch.tensor(1.0, device=dev)} for n, m in clip_models.items()}
    predictors = None
    if args.workload == "c4":
        from clip_diffusion_b200.models import load_aesthetic_predictors

        predictors = load_aesthetic_predictors(names, dev)
    denoised_fn = make_denoised_function(0.995)  # reference defaults: dynamic thresholding 0.995, eta 0.8 (sample.py:66-71)
    x_host = torch.randn(1, 3, size, size, generator=g).pin_memory()
    out_host = torch.empty(2, 3, size, size).pin_memory()
    x_dev = x_host.to(dev)
    x_in_fixed = torch.tanh(x_dev).contiguous()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def tmax(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def next_i(i):  # walk the DDIM schedule downwards, wrapping so that any --steps/--warmup works
        return i - 1 if i > 0 else ddim - 1

    W, K = max(args.warmup, 3), args.steps

    def measure(scaling, profile):
        """W warm-up steps, then K timed steps with the state resident in HBM, K timed steps end to end through pinned host
        buffers and (profile=True) K more steps with CUDA events around every C-ABI call for the kernel rooflines."""
        n_over, n_inner = scaled_cuts(args.workload, world, scaling)
        cfg = make_cfg(n_over, n_inner, batches)
        init_image = None
        if args.workload == "c4":
            cfg.aesthetic_scale = 500
            cfg.MS_SSIM_scale, cfg.LPIPS_scale = 1000.0, 0.0
            init_image = torch.tanh(torch.randn(1, 3, size, size, generator=torch.Generator().manual_seed(9))).to(dev)
        guidance = GuidanceStep(diffusion, unet, clip_models, text, aesthetic_predictors=predictors, config=cfg, rank=rank, world_size=world,
                                range_scale=150.0 if args.workload == "c3" else 0.0, init_image_tensor=init_image)

        def step(x, i):
            if clip_only:
                gbuf = torch.zeros(3, size, size, device=dev)
                guidance.clip_guidance_grad(x_in_fixed, 1000 - (int(diffusion.timestep_map[i]) + 1), gbuf)
                if world > 1:
                    dist.all_reduce(gbuf)
                return {"sample": x, "pred_xstart": gbuf.unsqueeze(0)}
            return guidance.ddim_step(x, i, eta=0.8, denoised_fn=denoised_fn, reuse_forward=not args.two_forwards)

        i = ddim - 1
        x = x_dev
        # nvidia-smi needs ~0.5 s before its first sample: start it before the warm-up so that it is streaming during the timed regions
        clocks = ClockSampler(local_rank) if (rank == 0 and profile) else None
        for _ in range(W):
            x = step(x, i)["sample"]
            i = next_i(i)
        res = {"cuts_per_step": (n_over + n_inner) * batches * len(names), "n_over": n_over, "n_inner": n_inner}
        # ---- timed region 1: inputs resident in HBM -------------------------------------------------
        barrier()
        k0 = _lib.kernel_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        use_range = profile and os.environ.get("CG_BENCH_PROFILER_RANGE") == "1"  # ncu --profile-from-start off: profile the timed region only
        if use_range:
            torch.cuda.profiler.start()
        wall0 = time.time()
        e0.record()
        for _ in range(K):
            last = step(x, i)
            x = last["sample"]
            i = next_i(i)
        e1.record()
        res["host_enqueue_ms"] = (time.time() - wall0) * 1e3 / K  # host time to ISSUE a step (the GPU runs behind it): the floor of the e2e step
        barrier()
        if use_range:
            torch.cuda.profiler.stop()
        wall1 = time.time()
        res["ms"] = tmax(e0.elapsed_time(e1))
        res["launches"] = _lib.kernel_launches - k0
        if unet_graphed:  # our GroupNorm / resample / concat kernels replayed inside the UNet's CUDA graphs (one forward + one backward per step)
            res["launches"] += K * unet.own_kernels_per_replay
        if profile and rank == 0 and args.dump_outputs:  # the last timed step's result, copied outside the timed region
            res["outputs"] = {"sample": last["sample"].float().cpu(), "pred_xstart": last["pred_xstart"].float().cpu()}
        if not profile:
            return res
        if clocks is not None and os.environ.get("CG_BENCH_CLOCKS_ALL_REGIONS") != "1":
            clocks.stop()  # nvidia-smi polling takes driver locks: harmless while launches are queued ahead, visible in the synchronised region below
        # ---- timed region 2: end to end through host buffers ------------------------------------------
        barrier()
        e0.record()
        for _ in range(K):
            xd = x_host.to(dev, non_blocking=True)
            out = step(xd, i)
            out_host[0].copy_(out["sample"][0], non_blocking=True)
            out_host[1].copy_(out["pred_xstart"][0].float(), non_blocking=True)
            torch.cuda.current_stream().synchronize()  # the caller consumes the step result (PNG every step, sample.py:290-295)
            i = next_i(i)
        e1.record()
        barrier()
        res["ms_e2e"] = tmax(e0.elapsed_time(e1))
        # ---- timed region 3: the same K steps with CUDA events around every C-ABI call (kernel rooflines; not part of `value`) ----
        barrier()
        _lib.PROFILE, _lib.PROFILE_NAMES = [], PROFILED
        e0.record()
        for _ in range(K):
            x = step(x, i)["sample"]
            i = next_i(i)
        e1.record()
        barrier()
        res["prof"], _lib.PROFILE = _lib.PROFILE, None
        res["ms_prof"] = e0.elapsed_time(e1)
        # samples inside timed region 1; if the region was shorter than the sampling period, the samples of the three timed regions (all under load)
        res["clocks"] = clocks.summary(wall0, wall1, time.time()) if clocks else None
        return res

    main_res = measure(args.scaling, profile=True)
    weak_res = measure("weak", profile=False) if (world > 1 and args.scaling == "strong") else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, main_res["outputs"])
    ms, ms_e2e, cuts_per_step = main_res["ms"], main_res["ms_e2e"], main_res["cuts_per_step"]
    tf_peak, hbm_peak, peak_src = measured_peaks()
    traffic = None  # dram bytes per GEMM launch from the committed ncu capture of this same command (profiles/)
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic_%s.json" % args.workload)
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get("avg_dram_bytes_per_launch")
    value = K / (ms / 1e3)
    e2e = K / (ms_e2e / 1e3)
    roof, fams = kernel_rooflines(main_res["prof"], main_res["ms_prof"] / K, tf_peak, hbm_peak, peak_src, traffic)
    n_cut = main_res["n_over"] + main_res["n_inner"]
    line = {
        "metric": METRIC % (size, size), "value": cuts_per_step * value, "unit": "cutouts/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(args.workload, world, args.scaling),
        "impl_details": {"unet_cuda_graphs": unet_graphed, "unet": "fp16, replicated, %s; %s" % ("channels_last cuDNN convs + fused NHWC GroupNorm/scale-shift/SiLU kernels" if args.unet_layout == "nhwc" else "NCHW stock PyTorch", "two forwards per step (sampler + cond_fn) like the reference" if args.two_forwards else "one grad-enabled forward shared by sampler and cond_fn (identical results)"),
                         "clip": "bf16 operands / fp32 accumulate + fp32 residual stream, random init",
                         "parallelism": "%d cutouts per (model, step) sharded over %d rank(s) = %d per rank, 1 all-reduce of the image gradient per step" % (n_cut, world, -(-n_cut // world)),
                         "cutouts_per_rank": -(-cuts_per_step // world),
                         "l2": "working set (1.1 GB UNet + ViT weights + activations) far exceeds the 126 MB L2; no flush"},
        "steps_per_s": value,
        "e2e": {"value": cuts_per_step * e2e, "unit": "cutouts/s", "steps_per_s": e2e, "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4},
        "gpu_launches": main_res["launches"],
        "host_enqueue_ms_per_step": main_res.get("host_enqueue_ms"),
        "clocks": main_res["clocks"],
        "roofline": roof,
    }
    for key, label in (("attn_fwd", "roofline_attention_fwd"), ("attn_bwd", "roofline_attention_bwd"), ("cutouts_fwd", "roofline_cutouts_fwd"),
                       ("cutouts_bwd", "roofline_cutouts_bwd"), ("layernorm_fwd", "roofline_layernorm_fwd"), ("layernorm_bwd", "roofline_layernorm_bwd"),
                       ("image_losses", "roofline_image_losses")):
        if key in fams:
            line[label] = fams[key]
    if weak_res is not None:
        wv = K / (weak_res["ms"] / 1e3)
        line["weak"] = {"value": weak_res["cuts_per_step"] * wv, "unit": "cutouts/s", "steps_per_s": wv, "ms_per_step": weak_res["ms"] / K,
                        "cutouts_per_step": weak_res["cuts_per_step"], "note": "secondary: every rank keeps the workload's cutouts (N x cutouts per step)"}
    if unet is not None and args.unet_layout == "nhwc":
        line["roofline_unet_norm"] = unet_norm_roofline(dev, hbm_peak)
    if world == 1 and not args.no_cpu_baseline and not clip_only:
        torch.set_num_threads(os.cpu_count() or 1)
        cstep, cx, cddim, ccuts = build_cpu_reference(args.workload)
        t0 = time.time()
        cstep(cx, cddim - 1)
        dt = time.time() - t0
        line["cpu_baseline"] = {"value": ccuts / dt, "unit": "cutouts/s", "steps_per_s": 1.0 / dt, "cores": torch.get_num_threads(), "kind": "port",
                                "sample": "1 full guidance step of the same workload, fp32, no warm-up (%.1f s)" % dt}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
