"""Timings of the CLIP text tower (CLIPModelB200.encode_text) on the sm_100a kernels, with CUDA events after warm-up:
  * encode_text for N = 1, 16 and 397 prompts (397: the reference's precomputed style list) on the 512- and 768-wide towers;
  * the causal attention kernel alone at N = 397 (both head counts);
  * the same prompts through the fp32 oracle (oracle/clip_text.py) moved to the GPU in bf16: the stock-PyTorch baseline.
Random weights (seeded) and clip.tokenize-shaped random prompts; throughput does not depend on the values.  The GPU name, power limit
and max SM clock are printed in the same run.
Usage (GPU machine):  python tools/bench_text.py > profiles/<name>.txt"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from clip_diffusion_b200 import _lib, models
from oracle.clip_text import OracleCLIPText, random_prompt_tokens


def timeit(fn, iters=20, warmup=3):
    """median of `iters` single calls, each bracketed by CUDA events (the working set stays in L2: this is the once-per-job call)"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def device_line():
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "nvidia-smi unavailable"
    return "device: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(), q)


def text_flops(n, T, D, L):
    """2 x MAC of the transformer (QKV, out, MLP GEMMs + causal QK^T / PV counted in full)"""
    return n * L * (24 * T * D * D + 4 * T * T * D)


def main():
    assert torch.cuda.is_available(), "bench_text.py measures the GPU: no CPU fallback"
    print(device_line())
    g = torch.Generator().manual_seed(0)
    prompts = random_prompt_tokens(torch.randint(0, 40, (397,), generator=g).tolist(), 77, g)
    for name in ("ViT-B/32", "ViT-L/14"):
        context, vocab, D, L, heads, E = models.CLIP_TEXT_CONFIGS[name]
        m = models.CLIPModelB200(name, None, "cuda")
        sd = models.random_clip_text_state_dict(name, seed=1)
        oracle = OracleCLIPText(name, state_dict=sd).to(device="cuda", dtype=torch.bfloat16)
        m.encode_text(prompts[:1].cuda())  # builds the tower
        for n in (1, 16, 397):
            tok = prompts[:n].cuda()
            us = timeit(lambda: m.encode_text(tok))
            with torch.no_grad():
                us_ref = timeit(lambda: oracle.encode_text(tok))
            tf = text_flops(n, context, D, L) / us / 1e6
            print("%-10s width %4d  N = %3d   encode_text %9.1f us (%6.1f TFLOP/s)   stock PyTorch bf16 %9.1f us   ratio %.2fx"
                  % (name, D, n, us, tf, us_ref, us_ref / us))
        n = 397
        qkv = (torch.randn(n * context, 3 * D, generator=g) * 0.8).bfloat16().cuda()
        ctx = torch.empty(n * context, D, device="cuda", dtype=torch.bfloat16)
        lse = torch.empty(n, heads, context, device="cuda")
        us = timeit(lambda: _lib.call("cg_attention_causal_fwd", _lib.ptr(qkv), n, context, heads, _lib.ptr(ctx), _lib.ptr(lse)), iters=50)
        print("%-10s cg_attention_causal_fwd  N = %d  T = %d  heads = %2d   %8.1f us" % (name, n, context, heads, us))
        del m, oracle
        torch.cuda.empty_cache()
    print(device_line())


if __name__ == "__main__":
    main()
