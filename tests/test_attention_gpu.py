"""GPU tests of the attention kernels beyond single-shape parity (test_vit_gpu.py::test_attention_fwd_bwd and
test_text_gpu.py::test_causal_attention_fwd hold those): the lazy rescale of the tcgen05 forward in a child process first, the
forward -> backward chain, and bit-exact invariance of every image's results under the order of the batch and under repetition (the
persistent kernels carry warpgroup references, buffer parities and per-item constants from one item to the next)."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import attention as A

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_lazy_rescale_forward_in_subprocess():
    """staircase_up makes every warpgroup move its reference maximum on every block after its first, so the rescale of the O
    accumulator in TMEM (and its wait on the previous block's P V MMAs) runs in both instantiations of the tcgen05 forward.  Run it
    once in a child process with a timeout before the in-process tests, so that a hang or a fault there is reported, not inherited."""
    code = r'''
import sys, torch
sys.path.insert(0, %r)
from oracle import attention as A
for causal, n, T, heads in [(False, 2, 200, 2), (False, 2, 257, 2), (True, 2, 200, 2), (True, 2, 257, 2)]:
    qkv, _ = A.staircase_up(n, T, heads, 1, causal=causal)
    qkv = qkv.cuda()
    ref = A.attention_fwd(*A.split_qkv(qkv, n, T, heads), causal=causal)
    ctx, lse = A.attention_fwd_guarded(qkv, n, T, heads, causal=causal)
    r = A.worst_ratios({"o": A.rows_to_heads(ctx, n, T, heads), "lse": lse}, ref, A.fwd_bounds(ref))
    print("RESCALE causal=%%d T=%%d o=%%.3g lse=%%.3g" %% (causal, T, r["o"], r["lse"]), flush=True)
    assert max(r.values()) <= 1.0, r
torch.cuda.synchronize()
print("DONE")
''' % ROOT
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0 and "DONE" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


@pytest.mark.parametrize("n,T,heads,regime", [(2, 197, 4, "sharp"), (2, 257, 4, "staircase_up"), (3, 200, 1, "sink_query"),
                                              (3, 256, 16, "neighbour"), (2, 577, 4, "sharp")])
def test_attention_forward_then_backward(n, T, heads, regime, record_property):
    """The backward fed with the kernel forward's own bf16 ctx and fp32 lse (the reference takes the same tensors)."""
    qkv, dctx = A.make_inputs(regime, n, T, heads, 7 * T + heads)
    worst = A.check_attention(n, T, heads, qkv, dctx, chained=True)
    record_property("err_over_bound", {"kernel": "chained", "regime": regime, **worst})
    assert max(worst.values()) <= 1.0, worst


@pytest.mark.parametrize("causal,T,heads,n", [(False, 197, 4, 76), (False, 257, 4, 76), (True, 200, 4, 76)])
def test_attention_batch_order_and_repeat_invariance(causal, T, heads, n, record_property):
    """A batch of n * heads > 2 x 148 items (several per CTA of the persistent kernels) alternating huge_pos and flat images, then the same
    images rolled by 1 and by 37, and the first batch again: every image's ctx, lse (and dqkv) must be bit-identical each time, and
    the first run within the error model."""
    D = heads * 64
    assert n * heads > 2 * 148
    regimes = ["huge_pos" if i % 2 == 0 else "flat" for i in range(n)]
    qkv, dctx = A.mixed(regimes, T, heads, 3, causal=causal)
    qkv, dctx = qkv.cuda(), dctx.cuda()

    def run(qkv, dctx):
        ctx, lse = A.attention_fwd_guarded(qkv, n, T, heads, causal=causal)
        if causal:
            return ctx, lse, None
        return ctx, lse, A.attention_bwd_guarded(qkv, ctx, dctx, lse, n, T, heads)

    base = run(qkv, dctx)
    if causal:
        ref = A.attention_fwd(*A.split_qkv(qkv, n, T, heads), causal=True)
        worst = A.worst_ratios({"o": A.rows_to_heads(base[0], n, T, heads), "lse": base[1]}, ref, A.fwd_bounds(ref))
        del ref
    else:
        worst = A.check_attention(n, T, heads, qkv, dctx, chained=True)
    record_property("err_over_bound", {"kernel": "persistent" + (" causal" if causal else ""), "regime": "huge_pos|flat", **worst})
    assert max(worst.values()) <= 1.0, worst
    again = run(qkv, dctx)
    for a, b in zip(base, again):
        assert a is None or torch.equal(a, b), "a second run of the same batch differs"
    for shift in (1, 37):
        rolled = run(qkv.view(n, T, 3 * D).roll(shift, 0).reshape(n * T, 3 * D), dctx.view(n, T, D).roll(shift, 0).reshape(n * T, D))
        for name, a, b in zip(("ctx", "lse", "dqkv"), base, rolled):
            if a is None:
                continue
            want = (a.view(n, heads, T) if name == "lse" else a.view(n, T, -1)).roll(shift, 0)
            got = b.view(n, heads, T) if name == "lse" else b.view(n, T, -1)
            assert torch.equal(want, got), "%s of an image depends on its place in the batch (roll %d)" % (name, shift)
