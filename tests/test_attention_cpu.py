"""CPU tests of the attention oracle (oracle/attention.py): the float64 reference against autograd, every input regime's defining
property, and the error model: a float64 restatement of the tcgen05 forward's online softmax (bf16 P, lazy rescale of the reference
maximum, two warpgroups merged at the end) stays inside the bounds, and the same restatement with a dropped sink key or without the
rescale of its row sum or accumulator falls outside them."""
import pytest
import torch

from oracle import attention as A


def _rand(n, h, T, seed, std=1.0):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(n, h, T, 64, generator=g, dtype=torch.float64) * std for _ in range(4)]


@pytest.mark.parametrize("causal", [False, True])
def test_forward_matches_masked_softmax(causal):
    q, k, v, _ = _rand(2, 3, 70, 1)
    ref = A.attention_fwd(q, k, v, causal)
    s = (q @ k.transpose(-1, -2)) * 0.125
    if causal:
        s = s.masked_fill(torch.ones(70, 70, dtype=torch.bool).triu(1), float("-inf"))
    torch.testing.assert_close(ref["o"], torch.softmax(s, -1) @ v, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(ref["lse"], torch.logsumexp(s, -1), rtol=1e-12, atol=1e-12)
    assert (ref["pv_abs"] >= ref["o"].abs() - 1e-12).all()
    assert (ref["sabs"] >= s.abs().nan_to_num(0.0, 0.0, 0.0) - 1e-12).all()


def test_backward_matches_autograd():
    """With the unrounded forward output as ctx and the exact lse, attention_bwd is the gradient of sum(O * dO)."""
    q, k, v, dO = _rand(2, 2, 83, 2, std=1.5)
    q, k, v = [t.clone().requires_grad_() for t in (q, k, v)]
    o = torch.softmax((q @ k.transpose(-1, -2)) * 0.125, -1) @ v
    gq, gk, gv = torch.autograd.grad((o * dO).sum(), (q, k, v))
    fw = A.attention_fwd(q.detach(), k.detach(), v.detach())
    bw = A.attention_bwd(q.detach(), k.detach(), v.detach(), fw["o"], fw["lse"], dO)
    for name, want in (("dq", gq), ("dk", gk), ("dv", gv)):
        torch.testing.assert_close(bw[name], want, rtol=1e-10, atol=1e-12)
    # the magnitudes bound the values they stand for
    assert (bw["ptdo_abs"] >= bw["dv"].abs() - 1e-12).all()
    assert (0.125 * bw["shat_k"] >= bw["dq"].abs() - 1e-12).all() and (0.125 * bw["shat_q"] >= bw["dk"].abs() - 1e-12).all()


def test_backward_reads_the_given_ctx_and_lse():
    """delta comes from the ctx passed in (the kernel reads the bf16 one) and P from the lse passed in, not from a recomputation."""
    q, k, v, dO = _rand(1, 1, 40, 3)
    fw = A.attention_fwd(q, k, v)
    a = A.attention_bwd(q, k, v, fw["o"], fw["lse"], dO)
    b = A.attention_bwd(q, k, v, fw["o"].bfloat16(), fw["lse"], dO)
    c = A.attention_bwd(q, k, v, fw["o"], fw["lse"] + 0.1, dO)
    assert not torch.equal(a["dq"], b["dq"]) and torch.equal(a["dv"], b["dv"])
    torch.testing.assert_close(c["dv"], a["dv"] * torch.exp(torch.tensor(-0.1, dtype=torch.float64)), rtol=1e-12, atol=1e-14)


def _edge(T, causal=False):
    return int(not causal and T > 1 and (T - 1) % 64 == 0)


CASES = [(r, T, c) for r in A.REGIMES for T in (77, 129, 197, 257, 272, 577) for c in (False, True)
         if not (c and (T > 272 or r not in A.CAUSAL_AWARE + ("flat",)))]


@pytest.mark.parametrize("regime,T,causal", CASES)
def test_regime_inputs(regime, T, causal):
    """Every generator returns bf16 [n*T, 3D] / [n*T, D] and checks its own property (an AssertionError here is a broken regime)."""
    n, heads = 2, 3
    if regime == "sink":
        for pos in A.sink_positions(T, _edge(T, causal)):
            qkv, dO = A.make_inputs(regime, n, T, heads, 5, causal, pos=pos)
    else:
        qkv, dO = A.make_inputs(regime, n, T, heads, 5, causal)
    assert qkv.dtype == torch.bfloat16 and qkv.shape == (n * T, 3 * heads * 64)
    assert dO.dtype == torch.bfloat16 and dO.shape == (n * T, heads * 64)
    assert torch.isfinite(qkv.float()).all() and torch.isfinite(dO.float()).all()


def test_sink_positions_cover_block_edges_and_the_edge_key():
    assert A.sink_positions(257, 1) == [0, 63, 64, 255, 256]
    assert A.sink_positions(197, 0) == [0, 63, 64, 196]
    assert A.sink_positions(50, 0) == [0, 49]


def test_flat_inputs_are_the_original_test_inputs():
    g = torch.Generator().manual_seed(197 + 12)
    qkv = (torch.randn(2 * 197, 3 * 768, generator=g) * 0.8).bfloat16()
    dctx = (torch.randn(2 * 197, 768, generator=g) * 0.5).bfloat16()
    a, b = A.flat(2, 197, 12, 197 + 12)
    assert torch.equal(a, qkv) and torch.equal(b, dctx)


# ------------------------------------------------------------------------------------------ a restatement of the tcgen05 forward
def emulate_tc_forward(q, k, v, acc_rescale=True, lsum_rescale=True, drop_key=None):
    """Online softmax of attn_fwd_tc_kernel (non-causal, no edge token) in float64: 64-key blocks alternate between two warpgroups, each
    keeps a reference maximum that only moves when a block exceeds it by more than RESCALE_LOG2, P is rounded to bf16 for P V while the
    row sum takes the unrounded P, the partial results are merged at the end and O is rounded to bf16.  Returns O, lse and the number
    of (row, block) rescales."""
    T = k.shape[-2]
    s2 = A.logits(q, k) / A.LN2
    if drop_key is not None:
        s2[..., drop_key] = float("-inf")
    parts, rescales = [], 0
    for wg in (0, 1):
        mref = lsum = acc = None
        for b in range(wg, (T + 63) // 64, 2):
            blk, vb = s2[..., b * 64:(b + 1) * 64], v[..., b * 64:(b + 1) * 64, :]
            bm = blk.amax(-1, keepdim=True)
            if mref is None:
                mref, lsum, acc = bm, torch.zeros_like(bm), torch.zeros(*bm.shape[:-1], 64, dtype=torch.float64)
            else:
                grow = bm > mref + A.RESCALE_LOG2
                rescales += int(grow.sum())
                f = torch.where(grow, torch.exp2(mref - bm), torch.ones_like(bm))
                if acc_rescale:
                    acc = acc * f
                if lsum_rescale:
                    lsum = lsum * f
                mref = torch.where(grow, bm, mref)
            p = torch.exp2(blk - mref)
            lsum = lsum + p.sum(-1, keepdim=True)
            acc = acc + p.bfloat16().double() @ vb
        if mref is not None:
            parts.append((mref, lsum, acc))
    M = torch.maximum(parts[0][0], parts[-1][0])
    L = sum(l * torch.exp2(m - M) for m, l, _ in parts)
    O = sum(a * torch.exp2(m - M) for m, _, a in parts) / L
    return O.bfloat16().double(), ((M * A.LN2 + torch.log(L)).squeeze(-1)).float().double(), rescales


def _fwd_ratios(q, k, v, **kw):
    ref = A.attention_fwd(q, k, v)
    o, lse, nres = emulate_tc_forward(q, k, v, **kw)
    return A.worst_ratios({"o": o, "lse": lse}, ref, A.fwd_bounds(ref)), nres


@pytest.mark.parametrize("regime,T", [("flat", 197), ("flat", 272), ("sharp", 256), ("sharp_kmean", 197), ("staircase_up", 200),
                                      ("staircase_up", 256), ("staircase_down", 256), ("huge_pos", 192), ("huge_neg", 192), ("sink", 256)])
def test_error_model_covers_the_online_softmax(regime, T):
    kw = {"pos": 64} if regime == "sink" else {}
    qkv, _ = A.make_inputs(regime, 2, T, 2, 11, **kw)
    q, k, v = A.split_qkv(qkv, 2, T, 2)
    r, _ = _fwd_ratios(q, k, v)
    assert r["o"] <= 0.5 and r["lse"] <= 0.5, r


def test_flat_inputs_never_rescale_and_the_staircase_always_does():
    """The original inputs leave the lazy rescale unexecuted; staircase_up rescales every row on every non-first block of a warpgroup."""
    for T, heads in ((197, 12), (257, 16), (272, 1)):
        q, k, v = A.split_qkv(A.flat(2, T, heads, T + heads)[0], 2, T, heads)
        assert emulate_tc_forward(q, k, v)[2] == 0
    n, heads, T = 2, 2, 256
    q, k, v = A.split_qkv(A.staircase_up(n, T, heads, 3)[0], n, T, heads)
    assert emulate_tc_forward(q, k, v)[2] == n * heads * T * (T // 64 - 2)


@pytest.mark.parametrize("mutation", [{"lsum_rescale": False}, {"acc_rescale": False}])
def test_bounds_reject_a_forward_without_the_rescale(mutation):
    n, heads, T = 2, 2, 200
    q, k, v = A.split_qkv(A.staircase_up(n, T, heads, 4)[0], n, T, heads)
    r, nres = _fwd_ratios(q, k, v, **mutation)
    assert nres > 0 and r["o"] > 10, r
    # on the original inputs the same mutation is invisible: the rescale never runs
    q, k, v = A.split_qkv(A.flat(n, T, heads, 9)[0], n, T, heads)
    r, nres = _fwd_ratios(q, k, v, **mutation)
    assert nres == 0 and r["o"] <= 0.5, r


@pytest.mark.parametrize("T,pos", [(256, 0), (256, 63), (256, 64), (256, 255), (197, 196)])
def test_bounds_reject_a_dropped_sink_key(T, pos):
    qkv, _ = A.sink(1, T, 2, 6, pos)
    q, k, v = A.split_qkv(qkv, 1, T, 2)
    r, _ = _fwd_ratios(q, k, v, drop_key=pos)
    assert r["o"] > 10 and r["lse"] > 10, r


def test_bounds_reject_a_leaked_neighbour_key():
    """A tail block that lets image m+1's first rows into image m's softmax (no mask beyond T) is far outside the bound."""
    n, heads, T = 2, 1, 200
    qkv, _ = A.neighbour(n, T, heads, 7)
    q, k, v = A.split_qkv(qkv, n, T, heads)
    ref = A.attention_fwd(q[:1], k[:1], v[:1])
    leak = A.attention_fwd(q[:1], torch.cat([k[:1], k[1:, :, :8]], -2), torch.cat([v[:1], v[1:, :, :8]], -2))
    assert A.worst_ratios({"o": leak["o"]}, ref, {"o": A.fwd_bounds(ref)["o"]})["o"] > 1e3


def test_bounds_reject_a_backward_with_a_stale_delta():
    """delta from the float64 O instead of the bf16 ctx the kernel reads is a real (small) difference; a dS without the -delta term
    is far outside."""
    n, heads, T = 1, 2, 130
    qkv, dO = A.sharp(n, T, heads, 8)
    q, k, v = A.split_qkv(qkv, n, T, heads)
    dO = A.rows_to_heads(dO, n, T, heads)
    fw = A.attention_fwd(q, k, v)
    ctx = fw["o"].bfloat16()
    ref = A.attention_bwd(q, k, v, ctx, fw["lse"].float(), dO)
    b = A.bwd_bounds(ref)
    same = A.attention_bwd(q, k, v, ctx, fw["lse"].float(), dO)
    assert max(A.worst_ratios(same, ref, b).values()) == 0.0
    no_delta = A.attention_bwd(q, k, v, torch.zeros_like(ctx), fw["lse"].float(), dO)
    r = A.worst_ratios(no_delta, ref, b)
    assert r["dq"] > 10 and r["dk"] > 10 and r["dv"] == 0.0, r
