"""Float64 reference of the fused attention kernels (csrc/vit_attention_tc.cu, csrc/vit_attention.cu), their error model, and input
regimes that reach the kernels' rarely taken paths (TEST-ONLY, torch; runs on whatever device the inputs are on).

Layout of the kernels: packed qkv [n*T, 3*D] bf16 (q | k | v, head h = columns h*64 .. h*64+63 of each third), ctx / dO [n*T, D],
lse [n, heads, T] fp32, scale 0.125 (head_dim 64).  The reference works on [n, heads, T, 64] float64 tensors.

Error model (u = 2^-8, the unit roundoff of bf16).  The kernels round P and dS to bf16 for the MMAs, accumulate in fp32, take the row
sum from the unrounded fp32 P and round their outputs to bf16.  Per element, with the magnitudes returned by the reference:

    |O - O_ref|     <= 2^-6 (P @ |V|)                     2x the worst case of P rounding plus output rounding (2u)
    |lse - lse_ref| <= 1e-4 + 2^-18 max_j Sabs_ij + 1e-6 |lse_ref|      Sabs = 0.125 |Q| @ |K|^T: fp32 / tensor-core sums of 64 products
    |dV - dV_ref|   <= 2^-6 (P^T @ |dO|)
    |dQ - dQ_ref|   <= 2^-6 0.125 (S^ @ |K|)              S^ = P o (|dO @ V^T| + |delta|): dS = P (dP - delta) rounded to bf16
    |dK - dK_ref|   <= 2^-6 0.125 (S^^T @ |Q|)

plus TINY = 1e-20 on the four tensor bounds: the kernels evaluate exp2 with flush-to-zero, so a P below 2^-126 (a key more than 87 nats
under its row's maximum) is exactly 0 there; every such term is far below TINY.  The backward reference is fed exactly what the kernel
reads: the bf16 ctx (delta = rowsum(dO o ctx)) and the fp32 lse (P = exp(0.125 Q K^T - lse)).

Input regimes (each generator asserts its defining property on the bf16-rounded values before it returns):
    flat           qkv = 0.8 N(0,1): logit std 0.64, softmax close to uniform (the inputs of the original tests)
    sharp          q, k = 2.5 N(0,1): logit std ~6, row maximum ~18 nats above the row mean;  sharp_kmean: the same with k += 1
    staircase_up   every 64-key block's smallest logit >= 12 log2 units above the largest logit of every earlier block, for every row:
                   the lazy rescale of the tcgen05 forward (RESCALE_LOG2 = 8) runs on every non-first block of every warpgroup
    staircase_down the reverse: later blocks sit >= 12 log2 units under every earlier block
    sink           one key (position `pos`) >= 25 nats above every other key of every row;  sink_query: the last query row gets a
                   staircase instead (the edge query row when T = 64 m + 1)
    huge_pos/neg   logits in [100, 200] / [-200, -100] nats, Sabs <= 300
    neighbour      rows 0-15 of image m+1 hold keys >= 30 nats above all of image m's keys for image m's queries, with |V| ~ 1e3: any
                   key beyond T that reaches a softmax or P V unmasked lands far outside the bound
"""
import math

import torch

SCALE = 0.125
HD = 64
LN2 = math.log(2.0)
U = 2.0 ** -8
C_TENSOR = 2.0 ** -6
TINY = 1e-20
RESCALE_LOG2 = 8.0  # the tcgen05 forward moves a warpgroup's reference maximum when a block exceeds it by more than this (log2 units)


# ---------------------------------------------------------------------------------------------------------------- layout helpers
def split_qkv(qkv, n, T, heads):
    """bf16 [n*T, 3*D] -> q, k, v float64 [n, heads, T, 64]."""
    D = heads * HD
    return [t.double().reshape(n, T, heads, HD).transpose(1, 2) for t in qkv.split(D, dim=1)]


def rows_to_heads(x, n, T, heads):
    """[n*T, heads*64] (any dtype) -> float64 [n, heads, T, 64]."""
    return x.double().reshape(n, T, heads, HD).transpose(1, 2)


def heads_to_rows(x):
    """[n, heads, T, 64] -> [n*T, heads*64]."""
    n, heads, T, _ = x.shape
    return x.transpose(1, 2).reshape(n * T, heads * HD)


def _causal_mask(T, device):
    return torch.ones(T, T, dtype=torch.bool, device=device).triu(1)


# ---------------------------------------------------------------------------------------------------------------- reference
def logits(q, k, causal=False):
    s = SCALE * (q.double() @ k.double().transpose(-1, -2))
    if causal:
        s = s.masked_fill(_causal_mask(s.shape[-1], s.device), float("-inf"))
    return s


def attention_fwd(q, k, v, causal=False):
    """float64 forward: O, lse and the bound magnitudes P @ |V| and Sabs = 0.125 |Q| @ |K|^T (0 at masked keys)."""
    q, k, v = q.double(), k.double(), v.double()
    s = logits(q, k, causal)
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse.unsqueeze(-1))
    sabs = SCALE * (q.abs() @ k.abs().transpose(-1, -2))
    if causal:
        sabs = sabs.masked_fill(_causal_mask(s.shape[-1], s.device), 0.0)
    return {"o": p @ v, "lse": lse, "pv_abs": p @ v.abs(), "sabs": sabs}


def attention_bwd(q, k, v, ctx, lse, dO):
    """float64 backward on exactly the tensors the kernel reads: P = exp(0.125 Q K^T - lse) with the given (fp32) lse, and
    delta = rowsum(dO o ctx) with the given (bf16) ctx.  Returns dq, dk, dv and the magnitudes P^T @ |dO|, S^ @ |K|, S^^T @ |Q|."""
    q, k, v, ctx, dO = q.double(), k.double(), v.double(), ctx.double(), dO.double()
    p = torch.exp(logits(q, k) - lse.double().unsqueeze(-1))
    dp = dO @ v.transpose(-1, -2)
    delta = (dO * ctx).sum(-1, keepdim=True)
    ds = p * (dp - delta)
    shat = p * (dp.abs() + delta.abs())
    return {"dq": SCALE * (ds @ k), "dk": SCALE * (ds.transpose(-1, -2) @ q), "dv": p.transpose(-1, -2) @ dO,
            "ptdo_abs": p.transpose(-1, -2) @ dO.abs(), "shat_k": shat @ k.abs(), "shat_q": shat.transpose(-1, -2) @ q.abs()}


# ---------------------------------------------------------------------------------------------------------------- bounds
def fwd_bounds(ref):
    return {"o": C_TENSOR * ref["pv_abs"] + TINY,
            "lse": 1e-4 + 2.0 ** -18 * ref["sabs"].amax(-1) + 1e-6 * ref["lse"].abs()}


def bwd_bounds(ref):
    return {"dq": C_TENSOR * SCALE * ref["shat_k"] + TINY, "dk": C_TENSOR * SCALE * ref["shat_q"] + TINY,
            "dv": C_TENSOR * ref["ptdo_abs"] + TINY}


def worst_ratios(got, ref, bounds):
    """max |got - ref| / bound per output (inf when an output holds a non-finite value).  <= 1 everywhere: within the error model."""
    out = {}
    for name, b in bounds.items():
        g = got[name].double().to(b.device)
        if not torch.isfinite(g).all():
            out[name] = float("inf")
            continue
        out[name] = ((g - ref[name].to(b.device)).abs() / b).max().item()
    return out


# ---------------------------------------------------------------------------------------------------------------- input regimes
def _bf(x):
    return x.bfloat16().double()


def _noise(g, shape, std, zero_dims=1):
    """N(0, std^2) in the last dimension's columns >= zero_dims, exactly 0 in the first zero_dims (the directions the regimes steer)."""
    x = torch.randn(*shape, generator=g, dtype=torch.float64) * std
    x[..., :zero_dims] = 0.0
    return x


def _pack(q, k, v, g):
    """[n, heads, T, 64] float64 -> bf16 qkv [n*T, 3*D] and dO = 0.5 N(0,1) bf16 [n*T, D]."""
    qkv = torch.cat([heads_to_rows(t) for t in (q, k, v)], dim=1).bfloat16()
    dO = (torch.randn(qkv.shape[0], qkv.shape[1] // 3, generator=g) * 0.5).bfloat16()
    return qkv, dO


def _block_extrema(s, T):
    """Per-row max / min of each 64-key block over the finite (kept) logits: [..., T, nblocks] each (-inf / +inf for none)."""
    nb = (T + 63) // 64
    mx, mn = [], []
    for b in range(nb):
        blk = s[..., b * 64:(b + 1) * 64]
        fin = torch.isfinite(blk)
        mx.append(torch.where(fin, blk, torch.full_like(blk, float("-inf"))).amax(-1))
        mn.append(torch.where(fin, blk, torch.full_like(blk, float("inf"))).amin(-1))
    return torch.stack(mx, -1), torch.stack(mn, -1)


def staircase_rise(s, T):
    """Smallest (over rows and non-first blocks with a kept key) of  min(block b) - max(blocks < b), in nats."""
    mx, mn = _block_extrema(s, T)
    prev = torch.cummax(mx, -1).values[..., :-1]
    rise = mn[..., 1:] - prev
    return rise[torch.isfinite(rise)].min().item() if torch.isfinite(rise).any() else float("inf")


def staircase_fall(s, T):
    """Smallest of  min(blocks < b) - max(block b), in nats (over rows and non-first blocks with a kept key)."""
    mx, mn = _block_extrema(s, T)
    prev = torch.cummin(mn, -1).values[..., :-1]
    fall = prev - mx[..., 1:]
    return fall[torch.isfinite(fall)].min().item() if torch.isfinite(fall).any() else float("inf")


def flat(n, T, heads, seed):
    """The original tests' inputs (same generator draws): qkv = 0.8 N(0,1), dO = 0.5 N(0,1)."""
    D = heads * HD
    g = torch.Generator().manual_seed(seed)
    qkv = (torch.randn(n * T, 3 * D, generator=g) * 0.8).bfloat16()
    dO = (torch.randn(n * T, D, generator=g) * 0.5).bfloat16()
    s = logits(*split_qkv(qkv, n, T, heads)[:2])
    assert s.numel() < 2 or s.std().item() < 1.0, "flat: logit std %g" % s.std().item()
    return qkv, dO


def sharp(n, T, heads, seed, kmean=0.0):
    g = torch.Generator().manual_seed(seed)
    shape = (n, heads, T, HD)
    q = _bf(torch.randn(*shape, generator=g, dtype=torch.float64) * 2.5)
    k = _bf(torch.randn(*shape, generator=g, dtype=torch.float64) * 2.5 + kmean)
    v = _bf(torch.randn(*shape, generator=g, dtype=torch.float64) * 0.8)
    s = logits(q, k)
    sd = (s - s.mean(-1, keepdim=True)).std().item()
    assert 5.0 < sd < 7.5, "sharp: centred logit std %g" % sd
    assert (s.amax(-1) - s.mean(-1)).mean().item() > 12.0, "sharp: row maxima too close to the row means"
    return _pack(q, k, v, g)


def sharp_kmean(n, T, heads, seed):
    return sharp(n, T, heads, seed, kmean=1.0)


def _staircase_keys(T, up, step=12.0):
    """Key component along e0 (with the query component 8 along e0 the logit moves by `step` nats per 64-key block)."""
    nb = (T + 63) // 64
    lvl = torch.tensor([(j // 64) if up else (nb - 1 - j // 64) for j in range(T)], dtype=torch.float64)
    return lvl * (step / (SCALE * 8.0))


def staircase(n, T, heads, seed, up=True, causal=False):
    g = torch.Generator().manual_seed(seed)
    shape = (n, heads, T, HD)
    q = _noise(g, shape, 0.3)
    q[..., 0] = 8.0
    k = _noise(g, shape, 0.3)
    k[..., 0] = _staircase_keys(T, up)
    q, k = _bf(q), _bf(k)
    v = _bf(torch.randn(*shape, generator=g, dtype=torch.float64) * 0.8)
    s = logits(q, k, causal)
    if T > 64:
        if up:
            r = staircase_rise(s, T)
            assert r >= 12 * LN2, "staircase_up: smallest block rise %g nats" % r
        else:
            f = staircase_fall(s, T)
            assert f >= 12 * LN2, "staircase_down: smallest block fall %g nats" % f
    return _pack(q, k, v, g)


def staircase_up(n, T, heads, seed, causal=False):
    return staircase(n, T, heads, seed, True, causal)


def staircase_down(n, T, heads, seed, causal=False):
    return staircase(n, T, heads, seed, False, causal)


def sink_positions(T, edge):
    """0, 63, 64, the last column of the pipeline's tail block (T - edge - 1) and T - 1 (the edge key when edge = 1), inside [0, T)."""
    return sorted({p for p in (0, 63, 64, T - edge - 1, T - 1) if 0 <= p < T})


def sink(n, T, heads, seed, pos, query_staircase=False):
    g = torch.Generator().manual_seed(seed)
    shape = (n, heads, T, HD)
    q = _noise(g, shape, 0.7, zero_dims=2)
    q[..., 0] = 8.0
    k = _noise(g, shape, 0.7, zero_dims=2)
    k[..., pos, 0] = 30.0 / (SCALE * 8.0)
    if query_staircase:
        q[..., T - 1, :] = _noise(g, (n, heads, HD), 0.3, zero_dims=2)
        q[..., T - 1, 1] = 8.0
        k[..., 1] = _staircase_keys(T, True)
    q, k = _bf(q), _bf(k)
    v = _bf(torch.randn(*shape, generator=g, dtype=torch.float64) * 0.8)
    s = logits(q, k)
    rows = slice(0, T - 1) if query_staircase else slice(0, T)
    sr = s[..., rows, :]
    rest = torch.cat([sr[..., :pos], sr[..., pos + 1:]], -1)
    if rest.shape[-1]:
        gap = (sr[..., pos] - rest.amax(-1)).min().item()
        assert gap >= 25.0, "sink: key %d only %g nats above the rest" % (pos, gap)
    if query_staircase and T > 64:
        r = staircase_rise(s[..., T - 1:, :], T)
        assert r >= 12 * LN2, "sink_query: smallest block rise of the last query row %g nats" % r
    return _pack(q, k, v, g)


def sink_query(n, T, heads, seed, pos=0):
    return sink(n, T, heads, seed, pos, query_staircase=True)


def huge(n, T, heads, seed, sign=1.0, causal=False):
    g = torch.Generator().manual_seed(seed)
    shape = (n, heads, T, HD)
    q = _noise(g, shape, 1.0)
    q[..., 0] = 8.0 * sign
    k = _noise(g, shape, 1.0)
    k[..., 0] = 150.0 + torch.randint(-4, 5, (n, heads, T), generator=g).double()
    q, k = _bf(q), _bf(k)
    v = _bf(torch.randn(*shape, generator=g, dtype=torch.float64) * 0.8)
    ref = attention_fwd(q, k, v, causal)
    s = logits(q, k, causal)
    fin = s[torch.isfinite(s)].abs()
    assert fin.min().item() >= 100.0 and fin.max().item() <= 200.0, "huge: |logits| in [%g, %g]" % (fin.min(), fin.max())
    assert ref["sabs"].max().item() <= 300.0, "huge: Sabs %g" % ref["sabs"].max()
    return _pack(q, k, v, g)


def huge_pos(n, T, heads, seed, causal=False):
    return huge(n, T, heads, seed, 1.0, causal)


def huge_neg(n, T, heads, seed, causal=False):
    return huge(n, T, heads, seed, -1.0, causal)


def neighbour(n, T, heads, seed, causal=False):
    """Image m's queries point along e_(m mod 2); rows 0-15 of image m+1 carry keys 40 / (0.125 * 8) along that direction (and |V| ~ 1e3),
    image m's own keys have no component there."""
    assert n >= 2 and T >= 16
    g = torch.Generator().manual_seed(seed)
    shape = (n, heads, T, HD)
    q = _noise(g, shape, 1.0, zero_dims=2)
    k = _noise(g, shape, 1.0, zero_dims=2)
    v = torch.randn(*shape, generator=g, dtype=torch.float64) * 0.8
    for m in range(n):
        q[m, ..., m % 2] = 8.0
        if m >= 1:
            k[m, :, :16, (m - 1) % 2] = 40.0 / (SCALE * 8.0)
            v[m, :, :16] *= 1250.0
    q, k, v = _bf(q), _bf(k), _bf(v)
    for m in range(n - 1):
        own = logits(q[m], k[m], causal)
        cross = logits(q[m], k[m + 1, :, :16])
        gap = (cross.amin(-1) - own.amax(-1)).min().item()
        assert gap >= 30.0, "neighbour: image %d's neighbour keys only %g nats above its own" % (m, gap)
    assert v[1:, :, :16].abs().mean().item() > 500.0
    return _pack(q, k, v, g)


REGIMES = {"flat": flat, "sharp": sharp, "sharp_kmean": sharp_kmean, "staircase_up": staircase_up, "staircase_down": staircase_down,
           "sink": sink, "sink_query": sink_query, "huge_pos": huge_pos, "huge_neg": huge_neg, "neighbour": neighbour}
CAUSAL_AWARE = ("staircase_up", "staircase_down", "huge_pos", "huge_neg", "neighbour")  # generators whose check depends on the mask


def make_inputs(regime, n, T, heads, seed, causal=False, **kw):
    """bf16 qkv [n*T, 3D] and dO [n*T, D] of a regime (kw: `pos` of a sink)."""
    fn = REGIMES[regime]
    if regime in CAUSAL_AWARE:
        kw["causal"] = causal
    return fn(n, T, heads, seed, **kw)


def mixed(regimes, T, heads, seed, causal=False):
    """One image per entry of `regimes` (image i from seed + i), stacked into one batch."""
    parts = [make_inputs(r, 1, T, heads, seed + i, causal) for i, r in enumerate(regimes)]
    return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])


# ---------------------------------------------------------------------------------------------------------------- guarded buffers
GUARD = 512  # sentinel elements on each side of an output buffer
_SENTINEL = {torch.bfloat16: (torch.int16, 0x5AA5), torch.float32: (torch.int32, 0x5AA55AA5)}


class Guarded:
    """An output buffer filled with NaN inside a larger allocation whose GUARD elements on either side hold a sentinel bit pattern:
    after a kernel, every element must be finite (written) and every guard bit-identical (nothing written outside)."""

    def __init__(self, shape, dtype, device="cuda"):
        numel = math.prod(shape)
        self.bits_dtype, self.pattern = _SENTINEL[dtype]
        self.buf = torch.empty(2 * GUARD + numel, dtype=dtype, device=device)
        self.buf.view(self.bits_dtype).fill_(self.pattern)
        self.t = self.buf[GUARD:GUARD + numel].view(shape)
        self.t.fill_(float("nan"))

    def guards_intact(self):
        bits = self.buf.view(self.bits_dtype)
        return bool((bits[:GUARD] == self.pattern).all()) and bool((bits[-GUARD:] == self.pattern).all())


def nan_tailed(x, extra=4096, device="cuda"):
    """A device copy of x at the start of an allocation whose remaining `extra` elements are NaN: a read past the end of x that reaches
    the arithmetic shows up as a NaN in the result."""
    buf = torch.full((x.numel() + extra,), float("nan"), dtype=x.dtype, device=device)
    buf[:x.numel()] = x.reshape(-1).to(device)
    return buf[:x.numel()].view(x.shape)


# ---------------------------------------------------------------------------------------------------------------- kernel harness
# (needs the built library and a GPU; the C ABI of include/clipguide_b200.h)
def attention_fwd_guarded(qkv, n, T, heads, causal=False):
    """cg_attention_(causal_)fwd with qkv followed by NaN rows and NaN-filled, sentinel-guarded ctx / lse: returns ctx [n*T, D] bf16 and
    lse [n, heads, T] after checking that every element was written and nothing outside them was."""
    from clip_diffusion_b200 import _lib

    P = _lib.ptr
    qc = nan_tailed(qkv)
    ctx, lse = Guarded((n * T, heads * 64), torch.bfloat16), Guarded((n, heads, T), torch.float32)
    _lib.call("cg_attention_causal_fwd" if causal else "cg_attention_fwd", P(qc), n, T, heads, P(ctx.t), P(lse.t))
    torch.cuda.synchronize()
    assert ctx.guards_intact() and lse.guards_intact(), "forward wrote outside ctx / lse"
    assert torch.isfinite(ctx.t).all() and torch.isfinite(lse.t).all(), "forward left ctx / lse elements unwritten or non-finite"
    return ctx.t.clone(), lse.t.clone()


def attention_bwd_guarded(qkv, ctx, dctx, lse, n, T, heads):
    """cg_attention_bwd with every input followed by NaN and NaN-filled, sentinel-guarded dqkv / delta workspace: returns dqkv."""
    from clip_diffusion_b200 import _lib

    P = _lib.ptr
    qc, cc, dc, lc = (nan_tailed(t) for t in (qkv, ctx, dctx, lse))
    dqkv, delta = Guarded((n * T, 3 * heads * 64), torch.bfloat16), Guarded((n, heads, T), torch.float32)
    _lib.call("cg_attention_bwd", P(qc), P(cc), P(dc), P(lc), n, T, heads, P(dqkv.t), P(delta.t))
    torch.cuda.synchronize()
    assert dqkv.guards_intact() and delta.guards_intact(), "backward wrote outside dqkv / delta"
    assert torch.isfinite(dqkv.t).all(), "backward left dqkv elements unwritten or non-finite"
    if T > _lib.ATTN_TC_MAX_T:  # the mma.sync backward fills the delta workspace; the tcgen05 one keeps delta on chip
        assert torch.isfinite(delta.t).all()
    return dqkv.t.clone()


def check_attention(n, T, heads, qkv, dctx, chained=False):
    """Forward, and backward on the oracle's bf16 ctx / fp32 lse (or, chained, on the kernel's own), against the float64 reference
    within the error model above.  Returns the worst err / bound of each output."""
    qkv, dctx = qkv.cuda(), dctx.cuda()
    q, k, v = split_qkv(qkv, n, T, heads)
    ref = attention_fwd(q, k, v)
    ctx, lse = attention_fwd_guarded(qkv, n, T, heads)
    worst = worst_ratios({"o": rows_to_heads(ctx, n, T, heads), "lse": lse}, ref, fwd_bounds(ref))
    ctx_in, lse_in = (ctx, lse) if chained else (heads_to_rows(ref["o"]).bfloat16(), ref["lse"].float())
    del ref
    dqkv = attention_bwd_guarded(qkv, ctx_in, dctx, lse_in, n, T, heads)
    bref = attention_bwd(q, k, v, rows_to_heads(ctx_in, n, T, heads), lse_in, rows_to_heads(dctx, n, T, heads))
    got = dict(zip(("dq", "dk", "dv"), (rows_to_heads(t, n, T, heads) for t in dqkv.split(heads * 64, dim=1))))
    worst.update(worst_ratios(got, bref, bwd_bounds(bref)))
    return worst
