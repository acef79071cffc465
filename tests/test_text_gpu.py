"""GPU tests of the CLIP text tower (CLIPModelB200.encode_text): the causal tcgen05 attention forward against a masked softmax, the
whole tower against the fp32 CPU oracle (oracle/clip_text.py, cross-checked against transformers in test_text_cpu.py), causality end
to end, and the public path embed_text -> {"embeddings", "weights"} -> GuidanceStep."""
import pytest
import torch

pytestmark = pytest.mark.gpu

COS_MIN = 0.999
NAMES = ["ViT-B/32", "ViT-B/16", "ViT-L/14", "ViT-L/14@336px"]


@pytest.mark.parametrize("n,T,heads", [(1, 77, 8), (4, 77, 12), (200, 77, 8),  # (200 x 8 items: more than SMs, several per CTA)
                                       (2, 1, 2), (2, 2, 2), (2, 63, 2), (2, 64, 2), (2, 65, 2), (1, 128, 2), (2, 129, 2), (1, 200, 3),
                                       (1, 257, 2), (1, 272, 2)])
def test_causal_attention_fwd(n, T, heads):
    from clip_diffusion_b200 import _lib

    D = heads * 64
    g = torch.Generator().manual_seed(T + heads + n)
    qkv = (torch.randn(n * T, 3 * D, generator=g) * 0.8).bfloat16()
    q, k, v = [t.float().view(n, T, heads, 64).transpose(1, 2) for t in qkv.split(D, dim=1)]
    s = (q @ k.transpose(-1, -2)) * 0.125
    s = s.masked_fill(torch.ones(T, T, dtype=torch.bool).triu(1), float("-inf"))
    ref = torch.softmax(s, -1) @ v
    lse_ref = torch.logsumexp(s, -1)
    P = _lib.ptr
    qc = qkv.cuda()
    ctx = torch.full((n * T, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    lse = torch.full((n, heads, T), float("nan"), device="cuda")
    _lib.call("cg_attention_causal_fwd", P(qc), n, T, heads, P(ctx), P(lse))
    out = ctx.float().cpu().view(n, T, heads, 64).transpose(1, 2)
    assert torch.isfinite(out).all() and torch.isfinite(lse.cpu()).all()
    assert (out - ref).abs().max().item() < 2e-2 * max(1.0, ref.abs().max().item())
    assert (lse.cpu() - lse_ref).abs().max().item() < 2e-3


def _prompts(seed, n_extra=3):
    """clip.tokenize-shaped ids: the empty prompt (EOT at 1), a full one (EOT at 76) and random lengths in between."""
    from oracle.clip_text import random_prompt_tokens

    g = torch.Generator().manual_seed(seed)
    lengths = [0, 75] + torch.randint(1, 75, (n_extra,), generator=g).tolist()
    return random_prompt_tokens(lengths, 77, g)


@pytest.mark.parametrize("name", NAMES)
def test_text_tower_matches_oracle(name):
    from clip_diffusion_b200 import models
    from oracle.clip_text import OracleCLIPText

    sd = models.random_clip_text_state_dict(name, seed=3)
    mine = models.CLIPModelB200(name, dict(models.random_clip_state_dict(name, seed=3), **sd), "cuda")
    ref = OracleCLIPText(name, state_dict=sd)
    tokens = _prompts(len(name))
    want = ref.encode_text(tokens)
    got = mine.encode_text(tokens.cuda())
    assert got.dtype == torch.float32 and got.shape == want.shape and got.grad_fn is None
    cos = torch.nn.functional.cosine_similarity(got.cpu(), want, dim=-1)
    assert cos.min().item() >= COS_MIN, cos
    # int32 ids (what the kernels read) give the same result as int64
    assert torch.equal(mine.encode_text(tokens.int().cuda()), got)


def test_text_is_causal_end_to_end():
    """Ids after the EOT of a prompt never reach its embedding: replacing every one of them changes nothing, bit for bit."""
    from clip_diffusion_b200 import models

    m = models.CLIPModelB200("ViT-B/32", None, "cuda", seed=4)
    tokens = _prompts(9)
    eot = tokens.argmax(-1)
    noisy = tokens.clone()
    g = torch.Generator().manual_seed(10)
    for i, e in enumerate(eot.tolist()):
        noisy[i, e + 1:] = torch.randint(0, 49407, (76 - e,), generator=g)  # below the EOT id: it stays the first maximum
    assert not torch.equal(noisy, tokens)
    a = m.encode_text(tokens.cuda())
    b = m.encode_text(noisy.cuda())
    assert torch.equal(a, b)


def test_embed_text_feeds_the_guidance_step():
    from clip_diffusion_b200.models import load_clip_models
    from clip_diffusion_b200.sample import GuidanceStep
    from clip_diffusion_b200.utils.functional import embed_text

    models = load_clip_models(["ViT-B/32"], allow_random_init=True)
    m = models["ViT-B/32"]
    tokens = _prompts(12, n_extra=1).cuda()
    emb = embed_text(m, tokens)
    assert emb.shape == (3, m.visual.output_dim) and torch.isfinite(emb).all()
    # preprocessing.py:11-24: one {"embeddings", "weights"} dict per CLIP model
    text = {"ViT-B/32": {"embeddings": emb, "weights": torch.tensor([1.0, 0.5, -0.25], device="cuda")}}
    x_in = torch.tanh(torch.randn(1, 3, 256, 256, generator=torch.Generator().manual_seed(13))).cuda().contiguous()
    grad = GuidanceStep(None, None, models, text).clip_guidance_grad(x_in, 500, torch.zeros(3, 256, 256, device="cuda"))
    assert torch.isfinite(grad).all() and grad.abs().max().item() > 0
