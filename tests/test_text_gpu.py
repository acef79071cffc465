"""GPU tests of the CLIP text tower (CLIPModelB200.encode_text): the causal tcgen05 attention forward against a masked softmax, the
whole tower against the fp32 CPU oracle (oracle/clip_text.py, cross-checked against transformers in test_text_cpu.py), causality end
to end, and the public path embed_text -> {"embeddings", "weights"} -> GuidanceStep."""
import pytest
import torch

pytestmark = pytest.mark.gpu

COS_MIN = 0.999
NAMES = ["ViT-B/32", "ViT-B/16", "ViT-L/14", "ViT-L/14@336px"]


CAUSAL_SHAPES = [(1, 77, 8), (4, 77, 12), (200, 77, 8),  # (200 x 8 items: more than SMs, several per CTA)
                 (2, 1, 2), (2, 2, 2), (2, 63, 2), (2, 64, 2), (2, 65, 2), (1, 128, 2), (2, 129, 2), (1, 200, 3), (1, 257, 2), (1, 272, 2)]


def _causal_cases():
    """The original shapes on flat inputs; sharp regimes of oracle/attention.py at T = 77 (one block per warpgroup and tile: no rescale
    possible, a control), 200, 257 and 272, with 1, 4 and 16 heads."""
    cases = [pytest.param(n, T, heads, "flat", id="%d-%d-%d" % (n, T, heads)) for n, T, heads in CAUSAL_SHAPES]
    i = 0
    for regime in ("sharp", "sharp_kmean", "staircase_up", "staircase_down", "huge_pos", "huge_neg", "neighbour", "sink"):
        for T in (77, 200, 257, 272):
            heads, n = (1, 4, 16)[i % 3], 3 if regime == "neighbour" else 2
            i += 1
            cases.append(pytest.param(n, T, heads, regime, id="%d-%d-%d-%s" % (n, T, heads, regime)))
    return cases


@pytest.mark.parametrize("n,T,heads,regime", _causal_cases())
def test_causal_attention_fwd(n, T, heads, regime, record_property):
    """The causal tcgen05 forward against the float64 masked softmax within the error model of oracle/attention.py, in guarded buffers
    (oracle/attention.py: attention_fwd_guarded).  A sink sits at key 0, which every row keeps."""
    from oracle import attention as A

    seed = T + heads + n if regime == "flat" else 1000 * n + T + heads
    qkv, _ = A.make_inputs(regime, n, T, heads, seed, causal=True, **({"pos": 0} if regime == "sink" else {}))
    qkv = qkv.cuda()
    ref = A.attention_fwd(*A.split_qkv(qkv, n, T, heads), causal=True)
    ctx, lse = A.attention_fwd_guarded(qkv, n, T, heads, causal=True)
    worst = A.worst_ratios({"o": A.rows_to_heads(ctx, n, T, heads), "lse": lse}, ref, A.fwd_bounds(ref))
    record_property("err_over_bound", {"kernel": "tcgen05 causal", "regime": regime, **worst})
    assert max(worst.values()) <= 1.0, worst


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
