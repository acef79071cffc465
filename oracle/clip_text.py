"""Oracle restatement of the OpenAI CLIP text transformer, ``CLIP.encode_text`` (TEST-ONLY, CPU torch fp32).

The reference reaches it through embed_text (clip_diffusion/utils/functional.py:91-94) from
get_text_embeddings_and_text_weights (preprocessing.py:11-24); the ``clip`` package itself is not
vendored, so this restates the published architecture:

    x = token_embedding[tokens] + positional_embedding
    x = L x {x += MHA(ln_1 x, causal mask); x += c_proj(QuickGELU(c_fc(ln_2 x)))}
    out = ln_final(x)[arange(N), tokens.argmax(-1)] @ text_projection

with the residual blocks of oracle/clip_vit.py and OpenAI's causal mask (-inf above the diagonal).
Parity against openai/CLIP is UNPINNED; tests cross-check against transformers'
CLIPTextModelWithProjection(hidden_act="quick_gelu", eos_token_id=2: argmax pooling) with mapped weights.

State-dict keys follow OpenAI's top-level names (token_embedding.weight, transformer.resblocks.<i>.*, ...).
"""
import torch
from torch import nn

from oracle.clip_vit import Transformer

TEXT_CONFIGS = {
    # name: (context_length, vocab_size, width, layers, heads, embed_dim)
    "ViT-B/32": (77, 49408, 512, 12, 8, 512),
    "ViT-B/16": (77, 49408, 512, 12, 8, 512),
    "ViT-L/14": (77, 49408, 768, 12, 12, 768),
    "ViT-L/14@336px": (77, 49408, 768, 12, 12, 768),
}


def random_text_state_dict(name: str, seed: int = 1):
    """OpenAI's CLIP.initialize_parameters for the text side, with LayerNorm affines and biases perturbed so that tests see them."""
    context, vocab, width, layers, heads, embed = TEXT_CONFIGS[name]
    g = torch.Generator().manual_seed(seed)

    def randn(*s):
        return torch.randn(*s, generator=g)

    proj_std = width ** -0.5 * (2 * layers) ** -0.5
    sd = {"token_embedding.weight": 0.02 * randn(vocab, width), "positional_embedding": 0.01 * randn(context, width)}
    for i in range(layers):
        p = f"transformer.resblocks.{i}."
        sd[p + "attn.in_proj_weight"] = width ** -0.5 * randn(3 * width, width)
        sd[p + "attn.in_proj_bias"] = 0.02 * randn(3 * width)
        sd[p + "attn.out_proj.weight"] = proj_std * randn(width, width)
        sd[p + "attn.out_proj.bias"] = 0.02 * randn(width)
        sd[p + "mlp.c_fc.weight"] = (2 * width) ** -0.5 * randn(4 * width, width)
        sd[p + "mlp.c_fc.bias"] = 0.02 * randn(4 * width)
        sd[p + "mlp.c_proj.weight"] = proj_std * randn(width, 4 * width)
        sd[p + "mlp.c_proj.bias"] = 0.02 * randn(width)
        for n in ("ln_1", "ln_2"):
            sd[p + n + ".weight"] = 1.0 + 0.1 * randn(width)
            sd[p + n + ".bias"] = 0.1 * randn(width)
    sd["ln_final.weight"] = 1.0 + 0.1 * randn(width)
    sd["ln_final.bias"] = 0.1 * randn(width)
    sd["text_projection"] = width ** -0.5 * randn(width, embed)
    return sd


class OracleCLIPText(nn.Module):
    """The text half of the object ``clip.load`` returns: ``encode_text(tokens)`` on token ids [N, context]."""

    def __init__(self, name: str, state_dict=None, seed: int = 1):
        super().__init__()
        context, vocab, width, layers, heads, embed = TEXT_CONFIGS[name]
        self.context_length = context
        self.token_embedding = nn.Embedding(vocab, width)
        self.positional_embedding = nn.Parameter(torch.zeros(context, width))
        self.transformer = Transformer(width, layers, heads)
        self.ln_final = nn.LayerNorm(width)
        self.text_projection = nn.Parameter(torch.zeros(width, embed))
        # OpenAI's build_attention_mask: additive, -inf strictly above the diagonal
        self.register_buffer("attn_mask", torch.full((context, context), float("-inf")).triu_(1), persistent=False)
        sd = state_dict if state_dict is not None else random_text_state_dict(name, seed)
        self.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=True)
        self.eval().requires_grad_(False)

    def encode_text(self, text):
        x = self.token_embedding(text) + self.positional_embedding
        x = x.permute(1, 0, 2)  # [T, N, D]
        for blk in self.transformer.resblocks:  # ResidualAttentionBlock.forward with OpenAI's attn_mask
            y = blk.ln_1(x)
            x = x + blk.attn(y, y, y, need_weights=False, attn_mask=self.attn_mask.to(x.dtype))[0]
            x = x + blk.mlp(blk.ln_2(x))
        x = self.ln_final(x.permute(1, 0, 2))
        return x[torch.arange(x.shape[0], device=x.device), text.argmax(dim=-1)] @ self.text_projection


SOT, EOT = 49406, 49407  # clip.tokenize's <|startoftext|> and <|endoftext|>


def random_prompt_tokens(lengths, context=77, generator=None):
    """int64 [len(lengths), context] shaped like clip.tokenize output: SOT, `length` random word ids below SOT, EOT, zero padding
    (length 0: the empty prompt, EOT at position 1; length context - 2: EOT at the last position)."""
    out = torch.zeros(len(lengths), context, dtype=torch.long)
    for i, n in enumerate(lengths):
        if not 0 <= n <= context - 2:
            raise ValueError("a prompt holds 0 .. %d word tokens" % (context - 2))
        out[i, 0] = SOT
        out[i, 1:n + 1] = torch.randint(0, SOT, (n,), generator=generator)
        out[i, n + 1] = EOT
    return out
