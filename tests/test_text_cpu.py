"""CPU tests of the CLIP text tower: the fp32 oracle (oracle/clip_text.py) against transformers' CLIP text model, the state-dict
helpers, lazy loading of the text weights, token validation and the causal attention's argument check."""
import ctypes

import pytest
import torch


def test_oracle_text_matches_hf_clip():
    from transformers import CLIPTextConfig, CLIPTextModelWithProjection

    from oracle.clip_text import TEXT_CONFIGS, OracleCLIPText, random_prompt_tokens, random_text_state_dict

    name = "ViT-B/32"
    context, vocab, width, layers, heads, embed = TEXT_CONFIGS[name]
    sd = random_text_state_dict(name)
    m = OracleCLIPText(name, state_dict=sd)
    # eos_token_id = 2 selects the argmax pooling of OpenAI's checkpoints
    hf = CLIPTextModelWithProjection(CLIPTextConfig(vocab_size=vocab, hidden_size=width, intermediate_size=4 * width, projection_dim=embed,
                                                    num_hidden_layers=layers, num_attention_heads=heads, max_position_embeddings=context,
                                                    hidden_act="quick_gelu", attention_dropout=0.0, eos_token_id=2)).eval()
    hs = {"text_model.embeddings.token_embedding.weight": sd["token_embedding.weight"],
          "text_model.embeddings.position_embedding.weight": sd["positional_embedding"],
          "text_model.final_layer_norm.weight": sd["ln_final.weight"], "text_model.final_layer_norm.bias": sd["ln_final.bias"],
          "text_projection.weight": sd["text_projection"].t()}
    for i in range(layers):
        p, q = "transformer.resblocks.%d." % i, "text_model.encoder.layers.%d." % i
        w, b = sd[p + "attn.in_proj_weight"], sd[p + "attn.in_proj_bias"]
        for j, n in enumerate("qkv"):
            hs[q + "self_attn.%s_proj.weight" % n] = w[j * width:(j + 1) * width]
            hs[q + "self_attn.%s_proj.bias" % n] = b[j * width:(j + 1) * width]
        for a, c in (("self_attn.out_proj", "attn.out_proj"), ("layer_norm1", "ln_1"), ("layer_norm2", "ln_2"), ("mlp.fc1", "mlp.c_fc"), ("mlp.fc2", "mlp.c_proj")):
            hs[q + a + ".weight"], hs[q + a + ".bias"] = sd[p + c + ".weight"], sd[p + c + ".bias"]
    missing = hf.load_state_dict(hs, strict=False)
    assert not missing.unexpected_keys and all("position_ids" in k for k in missing.missing_keys)
    tokens = random_prompt_tokens([0, 5, 17, 40, context - 2], context, torch.Generator().manual_seed(0))
    with torch.no_grad():
        got, want = m.encode_text(tokens), hf(input_ids=tokens).text_embeds
    assert got.shape == (5, embed)
    assert (got - want).abs().max().item() <= 1e-5


@pytest.mark.parametrize("name", ["ViT-B/32", "ViT-B/16", "ViT-L/14", "ViT-L/14@336px"])
def test_text_state_dict_helpers_match_the_oracle(name):
    from clip_diffusion_b200 import models
    from oracle.clip_text import OracleCLIPText, random_text_state_dict

    sd = models.random_clip_text_state_dict(name, seed=2)
    assert list(sd) == models.clip_text_state_dict_keys(name)
    shapes = models.clip_text_state_dict_shapes(name)
    assert all(tuple(sd[k].shape) == shapes[k] for k in sd)
    ref = random_text_state_dict(name)
    assert sd.keys() == ref.keys() and all(sd[k].shape == ref[k].shape for k in sd)
    OracleCLIPText(name, state_dict=sd)  # strict load: same keys and shapes as OpenAI's module
    assert not any(k.startswith("visual.") for k in sd)


def _tiny_text_tower(name="text-tiny/32"):
    """A tiny registered vision tower with a tiny text tower under the same name (OpenAI's context length and vocabulary)."""
    from clip_diffusion_b200 import models

    models.register_clip_config(name, 64, 32, 128, 2, 2, 64)
    models.register_clip_text_config(name, 77, 49408, 128, 1, 2, 64)
    return name


def test_visual_only_checkpoint_loads_and_encode_text_names_the_missing_key(tmp_path, monkeypatch):
    from clip_diffusion_b200 import models

    name = _tiny_text_tower()
    monkeypatch.setenv("CLIPGUIDE_B200_WEIGHTS", str(tmp_path))
    torch.save(models.random_clip_state_dict(name), str(tmp_path / (name.replace("/", "_") + ".pt")))
    m = models.load_clip_models([name], "cpu")[name]
    tokens = torch.zeros(2, 77, dtype=torch.long)
    tokens[:, 0], tokens[:, 1] = 49406, 49407
    with pytest.raises(KeyError, match="token_embedding.weight"):
        m.encode_text(tokens)
    # a full checkpoint with one tensor of the wrong shape is refused too, also before any device work
    sd = dict(models.random_clip_state_dict(name), **models.random_clip_text_state_dict(name))
    sd["transformer.resblocks.0.mlp.c_fc.bias"] = torch.zeros(7)
    torch.save(sd, str(tmp_path / (name.replace("/", "_") + ".pt")))
    m = models.load_clip_models([name], "cpu")[name]
    with pytest.raises(ValueError, match="c_fc.bias"):
        m.encode_text(tokens)


def test_malformed_tokens_are_refused():
    from clip_diffusion_b200 import _lib, models

    name = _tiny_text_tower()
    m = models.CLIPModelB200(name, None, "cpu")
    good = torch.zeros(2, 77, dtype=torch.int32)
    good[:, 0], good[:, 1] = 49406, 49407
    bad = [good[0], good[:, :76], torch.zeros(2, 78, dtype=torch.int32), good.float(), good.bool(), good.unsqueeze(0)]
    for t in bad:
        with pytest.raises(ValueError):
            m.encode_text(t)
    for v in (-1, 49408):
        t = good.clone().long()
        t[1, 5] = v
        with pytest.raises(ValueError, match="token ids"):
            m.encode_text(t)
    with pytest.raises(_lib.ClipGuideError):  # well-formed, but a CPU tensor: no CPU fallback
        m.encode_text(good)
    assert m._text is None  # nothing was built


def test_causal_attention_refuses_long_sequences_before_any_cuda_call():
    from clip_diffusion_b200 import _lib

    lib = _lib.load()
    d = ctypes.c_void_p(16)
    assert lib.cg_attention_causal_fwd(d, 1, 273, 8, d, d, None) == -1
    assert b"272" in lib.cg_last_error()
    assert lib.cg_attention_causal_fwd(None, 1, 77, 8, d, d, None) == -1
    assert lib.cg_text_embed_fwd(d, d, d, 1, 77, 6, 49408, d, None) == -1
    assert lib.cg_text_pool_fwd(d, d, 0, 77, 512, d, d, d, None) == -1
