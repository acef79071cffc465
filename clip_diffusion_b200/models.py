"""CLIP towers for the guidance path, B200-native (mirror of clip_diffusion/models.py:33-84,188-240).

``load_clip_models(names, device)`` returns ``{name: model}`` where ``model`` exposes what the hot path
touches on an OpenAI ``clip`` model: ``model.visual.input_resolution`` (sample.py:167) and
``model.encode_image(image)`` (utils/functional.py:101).  The vision transformer itself -- which the
reference gets from the un-vendored ``clip`` package -- is implemented here on the C-ABI kernels:

  conv1 patch embed      tcgen05 GEMM, epilogue adds the positional embedding into the token rows
  LayerNorm              warp-per-row kernels, fp32 residual stream in, bf16 GEMM operand out
  QKV / out / MLP        tcgen05 GEMMs with fused bias / QuickGELU / residual epilogues
  attention              fused kernels (scores never leave the SM)
  backward               dgrad only: the towers are frozen (models.py:67-71), so every backward GEMM is
                         activation-gradient x pre-transposed weight, packed once at load

OpenAI's ModifiedResNet image tower (RN101, the fourth of Config.chosen_clip_models) runs on the same GEMM with ReLU-network
epilogues: NHWC bf16 activations, BatchNorm folded at load, 3x3 convolutions as im2col + GEMM, the attention pool on the ViT's
attention kernels.  It has the ViT tower's interface (patch 1: the cutout kernel's NHWC image), so the guidance step drives both alike.

``model.encode_text(tokens)`` (utils/functional.py:91-94, once per job) runs OpenAI's text transformer on the same kernels with
a causal attention forward; that tower is built on its first call.

There is no network here, so weights are constructor-style random init (SURVEY.md App. A.1) unless a
state dict in OpenAI's key naming is supplied.
"""
import math
import os

import torch
from torch import nn

from clip_diffusion_b200 import _lib
from clip_diffusion_b200.vit_ops import gemm_bf16_tn, gemm_bf16_tn_relu

# name: (input_resolution, patch, width, layers, heads, embed_dim)     E as in models.py:33-37
CLIP_CONFIGS = {
    "ViT-B/32": (224, 32, 768, 12, 12, 512),
    "ViT-B/16": (224, 16, 768, 12, 12, 512),
    "ViT-L/14": (224, 14, 1024, 24, 16, 768),
    "ViT-L/14@336px": (336, 14, 1024, 24, 16, 768),
}


# name: (context_length, vocab_size, width, layers, heads, embed_dim) of the text transformer (OpenAI clip/model.py build_model)
CLIP_TEXT_CONFIGS = {
    "ViT-B/32": (77, 49408, 512, 12, 8, 512),
    "ViT-B/16": (77, 49408, 512, 12, 8, 512),
    "ViT-L/14": (77, 49408, 768, 12, 12, 768),
    "ViT-L/14@336px": (77, 49408, 768, 12, 12, 768),
    "RN101": (77, 49408, 512, 12, 8, 512),
}

# name: (input_resolution, layers, width, heads, embed_dim) of OpenAI's ModifiedResNet (build_model infers them from the state dict)
CLIP_RESNET_CONFIGS = {
    "RN101": (224, (3, 4, 23, 3), 64, 32, 512),
}


# leaf names of one residual block's tensors ("<prefix><layer>.<leaf>"), in the order of OpenAI's state dict; the same in both towers
BLOCK_KEYS = ("attn.in_proj_weight", "attn.in_proj_bias", "attn.out_proj.weight", "attn.out_proj.bias", "mlp.c_fc.weight", "mlp.c_fc.bias",
              "mlp.c_proj.weight", "mlp.c_proj.bias", "ln_1.weight", "ln_1.bias", "ln_2.weight", "ln_2.bias")


def _block_keys(prefix, layers):
    return ["%s%d.%s" % (prefix, i, k) for i in range(layers) for k in BLOCK_KEYS]


def _check_width(width, heads):
    if width != heads * 64 or width % 128:  # head_dim 64; the GEMMs tile N by 128
        raise ValueError("width must equal heads*64 and be a multiple of 128")


def register_clip_config(name, input_resolution, patch, width, layers, heads, embed_dim):
    """Extra tower shapes (tests use tiny ones).  width must be heads*64 and a multiple of 128."""
    _check_width(width, heads)
    CLIP_CONFIGS[name] = (input_resolution, patch, width, layers, heads, embed_dim)


def register_clip_text_config(name, context, vocab, width, layers, heads, embed_dim):
    """Extra text-tower shapes (tests use tiny ones), same width constraints as register_clip_config; context <= _lib.ATTN_TC_MAX_T."""
    _check_width(width, heads)
    if not 0 < context <= _lib.ATTN_TC_MAX_T:
        raise ValueError("the context length must lie in [1, %d]" % _lib.ATTN_TC_MAX_T)
    CLIP_TEXT_CONFIGS[name] = (context, vocab, width, layers, heads, embed_dim)


def register_clip_resnet_config(name, input_resolution, layers, width, heads, embed_dim):
    """Extra ModifiedResNet shapes (tests use tiny ones).  The attention pool's width 32*width must equal heads*64; its T = (res/32)^2 + 1
    is at most _lib.ATTN_TC_MAX_T; embed_dim (the N of the c_proj GEMM) is a multiple of 128."""
    if len(layers) != 4 or min(layers) < 1 or input_resolution % 32 or width % 2:
        raise ValueError("a ModifiedResNet has four stages of >= 1 block, an input resolution divisible by 32 and an even width")
    if 32 * width != 64 * heads or embed_dim % 128 or (input_resolution // 32) ** 2 + 1 > _lib.ATTN_TC_MAX_T:
        raise ValueError("the attention pool needs 32*width == heads*64, embed_dim % 128 == 0 and (res/32)^2 + 1 <= %d" % _lib.ATTN_TC_MAX_T)
    CLIP_RESNET_CONFIGS[name] = (input_resolution, tuple(layers), width, heads, embed_dim)


def random_clip_state_dict(name, seed=1):
    """Random weights with the shapes/keys of OpenAI's ``visual.*`` state dict.  Linear/conv layers use
    PyTorch's default uniform(+-1/sqrt(fan_in)); embeddings and proj use width^-0.5 * randn (App. A.1);
    LayerNorm affine and attention biases are perturbed away from (1, 0) so that tests exercise them."""
    res, patch, width, layers, heads, embed = CLIP_CONFIGS[name]
    g = torch.Generator().manual_seed(seed)
    u = lambda *s, fan: (torch.rand(*s, generator=g) * 2 - 1) / math.sqrt(fan)
    n = lambda *s: torch.randn(*s, generator=g)
    sd = {
        "visual.conv1.weight": u(width, 3, patch, patch, fan=3 * patch * patch),
        "visual.class_embedding": width ** -0.5 * n(width),
        "visual.positional_embedding": width ** -0.5 * n((res // patch) ** 2 + 1, width),
        "visual.proj": width ** -0.5 * n(width, embed),
    }
    for ln in ("ln_pre", "ln_post"):
        sd["visual.%s.weight" % ln] = 1 + 0.1 * n(width)
        sd["visual.%s.bias" % ln] = 0.1 * n(width)
    for i in range(layers):
        p = "visual.transformer.resblocks.%d." % i
        sd[p + "attn.in_proj_weight"] = u(3 * width, width, fan=width) * math.sqrt(1.5)
        sd[p + "attn.in_proj_bias"] = 0.02 * n(3 * width)
        sd[p + "attn.out_proj.weight"] = u(width, width, fan=width)
        sd[p + "attn.out_proj.bias"] = 0.02 * n(width)
        sd[p + "mlp.c_fc.weight"] = u(4 * width, width, fan=width)
        sd[p + "mlp.c_fc.bias"] = u(4 * width, fan=width)
        sd[p + "mlp.c_proj.weight"] = u(width, 4 * width, fan=4 * width)
        sd[p + "mlp.c_proj.bias"] = u(width, fan=4 * width)
        for ln in ("ln_1", "ln_2"):
            sd[p + ln + ".weight"] = 1 + 0.1 * n(width)
            sd[p + ln + ".bias"] = 0.1 * n(width)
    return sd


def clip_text_state_dict_keys(name):
    """The text-tower keys of an OpenAI CLIP state dict (everything encode_text reads), in OpenAI's naming."""
    return list(clip_text_state_dict_shapes(name))


def clip_text_state_dict_shapes(name):
    """{key: shape} of the text tower from CLIP_TEXT_CONFIGS, in the order of OpenAI's state dict."""
    context, vocab, width, layers, heads, embed = CLIP_TEXT_CONFIGS[name]
    block = {"attn.in_proj_weight": (3 * width, width), "attn.in_proj_bias": (3 * width,), "attn.out_proj.weight": (width, width),
             "mlp.c_fc.weight": (4 * width, width), "mlp.c_fc.bias": (4 * width,), "mlp.c_proj.weight": (width, 4 * width)}
    shapes = {"token_embedding.weight": (vocab, width), "positional_embedding": (context, width)}
    # block keys are looked up by their leaf ("transformer.resblocks.<i>.<leaf>"); every other block tensor is [width]
    shapes.update((k, block.get(k.split(".", 3)[-1], (width,))) for k in _block_keys("transformer.resblocks.", layers))
    shapes.update({"ln_final.weight": (width,), "ln_final.bias": (width,), "text_projection": (width, embed)})
    return shapes


def random_clip_text_state_dict(name, seed=1):
    """Random weights with the keys and shapes of OpenAI's text tower.  Standard deviations follow OpenAI's
    ``CLIP.initialize_parameters`` (token 0.02, positional 0.01, attention width^-0.5, out / c_proj width^-0.5 (2 layers)^-0.5,
    c_fc (2 width)^-0.5, projection width^-0.5); LayerNorm affines and biases are perturbed as in random_clip_state_dict."""
    context, vocab, width, layers, heads, embed = CLIP_TEXT_CONFIGS[name]
    g = torch.Generator().manual_seed(seed)
    u = lambda *s, fan: (torch.rand(*s, generator=g) * 2 - 1) / math.sqrt(fan)
    n = lambda *s: torch.randn(*s, generator=g)
    attn_std, proj_std, fc_std = width ** -0.5, width ** -0.5 * (2 * layers) ** -0.5, (2 * width) ** -0.5
    sd = {"token_embedding.weight": 0.02 * n(vocab, width), "positional_embedding": 0.01 * n(context, width)}
    for i in range(layers):
        p = "transformer.resblocks.%d." % i
        sd[p + "attn.in_proj_weight"] = attn_std * n(3 * width, width)
        sd[p + "attn.in_proj_bias"] = 0.02 * n(3 * width)
        sd[p + "attn.out_proj.weight"] = proj_std * n(width, width)
        sd[p + "attn.out_proj.bias"] = 0.02 * n(width)
        sd[p + "mlp.c_fc.weight"] = fc_std * n(4 * width, width)
        sd[p + "mlp.c_fc.bias"] = u(4 * width, fan=width)
        sd[p + "mlp.c_proj.weight"] = proj_std * n(width, 4 * width)
        sd[p + "mlp.c_proj.bias"] = u(width, fan=4 * width)
        for ln in ("ln_1", "ln_2"):
            sd[p + ln + ".weight"] = 1 + 0.1 * n(width)
            sd[p + ln + ".bias"] = 0.1 * n(width)
    sd["ln_final.weight"] = 1 + 0.1 * n(width)
    sd["ln_final.bias"] = 0.1 * n(width)
    sd["text_projection"] = width ** -0.5 * n(width, embed)
    return sd


def _bf16(t, device):
    return t.to(device=device, dtype=torch.bfloat16).contiguous()


def _f32(t, device):
    return t.to(device=device, dtype=torch.float32).contiguous()


def _pack_blocks(sd, prefix, layers, device, transposed):
    """The residual blocks of a state dict under ``prefix``, on the device: each W [N, K] bf16 as the GEMMs' B operand, with
    ``transposed`` also W^T as the B operand of the dgrad GEMMs; biases and LayerNorm affines fp32."""
    blocks = []
    for i in range(layers):
        p = "%s%d." % (prefix, i)
        blk = {"ln1": (_f32(sd[p + "ln_1.weight"], device), _f32(sd[p + "ln_1.bias"], device)),
               "ln2": (_f32(sd[p + "ln_2.weight"], device), _f32(sd[p + "ln_2.bias"], device))}
        for key, w, b in (("qkv", "attn.in_proj_weight", "attn.in_proj_bias"), ("out", "attn.out_proj.weight", "attn.out_proj.bias"),
                          ("fc", "mlp.c_fc.weight", "mlp.c_fc.bias"), ("proj", "mlp.c_proj.weight", "mlp.c_proj.bias")):
            blk["w_" + key], blk["b_" + key] = _bf16(sd[p + w], device), _f32(sd[p + b], device)
            if transposed:
                blk["w_" + key + "_t"] = _bf16(sd[p + w].t(), device)
        blocks.append(blk)
    return blocks


def _block_forward(attention, blk, n, T, heads, x, out, L, h, hg):
    """One residual block on fp32 [n*T, D] residual streams, x -> out (may be x), with ``attention`` the C-ABI entry point
    (cg_attention_fwd or cg_attention_causal_fwd).  ``L`` receives the activations the vision backward reads; h, hg are bf16 scratch."""
    M, D = n * T, x.shape[1]
    P, C = _lib.ptr, _lib.call
    C("cg_layernorm_fwd", P(x), P(blk["ln1"][0]), P(blk["ln1"][1]), M, D, D, P(h), None, P(L["mean1"]), P(L["rstd1"]))
    gemm_bf16_tn(h, blk["w_qkv"], _lib.EPI_BIAS_BF16, bias=blk["b_qkv"], out=L["qkv"])
    C(attention, P(L["qkv"]), n, T, heads, P(L["ctx"]), P(L["lse"]))
    gemm_bf16_tn(L["ctx"], blk["w_out"], _lib.EPI_BIAS_RESID_F32, bias=blk["b_out"], out=L["x_mid"], aux=x)
    C("cg_layernorm_fwd", P(L["x_mid"]), P(blk["ln2"][0]), P(blk["ln2"][1]), M, D, D, P(h), None, P(L["mean2"]), P(L["rstd2"]))
    gemm_bf16_tn(h, blk["w_fc"], _lib.EPI_BIAS_QGELU_BF16, bias=blk["b_fc"], out=hg, aux=L["u"])
    gemm_bf16_tn(hg, blk["w_proj"], _lib.EPI_BIAS_RESID_F32, bias=blk["b_proj"], out=out, aux=L["x_mid"])


class _GraphTower:
    """What the image towers share: the interface the guidance step and _EncodeImageFn use (input_resolution, patch, kpad, grid,
    output_dim, forward_patches, backward_patches), per-batch-size workspaces with stable addresses, the generation id that makes a
    stale backward an error, and CUDA-graph passes.  A subclass sets those attributes and provides _new_workspace(n) (its activation
    buffers), _forward_body(ws, n) (patches -> emb) and _backward_body(ws, n) (demb -> dpatch)."""

    def _init_graph_tower(self):
        self._ws = {}  # persistent activation workspaces per batch size (stable addresses => TMA descriptor cache hits)
        self._generation = 0  # bumped by every forward: the saved activations live in the shared workspace, not in an autograd ctx
        # CUDA graphs: a tower pass is ~7 C-ABI calls per layer and direction on fixed buffers; issuing them one by one costs the host
        # ~12 ms per step for ViT-L/14 (measured: bench.py `host_enqueue_ms_per_step`), which bounds the small configurations and the
        # end-to-end step.  The first pass of a batch size runs eagerly (function attributes, descriptor cache, scratch allocation), the
        # second is captured, later ones are replayed.  use_graphs = False keeps every pass eager.
        self.use_graphs = True

    # ------------------------------------------------------------------ workspaces
    def _workspace(self, n):
        ws = self._ws.get(n)
        if ws is not None:
            return ws
        dev = self.device
        ws = self._new_workspace(n)
        # static input / output buffers of the (graph-replayable) passes
        ws.update({
            "patches": torch.empty(n, self.grid ** 2, self.kpad, device=dev, dtype=torch.bfloat16),
            "emb": torch.empty(n, self.output_dim, device=dev, dtype=torch.float32),
            "demb": torch.empty(n, self.output_dim, device=dev, dtype=torch.float32),
            "dpatch": torch.empty(n, self.grid ** 2, self.kpad, device=dev, dtype=torch.float32),
            "graphs": {},
        })
        if len(self._ws) >= 4:  # bound the footprint when batch sizes keep changing (cut schedules)
            self._ws.pop(next(iter(self._ws)))
        self._ws[n] = ws
        return ws

    # ------------------------------------------------------------------ forward
    def forward_patches(self, patches):
        """patches: [N, g*g, Kpad] bf16 im2col rows of the (CLIP-normalised) images -> embeddings [N, E] fp32."""
        n = patches.shape[0]
        g2 = self.grid ** 2
        if patches.shape[1] != g2 or patches.shape[2] != self.kpad or patches.dtype != torch.bfloat16:
            raise ValueError("expected bf16 patches of shape [N, %d, %d], got %s %s" % (g2, self.kpad, tuple(patches.shape), patches.dtype))
        ws = self._workspace(n)
        if patches.data_ptr() != ws["patches"].data_ptr():
            ws["patches"].copy_(patches)
        self._run_pass(ws, "fwd", lambda: self._forward_body(ws, n))
        self._last_n = n
        self._generation += 1
        ws["generation"] = self._generation
        return ws["emb"].clone()

    def _run_pass(self, ws, key, body):
        """Run one tower pass on the workspace buffers: eagerly, or as a CUDA graph (first call eager, second captured, then replayed).
        Per-call profiling (bench.py's kernel rooflines) needs the individual launches, so it forces the eager path."""
        if not self.use_graphs or _lib.PROFILE is not None:
            body()
            return
        st = ws["graphs"].setdefault(key, {"calls": 0, "graph": None, "launches": 0, "failed": False})
        if st["failed"]:
            body()
            return
        if st["graph"] is None:
            st["calls"] += 1
            if st["calls"] == 1:
                body()
                return
            k0, c0 = _lib.kernel_launches, _lib.launch_count
            graph = torch.cuda.CUDAGraph()
            try:
                # thread_local: other threads (NCCL watchdog, data loaders) may touch the CUDA API while this thread captures
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    body()
            except Exception as exc:  # keep the product path alive, loudly: the eager launches are the same kernels
                import warnings
                st["failed"] = True
                warnings.warn("CUDA graph capture of the %s %s pass failed (%s); this tower keeps issuing its kernels one by one" % (self.name, key, exc))
                torch.cuda.synchronize()
                body()
                return
            st["graph"], st["launches"], st["calls_per_pass"] = graph, _lib.kernel_launches - k0, _lib.launch_count - c0
            _lib.kernel_launches, _lib.launch_count = k0, c0  # capturing launched nothing; the replay below counts
        st["graph"].replay()
        _lib.kernel_launches += st["launches"]
        _lib.launch_count += st["calls_per_pass"]

    # ------------------------------------------------------------------ backward (input gradient only)
    def backward_patches(self, demb, generation=None):
        """demb [N, E] fp32 -> d(patches) [N, g*g, Kpad] fp32, for the activations of the latest forward.  The saved activations
        live in the tower's per-batch-size workspace, which the next forward of the same size overwrites: ``generation`` (the
        value of ``self._generation`` right after the forward this gradient belongs to) makes a stale backward an error instead
        of a silently wrong gradient."""
        n = demb.shape[0]
        ws = self._ws.get(n)
        if ws is None or "generation" not in ws:
            raise RuntimeError("backward_patches must follow forward_patches with the same batch size")
        if generation is None:
            if n != getattr(self, "_last_n", None):
                raise RuntimeError("backward_patches must follow forward_patches with the same batch size")
        elif ws["generation"] != generation:
            raise RuntimeError(
                "stale CLIP activations: another encode_image/forward_patches call with batch size %d ran on this tower between this "
                "forward (generation %d) and its backward (workspace now holds generation %d).  The tower keeps ONE set of saved "
                "activations per batch size; differentiate each embedding batch before embedding the next one of the same size "
                "(sample.py:199-214 does exactly that)." % (n, generation, ws["generation"]))
        ws["demb"].copy_(demb)
        self._run_pass(ws, "bwd", lambda: self._backward_body(ws, n))
        # the gradient buffer belongs to the workspace: consume it before the next backward of the same batch size (sample.py does)
        return ws["dpatch"]


class VisionTransformerB200(_GraphTower):
    """Frozen OpenAI-style CLIP vision transformer: forward + input-gradient backward on sm_100a kernels."""

    def __init__(self, name, state_dict, device):
        res, patch, width, layers, heads, embed = CLIP_CONFIGS[name]
        self.name = name
        self.input_resolution, self.patch, self.width, self.layers, self.heads, self.output_dim = res, patch, width, layers, heads, embed
        self.grid = res // patch
        self.tokens = self.grid ** 2 + 1
        self.kdim = 3 * patch * patch
        self.kpad = (self.kdim + 127) // 128 * 128  # K of the patch GEMM (x64) and N of its dgrad (x128)
        self.device = torch.device(device)
        sd, dev = state_dict, self.device
        w = sd["visual.conv1.weight"].reshape(width, self.kdim)
        wpad = torch.zeros(width, self.kpad)
        wpad[:, : self.kdim] = w
        self.w_patch = _bf16(wpad, dev)          # [D, Kpad]   fwd  B operand
        self.w_patch_t = _bf16(wpad.t(), dev)    # [Kpad, D]   dgrad B operand
        self.cls = _f32(sd["visual.class_embedding"], dev)
        self.pos = _f32(sd["visual.positional_embedding"], dev)
        self.ln_pre = (_f32(sd["visual.ln_pre.weight"], dev), _f32(sd["visual.ln_pre.bias"], dev))
        self.ln_post = (_f32(sd["visual.ln_post.weight"], dev), _f32(sd["visual.ln_post.bias"], dev))
        self.proj = _f32(sd["visual.proj"], dev)
        self.blocks = _pack_blocks(sd, "visual.transformer.resblocks.", layers, dev, transposed=True)
        self._init_graph_tower()

    def _new_workspace(self, n):
        dev, D, T, M = self.device, self.width, self.tokens, n * self.tokens
        f32 = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
        b16 = lambda *s: torch.empty(*s, device=dev, dtype=torch.bfloat16)
        return {
            "x0": f32(M, D), "mean0": f32(M), "rstd0": f32(M),
            "h": b16(M, D), "hg": b16(M, 4 * D),
            "layers": [
                {"x_in": f32(M, D), "mean1": f32(M), "rstd1": f32(M), "qkv": b16(M, 3 * D), "ctx": b16(M, D), "lse": f32(n, self.heads, T),
                 "x_mid": f32(M, D), "mean2": f32(M), "rstd2": f32(M), "u": b16(M, 4 * D)}
                for _ in range(self.layers)
            ],
            "x_out": f32(M, D), "meanp": f32(n), "rstdp": f32(n), "y": f32(n, D),
            # backward
            "dx": f32(M, D), "dxb": b16(M, D), "dy": f32(n, D), "du": b16(M, 4 * D), "dh": f32(M, D), "dctx": b16(M, D),
            "dqkv": b16(M, 3 * D), "delta": f32(n, self.heads, T), "dx0": f32(M, D), "dtok": b16(n * (T - 1), D),
        }

    def _forward_body(self, ws, n):
        g2, D, T, E = self.grid ** 2, self.width, self.tokens, self.output_dim
        M = n * T
        P, C = _lib.ptr, _lib.call
        a = ws["patches"].view(n * g2, self.kpad)
        gemm_bf16_tn(a, self.w_patch, _lib.EPI_PATCH_POS_F32, out=ws["x0"], pos=self.pos, g2=g2)
        C("cg_vit_set_cls_rows", P(self.cls), P(self.pos), n, T, D, P(ws["x0"]))
        x = ws["layers"][0]["x_in"] if self.layers else ws["x_out"]
        C("cg_layernorm_fwd", P(ws["x0"]), P(self.ln_pre[0]), P(self.ln_pre[1]), M, D, D, None, P(x), P(ws["mean0"]), P(ws["rstd0"]))
        for i, (blk, L) in enumerate(zip(self.blocks, ws["layers"])):
            x_next = ws["layers"][i + 1]["x_in"] if i + 1 < self.layers else ws["x_out"]
            _block_forward("cg_attention_fwd", blk, n, T, self.heads, L["x_in"], x_next, L, ws["h"], ws["hg"])
        # ln_post on the class-token rows (row stride T*D), then the projection
        C("cg_layernorm_fwd", P(ws["x_out"]), P(self.ln_post[0]), P(self.ln_post[1]), n, D, T * D, None, P(ws["y"]), P(ws["meanp"]), P(ws["rstdp"]))
        C("cg_vit_proj_fwd", P(ws["y"]), P(self.proj), n, D, E, P(ws["emb"]))

    # ------------------------------------------------------------------ backward (input gradient only)
    def _backward_body(self, ws, n):
        g2, D, T, E = self.grid ** 2, self.width, self.tokens, self.output_dim
        M = n * T
        P, C = _lib.ptr, _lib.call
        C("cg_vit_proj_bwd", P(ws["demb"]), P(self.proj), n, D, E, P(ws["dy"]))
        ws["dx"].zero_()
        ws["dxb"].zero_()
        C("cg_layernorm_bwd", P(ws["dy"]), P(ws["x_out"]), P(self.ln_post[0]), P(ws["meanp"]), P(ws["rstdp"]), n, D, T * D, 0, P(ws["dx"]), P(ws["dxb"]))
        for blk, L in zip(reversed(self.blocks), reversed(ws["layers"])):
            gemm_bf16_tn(ws["dxb"], blk["w_proj_t"], _lib.EPI_DQGELU_BF16, out=ws["du"], aux=L["u"])
            gemm_bf16_tn(ws["du"], blk["w_fc_t"], _lib.EPI_F32, out=ws["dh"])
            C("cg_layernorm_bwd", P(ws["dh"]), P(L["x_mid"]), P(blk["ln2"][0]), P(L["mean2"]), P(L["rstd2"]), M, D, D, 1, P(ws["dx"]), P(ws["dxb"]))
            gemm_bf16_tn(ws["dxb"], blk["w_out_t"], _lib.EPI_BF16, out=ws["dctx"])
            C("cg_attention_bwd", P(L["qkv"]), P(L["ctx"]), P(ws["dctx"]), P(L["lse"]), n, T, self.heads, P(ws["dqkv"]), P(ws["delta"]))
            gemm_bf16_tn(ws["dqkv"], blk["w_qkv_t"], _lib.EPI_F32, out=ws["dh"])
            C("cg_layernorm_bwd", P(ws["dh"]), P(L["x_in"]), P(blk["ln1"][0]), P(L["mean1"]), P(L["rstd1"]), M, D, D, 1, P(ws["dx"]), P(ws["dxb"]))
        C("cg_layernorm_bwd", P(ws["dx"]), P(ws["x0"]), P(self.ln_pre[0]), P(ws["mean0"]), P(ws["rstd0"]), M, D, D, 0, P(ws["dx0"]), None)
        C("cg_vit_tokens_to_bf16", P(ws["dx0"]), n, T, D, 1, P(ws["dtok"]))
        # fp32 output: this is the last rounding before the image gradient (the bf16 variant cost ~1e-3 of rel-L2 margin)
        gemm_bf16_tn(ws["dtok"], self.w_patch_t, _lib.EPI_F32, out=ws["dpatch"].view(n * g2, self.kpad))

    def flops_fwd_bwd(self, n):
        """Algorithmic FLOPs (2 x MAC) of forward + dgrad for n images (SURVEY.md section 8(d))."""
        T, D, L, E = self.tokens, self.width, self.layers, self.output_dim
        patch = 2 * (T - 1) * self.kdim * D + 2 * D * E
        fwd = 24 * T * D * D * L + 4 * T * T * D * L + patch
        bwd = 24 * T * D * D * L + 8 * T * T * D * L + patch
        return n * (fwd + bwd)


# ---------------------------------------------------------------------------------------------------------------------- ModifiedResNet
_BN_LEAVES = ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")
BN_EPS = 1e-5


def _resnet_blocks(name):
    """(prefix, inplanes, planes, stride, downsample) of every Bottleneck, in order (OpenAI ModifiedResNet._make_layer)."""
    _, layers, width, _, _ = CLIP_RESNET_CONFIGS[name]
    blocks, inplanes = [], width
    for li, nb in enumerate(layers):
        planes, stride = width * 2 ** li, 1 if li == 0 else 2
        for i in range(nb):
            s = stride if i == 0 else 1
            blocks.append(("visual.layer%d.%d." % (li + 1, i), inplanes, planes, s, s > 1 or inplanes != 4 * planes))
            inplanes = 4 * planes
    return blocks


def clip_resnet_state_dict_shapes(name):
    """{key: shape} of the ``visual.*`` tensors of an OpenAI ModifiedResNet CLIP, in the order of OpenAI's state dict."""
    res, _, width, _, embed = CLIP_RESNET_CONFIGS[name]
    shapes = {}

    def conv_bn(conv, bn, cout, cin, k):
        shapes[conv + ".weight"] = (cout, cin, k, k)
        shapes.update((bn + "." + leaf, () if leaf == "num_batches_tracked" else (cout,)) for leaf in _BN_LEAVES)

    for i, (cout, cin) in enumerate(((width // 2, 3), (width // 2, width // 2), (width, width // 2))):
        conv_bn("visual.conv%d" % (i + 1), "visual.bn%d" % (i + 1), cout, cin, 3)
    for p, cin, planes, _, ds in _resnet_blocks(name):
        conv_bn(p + "conv1", p + "bn1", planes, cin, 1)
        conv_bn(p + "conv2", p + "bn2", planes, planes, 3)
        conv_bn(p + "conv3", p + "bn3", 4 * planes, planes, 1)
        if ds:
            conv_bn(p + "downsample.0", p + "downsample.1", 4 * planes, cin, 1)
    C = 32 * width
    shapes["visual.attnpool.positional_embedding"] = ((res // 32) ** 2 + 1, C)
    for proj in ("k_proj", "q_proj", "v_proj"):
        shapes["visual.attnpool.%s.weight" % proj], shapes["visual.attnpool.%s.bias" % proj] = (C, C), (C,)
    shapes["visual.attnpool.c_proj.weight"], shapes["visual.attnpool.c_proj.bias"] = (embed, C), (embed,)
    return shapes


def random_clip_resnet_state_dict(name, seed=1):
    """Random weights with the keys and shapes of OpenAI's ModifiedResNet ``visual.*`` tensors, chosen so that signal crosses every
    block: He-scaled convolutions, BatchNorm statistics and affines perturbed away from the identity, and a small bn3 gamma (~0.25)
    so that each Bottleneck's branch adds to its identity without swamping it (OpenAI's zero bn3 gamma would make every block an
    identity).  The attention pool follows OpenAI's initialize_parameters (std C^-1/2), with biases perturbed away from 0."""
    g = torch.Generator().manual_seed(seed)
    n = lambda *s: torch.randn(*s, generator=g)
    sd = {}
    for k, shape in clip_resnet_state_dict_shapes(name).items():
        leaf = k.rsplit(".", 1)[-1]
        bn3 = ".bn3." in k
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.tensor(0, dtype=torch.long)
        elif k.startswith("visual.attnpool."):
            C = shape[-1]
            sd[k] = C ** -0.5 * n(*shape) if leaf in ("weight", "positional_embedding") else 0.02 * n(*shape)
        elif len(shape) == 4:
            sd[k] = math.sqrt(2.0 / (shape[1] * shape[2] * shape[3])) * n(*shape)
        elif leaf == "weight":
            sd[k] = (0.25 if bn3 else 1.0) * (1 + 0.1 * n(*shape))
        elif leaf == "bias":
            sd[k] = (0.025 if bn3 else 0.1) * n(*shape)
        elif leaf == "running_mean":
            sd[k] = 0.1 * n(*shape)
        else:
            sd[k] = 1 + 0.2 * torch.rand(*shape, generator=g)
    return sd


def fold_batchnorm(weight, bn_weight, bn_bias, running_mean, running_var, eps=BN_EPS):
    """conv (no bias) followed by eval-mode BatchNorm as one convolution with bias, in float64:
    w' = w gamma / sqrt(var + eps), b' = beta - mean gamma / sqrt(var + eps)."""
    s = bn_weight.double() / torch.sqrt(running_var.double() + eps)
    return weight.double() * s.view(-1, *([1] * (weight.dim() - 1))), bn_bias.double() - running_mean.double() * s


def _r128(c):
    return (c + 127) // 128 * 128


def _r64(c):
    return (c + 63) // 64 * 64


def _padded(w, rows, cols):
    out = torch.zeros(rows, cols, dtype=w.dtype)
    out[: w.shape[0], : w.shape[1]] = w
    return out


def _resnet_device(device):
    device = torch.device(device)
    if device.type != "cuda":
        raise ValueError("the ModifiedResNet CLIP tower runs on a CUDA device only (got %s): it has no CPU path" % device)
    return device


class _Conv:
    """One convolution with its BatchNorm folded in, packed at load as the B operands of its GEMMs (bf16, channel counts padded:
    N to 128, K to 64, with zero rows / columns): ``w`` [cout', K] for the forward, ``b`` [cout'] fp32 its folded bias, ``wt`` the
    input gradient's operand -- W^T [cin', K(cout)] for a 1x1 convolution, the flipped W'[cin', (ky, kx, cout)] for a 3x3 one."""

    def __init__(self, sd, conv, bn, device, dgrad=True):
        w, b = fold_batchnorm(sd[conv + ".weight"], *(sd[bn + "." + leaf] for leaf in _BN_LEAVES[:4]))
        w = w.to(torch.bfloat16).double()  # the one rounding of the folded weights; every operand below is exact in bf16
        self.cout, self.cin, k = w.shape[0], w.shape[1], w.shape[2]
        self.k = _r64(k * k * self.cin)  # GEMM K of the forward
        self.w = _bf16(_padded(w.permute(0, 2, 3, 1).reshape(self.cout, -1), _r128(self.cout), self.k), device)
        self.b = _f32(_padded(b.view(-1, 1), _r128(self.cout), 1).view(-1), device)
        self.kt = _r64(k * k * self.cout)  # GEMM K of the input gradient
        if dgrad and k == 1:
            self.wt = _bf16(_padded(w.view(self.cout, self.cin).t(), _r128(self.cin), self.kt), device)
        elif dgrad:
            self.wt = _bf16(_padded(w.flip(2, 3).permute(1, 2, 3, 0).reshape(self.cin, -1), _r128(self.cin), self.kt), device)
        self.w_f32 = w  # host copy (the stem's stride-2 dgrad reads it as fp32)


class ModifiedResNetB200(_GraphTower):
    """Frozen OpenAI CLIP ModifiedResNet (the RN image towers): forward + input-gradient backward on sm_100a kernels.  Activations are
    NHWC bf16 rows with channel counts padded to 128 (zero channels); BatchNorm is folded into the convolutions; each 3x3 convolution is
    cg_im2col3x3_nhwc + a GEMM, the ReLUs, residuals and ReLU derivatives live in the GEMM epilogues.  The gradient's residual stream
    is fp32 with a bf16 copy as the next GEMM's operand.  Its input is the cutout kernel's NHWC image: patch 1, kpad 8 (3 channels)."""

    def __init__(self, name, state_dict, device):
        res, layers, width, heads, embed = CLIP_RESNET_CONFIGS[name]
        self.device = _resnet_device(device)
        self.name = name
        self.input_resolution, self.layers, self.width, self.heads, self.output_dim = res, layers, width, heads, embed
        self.patch, self.kpad, self.grid = 1, 8, res
        self.embed_width = 32 * width  # the attention pool's C
        self.spatial = res // 32
        self.tokens = self.spatial ** 2 + 1
        sd, dev = state_dict, self.device
        self.stem = [_Conv(sd, "visual.conv%d" % i, "visual.bn%d" % i, dev, dgrad=i > 1) for i in (1, 2, 3)]
        self.w_stem1_f32 = _f32(self.stem[0].w_f32, dev)  # [width/2, 3, 3, 3]
        self.blocks = []
        for p, cin, planes, stride, ds in _resnet_blocks(name):
            blk = {"cin": cin, "planes": planes, "stride": stride,
                   "c1": _Conv(sd, p + "conv1", p + "bn1", dev), "c2": _Conv(sd, p + "conv2", p + "bn2", dev),
                   "c3": _Conv(sd, p + "conv3", p + "bn3", dev), "ds": _Conv(sd, p + "downsample.0", p + "downsample.1", dev) if ds else None}
            self.blocks.append(blk)
        a = "visual.attnpool."
        C = self.embed_width
        self.pos = _f32(sd[a + "positional_embedding"], dev)
        w_qkv = torch.cat([sd[a + "q_proj.weight"], sd[a + "k_proj.weight"], sd[a + "v_proj.weight"]])
        self.w_qkv, self.w_qkv_t = _bf16(w_qkv, dev), _bf16(w_qkv.t(), dev)  # [3C, C], [C, 3C]
        self.b_qkv = _f32(torch.cat([sd[a + "q_proj.bias"], sd[a + "k_proj.bias"], sd[a + "v_proj.bias"]]), dev)
        self.w_c = _bf16(sd[a + "c_proj.weight"], dev)  # [E, C]
        self.w_c_t = _f32(sd[a + "c_proj.weight"].t(), dev)  # [C, E] fp32 (cg_vit_proj_bwd's proj)
        self.b_c = _f32(sd[a + "c_proj.bias"], dev)
        assert C == heads * 64
        self._init_graph_tower()

    def _geometry(self):
        """Per block: (spatial size of its input, of its output)."""
        h = self.input_resolution // 4
        out = []
        for blk in self.blocks:
            out.append((h, h // blk["stride"]))
            h //= blk["stride"]
        return out

    def _new_workspace(self, n):
        dev = self.device
        b16 = lambda *s: torch.empty(*s, device=dev, dtype=torch.bfloat16)
        f32 = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
        h1 = self.input_resolution // 2
        M1 = n * h1 * h1
        ws = {"stem": [b16(M1, c.w.shape[0]) for c in self.stem], "x0": b16(n * (h1 // 2) ** 2, self.stem[2].w.shape[0]), "blocks": []}
        col = M1 * max([c.k for c in self.stem] + [c.kt for c in self.stem[1:]])  # im2col rows: the largest of every 3x3 convolution
        grads = {}  # fp32 gradient and its bf16 copy per activation shape; a block without downsample updates its gradient in place
        scratch = 0
        for blk, (hi, ho) in zip(self.blocks, self._geometry()):
            Mi, Mo = n * hi * hi, n * ho * ho
            c1, c2, c3 = blk["c1"], blk["c2"], blk["c3"]
            ws["blocks"].append({"a1": b16(Mi, c1.w.shape[0]), "a2": b16(Mi, c2.w.shape[0]), "y": b16(Mo, c3.w.shape[0])})
            col = max(col, Mi * c2.k, Mi * c2.kt)
            scratch = max(scratch, Mo * c2.w.shape[0], Mo * _r128(blk["cin"]), Mo * c3.w.shape[0], Mi * c2.w.shape[0])
            for rows, cols in ((Mo, c3.w.shape[0]), (Mi, _r128(blk["cin"]))):
                if (rows, cols) not in grads:
                    grads[(rows, cols)] = (f32(rows, cols), b16(rows, cols))
        ws["grads"] = grads
        ws["col"] = b16(col)
        # bf16 scratch of the block: pooled a2 / pooled x / the downsample's output (forward), d(pooled a2) (backward)
        ws["s_pa2"], ws["s_px"], ws["s_idn"] = b16(scratch), b16(scratch), b16(scratch)
        ws["s_dz"] = b16(scratch)
        ws["s_dpx"] = f32(scratch)
        C, T = self.embed_width, self.tokens
        ws.update({"tok": b16(n * T, C), "qkv": b16(n * T, 3 * C), "ctx": b16(n * T, C), "lse": f32(n, self.heads, T),
                   "dy": f32(n, C), "dctx": b16(n * T, C), "dqkv": b16(n * T, 3 * C), "delta": f32(n, self.heads, T), "dtok": f32(n * T, C)})
        ws["dz_stem"] = [b16(M1, c.w.shape[0]) for c in self.stem]
        return ws

    @staticmethod
    def _view(buf, rows, cols):
        return buf[: rows * cols].view(rows, cols)

    def _im2col(self, ws, x, n, h, C, stride, kpad):
        P = _lib.ptr
        ho = (h - 1) // stride + 1
        col = self._view(ws["col"], n * ho * ho, kpad)
        _lib.call("cg_im2col3x3_nhwc", P(x), n, h, h, C, x.stride(0), stride, kpad, P(col))
        return col

    def _forward_body(self, ws, n):
        P, C_ = _lib.ptr, _lib.call
        relu = gemm_bf16_tn_relu
        R = self.input_resolution
        h1 = R // 2
        x = ws["patches"].view(n * R * R, self.kpad)
        s1, s2, s3 = ws["stem"]
        c1, c2, c3 = self.stem
        relu(self._im2col(ws, x, n, R, 3, 2, c1.k), c1.w, _lib.EPI_BIAS_RELU_BF16, bias=c1.b, out=s1)
        relu(self._im2col(ws, s1, n, h1, c2.cin, 1, c2.k), c2.w, _lib.EPI_BIAS_RELU_BF16, bias=c2.b, out=s2)
        relu(self._im2col(ws, s2, n, h1, c3.cin, 1, c3.k), c3.w, _lib.EPI_BIAS_RELU_BF16, bias=c3.b, out=s3)
        C_("cg_avgpool2x2_nhwc_fwd", P(s3), n, h1, h1, s3.shape[1], P(ws["x0"]))
        x = ws["x0"]
        for blk, L, (hi, ho) in zip(self.blocks, ws["blocks"], self._geometry()):
            b1, b2, b3, ds = blk["c1"], blk["c2"], blk["c3"], blk["ds"]
            relu(x[:, : b1.k], b1.w, _lib.EPI_BIAS_RELU_BF16, bias=b1.b, out=L["a1"])
            relu(self._im2col(ws, L["a1"], n, hi, b2.cin, 1, b2.k), b2.w, _lib.EPI_BIAS_RELU_BF16, bias=b2.b, out=L["a2"])
            pa2 = L["a2"]
            if blk["stride"] > 1:
                pa2 = self._view(ws["s_pa2"], n * ho * ho, L["a2"].shape[1])
                C_("cg_avgpool2x2_nhwc_fwd", P(L["a2"]), n, hi, hi, pa2.shape[1], P(pa2))
            idn = x
            if ds is not None:
                px = x
                if blk["stride"] > 1:
                    px = self._view(ws["s_px"], n * ho * ho, x.shape[1])
                    C_("cg_avgpool2x2_nhwc_fwd", P(x), n, hi, hi, x.shape[1], P(px))
                idn = self._view(ws["s_idn"], n * ho * ho, ds.w.shape[0])
                gemm_bf16_tn(px[:, : ds.k], ds.w, _lib.EPI_BIAS_BF16, bias=ds.b, out=idn)
            relu(pa2[:, : b3.k], b3.w, _lib.EPI_BIAS_RESID_RELU_BF16, bias=b3.b, resid=idn, out=L["y"])
            x = L["y"]
        # attention pool: tokens -> packed q|k|v -> attention -> c_proj of the query row 0 of every image
        C, T = self.embed_width, self.tokens
        C_("cg_resnet_attnpool_fwd", P(x), P(self.pos), n, T - 1, C, P(ws["tok"]))
        gemm_bf16_tn(ws["tok"], self.w_qkv, _lib.EPI_BIAS_BF16, bias=self.b_qkv, out=ws["qkv"])
        C_("cg_attention_fwd", P(ws["qkv"]), n, T, self.heads, P(ws["ctx"]), P(ws["lse"]))
        ws["emb"].zero_()
        gemm_bf16_tn(ws["ctx"].view(n, T * C)[:, :C], self.w_c, _lib.EPI_BIAS_RESID_F32, bias=self.b_c, out=ws["emb"], aux=ws["emb"])

    def _backward_body(self, ws, n):
        P, C_ = _lib.ptr, _lib.call
        relu = gemm_bf16_tn_relu
        C, T, E = self.embed_width, self.tokens, self.output_dim
        C_("cg_vit_proj_bwd", P(ws["demb"]), P(self.w_c_t), n, C, E, P(ws["dy"]))
        C_("cg_resnet_attnpool_dctx", P(ws["dy"]), n, T, C, P(ws["dctx"]))
        C_("cg_attention_bwd", P(ws["qkv"]), P(ws["ctx"]), P(ws["dctx"]), P(ws["lse"]), n, T, self.heads, P(ws["dqkv"]), P(ws["delta"]))
        gemm_bf16_tn(ws["dqkv"], self.w_qkv_t, _lib.EPI_F32, out=ws["dtok"])
        y_last = ws["blocks"][-1]["y"]
        g32, g16 = ws["grads"][tuple(y_last.shape)]
        C_("cg_resnet_attnpool_bwd", P(ws["dtok"]), P(y_last), n, T - 1, C, P(g32), P(g16))
        geo = self._geometry()
        for i in reversed(range(len(self.blocks))):
            blk, L, (hi, ho) = self.blocks[i], ws["blocks"][i], geo[i]
            b1, b2, b3, ds = blk["c1"], blk["c2"], blk["c3"], blk["ds"]
            x_in = ws["blocks"][i - 1]["y"] if i else ws["x0"]
            g32_in, g16_in = ws["grads"][(x_in.shape[0], x_in.shape[1])]
            # conv3 (1x1) dgrad; through the pool into a2's ReLU
            if blk["stride"] > 1:
                dp = self._view(ws["s_dz"], n * ho * ho, L["a2"].shape[1])
                gemm_bf16_tn(g16[:, : b3.kt], b3.wt, _lib.EPI_BF16, out=dp)
                dz2 = self._view(ws["s_pa2"], n * hi * hi, L["a2"].shape[1])
                C_("cg_avgpool2x2_nhwc_bwd", P(dp), 0, P(L["a2"]), n, hi, hi, dz2.shape[1], P(dz2), 0)
            else:
                dz2 = self._view(ws["s_pa2"], n * hi * hi, L["a2"].shape[1])
                relu(g16[:, : b3.kt], b3.wt, _lib.EPI_DRELU_BF16, mask=L["a2"], out=dz2)
            # conv2 (3x3) dgrad as a convolution of dz2 with the flipped weights, into a1's ReLU
            dz1 = self._view(ws["s_dz"], n * hi * hi, L["a1"].shape[1])
            relu(self._im2col(ws, dz2, n, hi, b2.cout, 1, b2.kt), b2.wt, _lib.EPI_DRELU_BF16, mask=L["a1"], out=dz1)
            # the identity path's gradient (in place when the block has no downsample), then conv1's dgrad joins it
            if ds is not None:
                if blk["stride"] > 1:
                    dpx = self._view(ws["s_dpx"], n * ho * ho, g32_in.shape[1])
                    gemm_bf16_tn(g16[:, : ds.kt], ds.wt, _lib.EPI_F32, out=dpx)
                    C_("cg_avgpool2x2_nhwc_bwd", P(dpx), 1, None, n, hi, hi, dpx.shape[1], P(g32_in), 1)
                else:
                    gemm_bf16_tn(g16[:, : ds.kt], ds.wt, _lib.EPI_F32, out=g32_in)
            relu(dz1[:, : b1.kt], b1.wt, _lib.EPI_RESID_DRELU, resid=g32_in, mask=x_in if i else None, out=g32_in, out_bf16=g16_in)
            g32, g16 = g32_in, g16_in
        # stem: the pool, then conv3 and conv2 (3x3, stride 1) as flipped convolutions, conv1 (stride 2) by its gather kernel
        R = self.input_resolution
        h1 = R // 2
        s1, s2, s3 = ws["stem"]
        c1, c2, c3 = self.stem
        d1, d2, d3 = ws["dz_stem"]
        C_("cg_avgpool2x2_nhwc_bwd", P(g32), 1, P(s3), n, h1, h1, s3.shape[1], P(d3), 0)
        relu(self._im2col(ws, d3, n, h1, c3.cout, 1, c3.kt), c3.wt, _lib.EPI_DRELU_BF16, mask=s2, out=d2)
        relu(self._im2col(ws, d2, n, h1, c2.cout, 1, c2.kt), c2.wt, _lib.EPI_DRELU_BF16, mask=s1, out=d1)
        C_("cg_conv3x3s2_dgrad", P(d1), n, R, R, c1.cout, d1.stride(0), P(self.w_stem1_f32), 3, self.kpad, P(ws["dpatch"]))

    def flops_fwd_bwd(self, n):
        """Algorithmic FLOPs (2 x MAC) of forward + input gradient for n images, unpadded channel counts."""
        R, h1 = self.input_resolution, self.input_resolution // 2
        conv = lambda m, cin, cout, k: 2 * m * cin * cout * k * k  # noqa: E731
        fwd = sum(conv(h1 * h1, c.cin, c.cout, 3) for c in self.stem)
        bwd = sum(conv(h1 * h1, c.cin, c.cout, 3) for c in self.stem)  # conv1's dgrad: same MACs
        for blk, (hi, ho) in zip(self.blocks, self._geometry()):
            cin, p = blk["cin"], blk["planes"]
            f = conv(hi * hi, cin, p, 1) + conv(hi * hi, p, p, 3) + conv(ho * ho, p, 4 * p, 1)
            if blk["ds"] is not None:
                f += conv(ho * ho, cin, 4 * p, 1)
            fwd += f
            bwd += f
        C, T, E = self.embed_width, self.tokens, self.output_dim
        fwd += 6 * T * C * C + 4 * T * T * C + 2 * C * E
        bwd += 6 * T * C * C + 8 * T * T * C + 2 * C * E
        return n * (fwd + bwd)


class TextTransformerB200:
    """Frozen OpenAI CLIP text transformer (``CLIP.encode_text``), forward only, on sm_100a kernels.  It runs once per job
    (preprocessing.py:11-24), so every pass is eager with per-call activation buffers: no CUDA graphs, no workspace cache."""

    def __init__(self, name, state_dict, device):
        context, vocab, width, layers, heads, embed = CLIP_TEXT_CONFIGS[name]
        self.name = name
        self.context_length, self.vocab_size, self.width, self.layers, self.heads, self.output_dim = context, vocab, width, layers, heads, embed
        self.device = torch.device(device)
        sd, dev = state_dict, self.device
        self.token_embedding = _f32(sd["token_embedding.weight"], dev)
        self.pos = _f32(sd["positional_embedding"], dev)
        self.ln_final = (_f32(sd["ln_final.weight"], dev), _f32(sd["ln_final.bias"], dev))
        self.proj = _f32(sd["text_projection"], dev)
        self.blocks = _pack_blocks(sd, "transformer.resblocks.", layers, dev, transposed=False)  # no dgrad

    def forward_tokens(self, tokens):
        """tokens: int32 [N, context] on the tower's device, ids in [0, vocab) -> embeddings [N, E] fp32."""
        n, T, D, E = tokens.shape[0], self.context_length, self.width, self.output_dim
        M = n * T
        dev = self.device
        f32 = lambda *s: torch.empty(*s, device=dev, dtype=torch.float32)
        b16 = lambda *s: torch.empty(*s, device=dev, dtype=torch.bfloat16)
        x, x_mid, mean, rstd = f32(M, D), f32(M, D), f32(M), f32(M)
        h, qkv, ctx, hg, u, lse = b16(M, D), b16(M, 3 * D), b16(M, D), b16(M, 4 * D), b16(M, 4 * D), f32(n, self.heads, T)
        y, emb = f32(n, D), f32(n, E)
        P, C = _lib.ptr, _lib.call
        # one set of buffers for every layer, which updates x in place (u: the pre-activation, unused)
        L = {"mean1": mean, "rstd1": rstd, "qkv": qkv, "ctx": ctx, "lse": lse, "x_mid": x_mid, "mean2": mean, "rstd2": rstd, "u": u}
        C("cg_text_embed_fwd", P(tokens), P(self.token_embedding), P(self.pos), n, T, D, self.vocab_size, P(x))
        for blk in self.blocks:
            _block_forward("cg_attention_causal_fwd", blk, n, T, self.heads, x, x, L, h, hg)
        C("cg_text_pool_fwd", P(x), P(tokens), n, T, D, P(self.ln_final[0]), P(self.ln_final[1]), P(y))
        C("cg_vit_proj_fwd", P(y), P(self.proj), n, D, E, P(emb))
        return emb


def _require_keys(sd, keys, where, tower):
    missing = [k for k in keys if k not in sd]
    if missing:
        raise KeyError("%s lacks %d %s keys (first: %s): expected OpenAI CLIP naming" % (where, len(missing), tower, missing[0]))


def _check_text_state_dict(name, sd, where):
    """KeyError naming the first missing text-tower key, ValueError on a shape that does not match CLIP_TEXT_CONFIGS (host only)."""
    shapes = clip_text_state_dict_shapes(name)
    _require_keys(sd, shapes, where, "text-tower")
    for k, shape in shapes.items():
        if tuple(sd[k].shape) != shape:
            raise ValueError("%s: %s has shape %s, the %s text tower needs %s" % (where, k, tuple(sd[k].shape), name, shape))


class _EncodeImageFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image, tower, normalize):
        _lib.require_cuda(image)
        if image.dim() != 4 or image.shape[1] != 3 or image.shape[2] != tower.input_resolution or image.shape[3] != tower.input_resolution:
            raise ValueError("expected [N,3,%d,%d] images, got %s" % (tower.input_resolution, tower.input_resolution, tuple(image.shape)))
        img = image.contiguous().float()
        n, cs = img.shape[0], img.shape[2]
        patches = torch.empty(n, tower.grid ** 2, tower.kpad, device=img.device, dtype=torch.bfloat16)
        _lib.call("cg_patchify_fwd", _lib.ptr(img), n, cs, tower.patch, tower.kpad, int(normalize), _lib.ptr(patches))
        emb = tower.forward_patches(patches)
        ctx.tower, ctx.normalize, ctx.shape, ctx.dtype = tower, normalize, image.shape, image.dtype
        ctx.generation = tower._generation
        return emb

    @staticmethod
    def backward(ctx, demb):
        tower = ctx.tower
        dpatch = tower.backward_patches(demb, generation=ctx.generation)
        n, _, cs, _ = ctx.shape
        dimg = torch.empty(ctx.shape, device=demb.device, dtype=torch.float32)
        _lib.call("cg_patchify_bwd", _lib.ptr(dpatch), 1, n, cs, tower.patch, tower.kpad, int(ctx.normalize), _lib.ptr(dimg))
        return dimg.to(ctx.dtype), None, None


class _Visual:
    """``clip_model.visual``: what sample.py:167 reads, callable like the OpenAI module."""

    def __init__(self, tower):
        self.tower = tower
        self.input_resolution = tower.input_resolution
        self.output_dim = tower.output_dim

    def __call__(self, image):
        return _EncodeImageFn.apply(image, self.tower, False)


class CLIPModelB200:
    """Value type of the dict returned by ``load_clip_models`` (models.py:74-84)."""

    def __init__(self, name, state_dict=None, device="cuda", seed=1):
        self.name = name
        if name in CLIP_RESNET_CONFIGS:
            _resnet_device(device)  # before the random init: the tower has no CPU path
            sd = state_dict if state_dict is not None else random_clip_resnet_state_dict(name, seed)
            self.visual = _Visual(ModifiedResNetB200(name, sd, device))
        elif name in CLIP_CONFIGS:
            sd = state_dict if state_dict is not None else random_clip_state_dict(name, seed)
            self.visual = _Visual(VisionTransformerB200(name, sd, device))
        else:
            raise ValueError("unsupported CLIP model %r: this path implements %s" % (name, sorted(CLIP_CONFIGS) + sorted(CLIP_RESNET_CONFIGS)))
        # the text tower is built on the first encode_text (image-only use keeps its memory and load time): until then the
        # checkpoint's non-visual tensors stay where the caller put them (load_clip_models: host memory); random init is seeded
        self._seed, self._text = seed, None
        self._text_sd = None if state_dict is None else {k: v for k, v in state_dict.items() if not k.startswith("visual.")}

    def encode_image(self, image):
        """image: CLIP-normalised [N,3,res,res] -> [N,E] fp32 (differentiable w.r.t. image)."""
        return self.visual(image)

    def encode_image_normalized_input(self, image01):
        """[0,1] image -> embedding with CLIP_NORMALIZE fused into the patchify kernel (embed_image's fast path)."""
        return _EncodeImageFn.apply(image01, self.visual.tower, True)

    def encode_text(self, text):
        """OpenAI ``CLIP.encode_text``: token ids [N, context] (int32 or int64, as ``clip.tokenize(...).to(device)`` gives them) ->
        [N, E] fp32 without grad_fn.  The sequence is pooled at its first maximal id (the end-of-text token)."""
        if self.name not in CLIP_TEXT_CONFIGS:
            raise ValueError("no text-tower configuration for %r (CLIP_TEXT_CONFIGS)" % self.name)
        context, vocab = CLIP_TEXT_CONFIGS[self.name][:2]
        if not isinstance(text, torch.Tensor) or text.dim() != 2 or text.shape[1] != context:
            raise ValueError("expected token ids of shape [N, %d], got %s" % (context, tuple(getattr(text, "shape", ()))))
        if text.dtype.is_floating_point or text.dtype.is_complex or text.dtype == torch.bool:
            raise ValueError("expected integer token ids, got %s" % text.dtype)
        if text.shape[0] == 0:
            raise ValueError("expected at least one sequence")
        lo, hi = torch.stack([text.min(), text.max()]).tolist()  # the one host read of the call
        if lo < 0 or hi >= vocab:
            raise ValueError("token ids must lie in [0, %d), got [%d, %d]" % (vocab, lo, hi))
        sd = None
        if self._text is None:
            sd = self._text_sd if self._text_sd is not None else random_clip_text_state_dict(self.name, self._seed)
            _check_text_state_dict(self.name, sd, "the %s checkpoint" % self.name)
        _lib.require_cuda(text)
        model_device = self.visual.tower.pos.device  # (an explicit index, unlike a bare "cuda")
        if text.device != model_device:
            raise ValueError("token ids are on %s, the model on %s" % (text.device, model_device))
        if self._text is None:
            self._text = TextTransformerB200(self.name, sd, model_device)
            self._text_sd = None
        with torch.no_grad():
            return self._text.forward_tokens(text.to(torch.int32).contiguous())

    def eval(self):
        return self

    def requires_grad_(self, flag=False):
        return self  # weights are frozen by construction (models.py:67-71)

    def to(self, device):
        return self


def load_clip_models(model_names, device=None, allow_random_init=False):
    """models.py:74-84.  Weights: ``$CLIPGUIDE_B200_WEIGHTS/<name with / -> _>.pt``, a state dict in OpenAI's key naming
    (``visual.conv1.weight`` ...; what ``clip.load(name).state_dict()`` holds).  A missing directory or file is an ERROR --
    guidance with random weights is meaningless -- unless the caller opts in with ``allow_random_init=True`` (benchmarks and
    tests: there is no network on the benchmark boxes, and throughput does not depend on the weight values).  Only the
    ``visual.*`` keys are checked here; the text tower's tensors (``token_embedding.weight`` ...) stay in host memory until the
    first ``encode_text``, which checks and uploads them (a visual-only checkpoint loads; its encode_text raises KeyError)."""
    device = device or "cuda"
    wdir = os.environ.get("CLIPGUIDE_B200_WEIGHTS")
    models = {}
    for i, name in enumerate(model_names):
        if name not in CLIP_CONFIGS and name not in CLIP_RESNET_CONFIGS:
            raise ValueError("unsupported CLIP model %r: this path implements %s" % (name, sorted(CLIP_CONFIGS) + sorted(CLIP_RESNET_CONFIGS)))
        sd = None
        path = os.path.join(wdir, name.replace("/", "_") + ".pt") if wdir else None
        if path and os.path.exists(path):
            sd = torch.load(path, map_location="cpu")
            keys = clip_resnet_state_dict_shapes(name) if name in CLIP_RESNET_CONFIGS else random_clip_state_dict_keys(name)
            _require_keys(sd, keys, path, "visual-tower")
        elif not allow_random_init:
            raise FileNotFoundError(
                "no weights for %r: set CLIPGUIDE_B200_WEIGHTS to a directory holding %s.pt (OpenAI CLIP state dict), or pass "
                "allow_random_init=True for benchmarking with seeded random weights" % (name, name.replace("/", "_")))
        models[name] = CLIPModelB200(name, sd, device, seed=1 + i)
    return models


def random_clip_state_dict_keys(name):
    """The ``visual.*`` keys the tower reads from a state dict."""
    _, _, _, layers, _, _ = CLIP_CONFIGS[name]
    return ["visual.conv1.weight", "visual.class_embedding", "visual.positional_embedding", "visual.proj", "visual.ln_pre.weight",
            "visual.ln_pre.bias", "visual.ln_post.weight", "visual.ln_post.bias"] + _block_keys("visual.transformer.resblocks.", layers)


class LinearAestheticPredictor(nn.Module):
    """models.py:188-196"""

    def __init__(self, input_dim):
        super().__init__()
        self.linear = nn.Linear(input_dim, 1)

    def forward(self, input):
        return self.linear(input)


class MLPAestheticPredictor(nn.Module):
    """models.py:200-217 -- five Linear layers, no activations; the dropouts are identity in eval mode"""

    def __init__(self, input_dim):
        super().__init__()
        dims = [input_dim, 1024, 128, 64, 16, 1]
        drops = [0.2, 0.2, 0.1, None, None]
        mods = []
        for a, b, p in zip(dims[:-1], dims[1:], drops):
            mods.append(nn.Linear(a, b))
            if p is not None:
                mods.append(nn.Dropout(p))
        self.layers = nn.Sequential(*mods)

    def forward(self, input):
        return self.layers(input)


def load_aesthetic_predictors(predictor_names, device=None):
    """models.py:220-240 with seeded random init instead of the downloaded checkpoints."""
    predictors = {}
    for i, name in enumerate(predictor_names):
        dim = CLIP_CONFIGS[name][5]
        with torch.random.fork_rng(devices=[]):  # do not disturb the job's global seed (functional.py:105-111)
            torch.manual_seed(100 + i)
            model = MLPAestheticPredictor(dim) if dim == 768 else LinearAestheticPredictor(dim)
        predictors[name] = model.eval().requires_grad_(False).to(device or "cuda")
    return predictors
