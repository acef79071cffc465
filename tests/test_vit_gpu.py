"""GPU parity of the ViT building blocks and the whole tower against the CPU oracle (oracle/clip_vit.py: fp32
restatement of the OpenAI VisionTransformer, cross-checked against transformers' CLIP in test_oracle_pins.py).
north_star tolerances: embedding cosine >= 0.999, input-gradient relative L2 <= 1e-2 (bf16 operands, fp32
accumulation and residual stream)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

COS_MIN = 0.999
GRAD_REL_MAX = 1e-2


def _lib_ops():
    from clip_diffusion_b200 import _lib

    return _lib


@pytest.mark.parametrize("M,D,stride", [(40, 128, 128), (300, 768, 768), (7, 1024, 1024 * 5), (1000, 256, 256)])
def test_layernorm_fwd_bwd(M, D, stride):
    _lib = _lib_ops()
    g = torch.Generator().manual_seed(M + D)
    buf = torch.randn(M, stride, generator=g) * 2 + 0.5
    x = buf[:, :D].clone().requires_grad_()
    gamma = 1 + 0.1 * torch.randn(D, generator=g)
    beta = 0.1 * torch.randn(D, generator=g)
    ref = torch.nn.functional.layer_norm(x, (D,), gamma, beta, 1e-5)
    dy = torch.randn(M, D, generator=g)
    (gref,) = torch.autograd.grad((ref * dy).sum(), x)
    P = _lib.ptr
    xb, gc, bc, dyc = buf.cuda(), gamma.cuda(), beta.cuda(), dy.cuda()  # keep device copies alive across the calls
    yb = torch.empty(M, D, device="cuda", dtype=torch.bfloat16)
    yf = torch.empty(M, D, device="cuda")
    mean = torch.empty(M, device="cuda"); rstd = torch.empty(M, device="cuda")
    _lib.call("cg_layernorm_fwd", P(xb), P(gc), P(bc), M, D, stride, P(yb), P(yf), P(mean), P(rstd))
    assert (yf.cpu() - ref.detach()).abs().max().item() < 2e-5
    assert (yb.float().cpu() - ref.detach()).abs().max().item() < 3e-2
    dx = torch.full((M, stride), 3.0, device="cuda")
    dxb = torch.zeros(M, stride, device="cuda", dtype=torch.bfloat16)
    _lib.call("cg_layernorm_bwd", P(dyc), P(xb), P(gc), P(mean), P(rstd), M, D, stride, 1, P(dx), P(dxb))
    assert ((dx[:, :D].cpu() - 3.0) - gref).abs().max().item() < 5e-5 * max(1.0, gref.abs().max().item())
    assert (dxb[:, :D].float().cpu() - (gref + 3.0)).abs().max().item() < 5e-2 * max(1.0, gref.abs().max().item())
    if stride > D:
        assert (dx[:, D:] == 3.0).all()


FWD_BWD_SHAPES = [(3, 50, 2), (2, 197, 12), (1, 257, 16), (1, 577, 4), (5, 5, 2), (2, 64, 3), (2, 65, 1), (1, 128, 2), (1, 129, 2),
                  (2, 256, 2), (1, 272, 1), (3, 257, 4), (1, 16, 1), (2, 192, 2), (2, 193, 1),
                  # more (image, head) items than SMs: the persistent kernels walk several items per CTA and pipeline across
                  # them (even / odd block counts per item, with and without the edge token T = 64 m + 1)
                  (40, 257, 4), (64, 50, 3), (30, 129, 5), (50, 65, 3), (52, 100, 3), (38, 272, 4), (75, 197, 2), (150, 257, 3),
                  (2, 130, 2), (2, 66, 1), (1, 2, 1), (3, 1, 2)]
# sharp logits (oracle/attention.py): T = 129 (edge token, 2 blocks: no warpgroup sees a second block, a control), 193 (edge, 3 blocks),
# 197, 200, 256, 257 (edge), 272 on the tcgen05 kernels; 273 and 577 on the mma.sync kernels
REGIME_T = (129, 193, 197, 200, 256, 257, 272, 273, 577)
REGIME_HEADS = (1, 4, 16)


def _fwd_bwd_cases():
    cases = [pytest.param(n, T, heads, "flat", None, id="%d-%d-%d" % (n, T, heads)) for n, T, heads in FWD_BWD_SHAPES]
    i = 0
    for regime in ("sharp", "sharp_kmean", "staircase_up", "staircase_down", "sink_query", "huge_pos", "huge_neg", "neighbour", "sink"):
        for T in REGIME_T:
            edge = int(T <= 272 and (T - 1) % 64 == 0)
            for pos in (_attn_oracle().sink_positions(T, edge) if regime == "sink" else [None]):
                heads, n = REGIME_HEADS[i % 3], 3 if regime == "neighbour" else 2
                i += 1
                cases.append(pytest.param(n, T, heads, regime, pos, id="%d-%d-%d-%s%s" % (n, T, heads, regime, "" if pos is None else pos)))
    return cases


def _attn_oracle():
    from oracle import attention

    return attention


@pytest.mark.parametrize("n,T,heads,regime,pos", _fwd_bwd_cases())
def test_attention_fwd_bwd(n, T, heads, regime, pos, record_property):
    """tcgen05/TMEM kernels (vit_attention_tc.cu) for T <= 272, mma.sync kernels (vit_attention.cu) beyond, against the float64 oracle
    within its error model (oracle/attention.py), in guarded buffers."""
    A = _attn_oracle()
    seed = T + heads if regime == "flat" else 1000 * n + T + heads
    qkv, dctx = A.make_inputs(regime, n, T, heads, seed, **({} if pos is None else {"pos": pos}))
    worst = A.check_attention(n, T, heads, qkv, dctx)
    record_property("err_over_bound", {"kernel": "tcgen05" if T <= 272 else "mma.sync", "regime": regime, **worst})
    assert max(worst.values()) <= 1.0, worst


TOWERS = {
    "test-tiny/32": (64, 32, 128, 2, 2, 64),
    "test-small/16": (64, 16, 256, 3, 4, 128),
    "test-k/14": (56, 14, 128, 2, 2, 64),
}


def _tower_pair(name, n):
    from clip_diffusion_b200 import models
    from oracle.clip_vit import CONFIGS, OracleCLIP

    if name in TOWERS:
        models.register_clip_config(name, *TOWERS[name])
        assert CONFIGS[name] == TOWERS[name]
    sd = models.random_clip_state_dict(name, seed=3)
    mine = models.CLIPModelB200(name, sd, "cuda")
    ref = OracleCLIP(name, state_dict=sd)
    res = mine.visual.input_resolution
    g = torch.Generator().manual_seed(n)
    img = torch.rand(n, 3, res, res, generator=g)
    return mine, ref, img


# the real towers at full size (random init): these are the shapes bench.py runs (c2 = ViT-B/16, target = ViT-L/14, c5 = ViT-L/14@336px)
@pytest.mark.parametrize("name,n", [("test-tiny/32", 4), ("test-small/16", 3), ("test-k/14", 5), ("ViT-B/32", 2), ("ViT-B/16", 4), ("ViT-L/14", 2),
                                    ("ViT-L/14@336px", 1)])
def test_tower_embedding_and_input_gradient(name, n):
    from clip_diffusion_b200.utils.functional import embed_image
    from oracle.cutouts import clip_normalize

    mine, ref, img = _tower_pair(name, n)
    xr = img.clone().requires_grad_()
    er = ref.encode_image(clip_normalize(xr))
    w = torch.randn(er.shape, generator=torch.Generator().manual_seed(7))
    (gr,) = torch.autograd.grad((er * w).sum(), xr)
    xc = img.cuda().requires_grad_()
    em = embed_image(mine, xc, clip_normalize=True)
    assert em.dtype == torch.float32 and em.shape == er.shape
    (gm,) = torch.autograd.grad((em * w.cuda()).sum(), xc)
    cos = torch.nn.functional.cosine_similarity(em.cpu(), er.detach(), dim=-1)
    assert cos.min().item() >= COS_MIN, cos
    rel = ((gm.cpu() - gr).norm() / gr.norm()).item()
    assert rel <= GRAD_REL_MAX, rel


def test_encode_image_matches_embed_image_unfused():
    """encode_image on an already-normalised tensor == embed_image(clip_normalize=True) up to bf16 rounding of the input."""
    from clip_diffusion_b200.utils.functional import CLIP_NORMALIZE, embed_image

    mine, _, img = _tower_pair("test-small/16", 2)
    a = embed_image(mine, img.cuda(), clip_normalize=True)
    b = mine.encode_image(CLIP_NORMALIZE(img.cuda()))
    assert torch.nn.functional.cosine_similarity(a, b, dim=-1).min().item() > 0.9999


def test_patchify_roundtrip():
    _lib = _lib_ops()
    n, cs, patch, kpad = 2, 56, 14, 640
    img = torch.rand(n, 3, cs, cs, device="cuda")
    pm = torch.empty(n, (cs // patch) ** 2, kpad, device="cuda", dtype=torch.bfloat16)
    _lib.call("cg_patchify_fwd", _lib.ptr(img), n, cs, patch, kpad, 0, _lib.ptr(pm))
    assert (pm[:, :, 3 * patch * patch:] == 0).all()
    back = torch.empty_like(img)
    _lib.call("cg_patchify_bwd", _lib.ptr(pm), 0, n, cs, patch, kpad, 0, _lib.ptr(back))
    assert (back - img).abs().max().item() < 4e-3  # bf16 rounding of values in [0,1]


def test_stale_workspace_backward_raises_instead_of_wrong_gradients():
    """ADVICE r1: the saved activations live in ONE workspace per (tower, batch size).  Two same-size forwards followed by the
    backward of the first must raise (generation id), never silently differentiate against the second forward's activations."""
    from clip_diffusion_b200.utils.functional import embed_image

    mine, _, img = _tower_pair("test-tiny/32", 3)
    a = img.cuda().requires_grad_()
    b = (1 - img).cuda().requires_grad_()
    ea = embed_image(mine, a)
    eb = embed_image(mine, b)  # same batch size: overwrites the saved activations of `ea`
    (gb,) = torch.autograd.grad(eb.sum(), b)  # latest forward: fine
    assert torch.isfinite(gb).all()
    with pytest.raises(RuntimeError, match="stale CLIP activations"):
        torch.autograd.grad(ea.sum(), a)
    # sequential use (sample.py:199-214: differentiate each batch before embedding the next) keeps working
    ea = embed_image(mine, a)
    (ga,) = torch.autograd.grad(ea.sum(), a)
    eb = embed_image(mine, b)
    (gb2,) = torch.autograd.grad(eb.sum(), b)
    assert torch.equal(gb, gb2) and torch.isfinite(ga).all()


def test_tower_cuda_graph_replay_equals_eager_launches():
    """The tower captures its forward / backward pass into CUDA graphs on the second call of a batch size and replays them afterwards
    (models.VisionTransformerB200._run_pass).  Same kernels on the same buffers: embeddings and patch gradients must be bit-identical
    with a tower that issues every launch eagerly, for every call (eager first call, capture, replays) and two batch sizes."""
    from clip_diffusion_b200 import models

    name = "test-small/16"
    models.register_clip_config(name, *TOWERS[name])
    sd = models.random_clip_state_dict(name, seed=5)
    graphed = models.CLIPModelB200(name, sd, "cuda").visual.tower
    eager = models.CLIPModelB200(name, sd, "cuda").visual.tower
    eager.use_graphs = False
    assert graphed.use_graphs
    g = torch.Generator().manual_seed(0)
    for it in range(5):
        for n in (3, 2):
            patches = (torch.randn(n, graphed.grid ** 2, graphed.kpad, generator=g) * 0.5).bfloat16().cuda()
            demb = torch.randn(n, graphed.output_dim, generator=g).cuda()
            e1, e2 = graphed.forward_patches(patches), eager.forward_patches(patches)
            assert torch.equal(e1, e2), (it, n)
            d1, d2 = graphed.backward_patches(demb).clone(), eager.backward_patches(demb).clone()
            assert torch.equal(d1, d2), (it, n)
    st = graphed._ws[3]["graphs"]
    assert st["fwd"]["graph"] is not None and st["bwd"]["graph"] is not None and not st["fwd"]["failed"] and not st["bwd"]["failed"]
