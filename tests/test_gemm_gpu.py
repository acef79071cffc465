"""GPU parity of the tcgen05/TMEM/TMA GEMM and its seven fused epilogues against the float64 oracle (oracle/gemm.py): per element within
its error model, bit for bit where the inputs make the result exact, on NaN-tailed operands into guarded outputs, on every tile variant
(forced in child processes), on the 128-bit epilogue path, and bit-identical under repetition and row rotation."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle():
    from oracle import gemm

    return gemm


def _assert_within(res, what):
    assert res["guards"], "%s: wrote outside its outputs" % what
    assert res["inexact"] == 0, "%s: %d elements differ from the exact result" % (what, res["inexact"])
    assert max(res["ratios"].values()) <= 1.0, (what, res["ratios"])


SHAPES = [(128, 128, 64), (128, 256, 128), (200, 384, 192), (1576, 2304, 768), (6304, 768, 3072), (50, 128, 64), (16448, 1024, 640), (777, 512, 1024)]


@pytest.mark.parametrize("M,N,K", SHAPES)
def test_gemm_plain_f32(M, N, K, record_property):
    G = _oracle()
    res = G.check_gemm(G.F32, G.gauss(M, N, K, 0, device="cuda"))
    record_property("err_over_bound", {"variant": G.VARIANTS[G.tile_variant(M, N, K, G.F32)], **res["ratios"]})
    _assert_within(res, "F32 %dx%dx%d" % (M, N, K))


@pytest.mark.parametrize("M,N,K", SHAPES[:5])
def test_gemm_epilogues(M, N, K, record_property):
    G = _oracle()
    from clip_diffusion_b200 import vit_ops

    inp = G.gauss(M, N, K, 1, device="cuda")
    worst = {}
    for epi in (G.BIAS_BF16, G.BIAS_RESID_F32, G.BIAS_QGELU_BF16, G.DQGELU_BF16, G.BF16):
        res = G.check_gemm(epi, inp)
        worst[G.EPI_NAMES[epi]] = max(res["ratios"].values())
        _assert_within(res, "%s %dx%dx%d" % (G.EPI_NAMES[epi], M, N, K))
    # bias + residual in place (aux aliases out)
    x = inp["resid"].clone()
    vit_ops.gemm_bf16_tn(inp["a"], inp["b"], G.BIAS_RESID_F32, bias=inp["bias"], out=x, aux=x)
    r = G.ratios({"out": x}, G.reference(G.BIAS_RESID_F32, inp))["out"]
    worst["BIAS_RESID_F32 in place"] = r
    record_property("err_over_bound", worst)
    assert r <= 1.0, r


def test_gemm_patch_pos_epilogue():
    G = _oracle()
    for regime in ("gauss", "exact"):
        res = G.check_gemm(G.PATCH_POS_F32, G.make_inputs(regime, 5 * 49, 256, 192, 2, g2=49, device="cuda"))
        _assert_within(res, "patch %s" % regime)  # includes: the class-token rows keep their value


def test_gemm_strided_operands_and_repeat():
    """Leading dimensions larger than K (column slices of a wider buffer, NaN in the gap), a gap between output rows, called twice
    (tensor-map cache)."""
    G = _oracle()
    inp = G.gauss(300, 128, 256, 3, device="cuda")
    for _ in range(2):
        _assert_within(G.check_gemm(G.F32, inp, lda_pad=256, ldb_pad=64, ldo_pad=128), "strided")


@pytest.mark.parametrize("epi", range(7), ids=["BIAS_BF16", "BIAS_RESID_F32", "BIAS_QGELU_BF16", "DQGELU_BF16", "F32", "BF16", "PATCH_POS_F32"])
def test_gemm_128bit_epilogue_path(epi, record_property):
    """out (and aux) 16- but not 32-byte aligned: the epilogue takes its 128-bit store / load path in this process."""
    G = _oracle()
    off = 4 if epi in G.F32_OUT else 8  # 16 bytes
    worst = {}
    for regime, (M, N, K, g2) in (("exact", (777, 512, 1024, 37)), ("gauss", (1576, 2304, 768, 197)), ("sweep", (256, 256, 256, 64))):
        res = G.check_gemm(epi, G.make_inputs(regime, M, N, K, 9, g2=g2, device="cuda"), offset=off)
        worst[regime] = max(res["ratios"].values())
        _assert_within(res, "%s %s offset %d" % (G.EPI_NAMES[epi], regime, off))
    record_property("err_over_bound", worst)


def test_gemm_rejects_bad_shapes():
    from clip_diffusion_b200 import _lib, vit_ops

    a = torch.zeros(16, 48, device="cuda", dtype=torch.bfloat16)
    b = torch.zeros(128, 48, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(_lib.ClipGuideError):
        vit_ops.gemm_bf16_tn(a, b, _lib.EPI_F32)
    a = torch.zeros(256, 64, device="cuda", dtype=torch.bfloat16)
    b = torch.zeros(256, 64, device="cuda", dtype=torch.bfloat16)
    bias = torch.zeros(256, device="cuda")
    f32, bf = torch.zeros(256, 256, device="cuda"), torch.zeros(256, 256, device="cuda", dtype=torch.bfloat16)
    bad = [
        dict(epi=_lib.EPI_F32, out=bf),                                       # out dtype
        dict(epi=_lib.EPI_BF16, out=torch.zeros(255, 256, device="cuda", dtype=torch.bfloat16)),  # out too small
        dict(epi=_lib.EPI_BIAS_BF16, bias=bias.double()),                     # bias dtype
        dict(epi=_lib.EPI_BIAS_BF16, bias=bias[:128]),                        # bias length
        dict(epi=_lib.EPI_BIAS_BF16, bias=torch.zeros(512, device="cuda")[::2]),  # bias not contiguous
        dict(epi=_lib.EPI_BIAS_RESID_F32, bias=bias, aux=bf),                 # aux dtype
        dict(epi=_lib.EPI_BIAS_RESID_F32, bias=bias, out=f32, aux=torch.zeros(256, 512, device="cuda")[:, :256]),  # aux row stride
        dict(epi=_lib.EPI_DQGELU_BF16, aux=None),                             # aux missing
        dict(epi=_lib.EPI_DQGELU_BF16, aux=torch.zeros(128, 256, device="cuda", dtype=torch.bfloat16)),  # aux too small
        dict(epi=_lib.EPI_PATCH_POS_F32, out=f32, pos=torch.zeros(2, 256, device="cuda"), g2=4),  # pos too small, out too small
    ]
    for kw in bad:
        epi = kw.pop("epi")
        with pytest.raises(_lib.ClipGuideError):
            vit_ops.gemm_bf16_tn(a, b, epi, **kw)


# tile variants: CG_GEMM_* are read once per process, so each forced variant runs the whole matrix in a child process, with a timeout
# (a cluster deadlock must not hang the suite)
FORCE = {"auto": {}, "pair256x256": {"CG_GEMM_PAIR": "1"}, "bn128": {"CG_GEMM_PAIR": "0", "CG_GEMM_BN": "128"},
         "bn256": {"CG_GEMM_PAIR": "0", "CG_GEMM_BN": "256"}, "wide0": {"CG_GEMM_WIDE": "0"}}
FORCED_VARIANT = {"pair256x256": 2, "bn128": 1, "bn256": 0}


def _run_child(force):
    code = "import sys; sys.path.insert(0, %r)\nfrom oracle import gemm as G\nG.run_matrix(G.matrix_cases(), G.INVARIANCE_SHAPES)\n" % ROOT
    env = {k: v for k, v in os.environ.items() if not k.startswith("CG_GEMM_")}
    env.update(FORCE[force])
    res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    line = [ln for ln in res.stdout.splitlines() if ln.startswith("GEMM_MATRIX ")]
    assert line, res.stdout[-3000:]
    return json.loads(line[-1][len("GEMM_MATRIX "):])


@pytest.mark.parametrize("force", list(FORCE))
def test_gemm_forced_tile_variant_in_subprocess(force, record_property):
    """7 epilogues x 4 regimes over the tail classes of every variant and the towers' real shapes, on the variant the environment
    forces; the variant of every case is what cg_gemm_tile_variant reports."""
    G = _oracle()
    out = _run_child(force)
    cases, sms = out["cases"], out["sms"]
    worst, failures = {}, []
    for c in cases:
        key = "%s/%s/%s" % (G.VARIANTS[c["variant"]], G.EPI_NAMES[c["epi"]], c["regime"])
        for name, r in c["ratios"].items():
            worst[key + "/" + name] = max(worst.get(key + "/" + name, 0.0), r)
        if not c["guards"] or c["inexact"] or max(c["ratios"].values()) > 1.0:
            failures.append(c)
    sigma = max([c["sigma_err"] for c in cases if "sigma_err" in c and c["regime"] == "sweep"] or [0.0])
    record_property("err_over_bound", worst)
    record_property("sigmoid_err_sweep", sigma)
    record_property("invariance", out["invariance"])
    assert not failures, failures[:5]
    assert len(cases) == len(G.matrix_cases())
    assert {(c["epi"], c["regime"]) for c in cases} == {(e, r) for e in range(7) for r in G.REGIMES}
    for inv in out["invariance"]:
        assert inv["identical"], inv
    if force in FORCED_VARIANT:
        v = FORCED_VARIANT[force]
        ran = [c for c in cases if c["variant"] == v]
        assert {c["epi"] for c in ran} == set(range(7)), "variant %s did not run every epilogue" % G.VARIANTS[v]
        classes = set().union(*(G.tail_classes(c["M"], c["N"], c["K"], v, sms) for c in ran))
        assert G.REQUIRED_CLASSES[v] <= classes, G.REQUIRED_CLASSES[v] - classes
        assert all(inv["variant"] == v for inv in out["invariance"])
    if force == "auto":
        by_shape = {(c["M"], c["N"], c["K"], c["epi"]): c["variant"] for c in cases}
        assert by_shape[(3136, 768, 3072, G.PATCH_POS_F32)] == 2  # ViT-B/32 patch embedding at 64 cutouts: the CTA pair
        assert by_shape[(16384, 1024, 640, G.PATCH_POS_F32)] == 0  # ViT-L/14's: 128 x 256
