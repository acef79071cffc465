"""Thin tensor-level wrappers over the C-ABI ViT building blocks (include/clipguide_b200.h, "CLIP ViT").
They only marshal torch tensors into pointers/sizes; all arithmetic is in csrc/vit_*.cu."""
import torch

from clip_diffusion_b200 import _lib

_F32_OUT = (_lib.EPI_BIAS_RESID_F32, _lib.EPI_F32, _lib.EPI_PATCH_POS_F32)
_AUX_DTYPE = {_lib.EPI_BIAS_RESID_F32: torch.float32, _lib.EPI_BIAS_QGELU_BF16: torch.bfloat16, _lib.EPI_DQGELU_BF16: torch.bfloat16}
_NEEDS_BIAS = (_lib.EPI_BIAS_BF16, _lib.EPI_BIAS_RESID_F32, _lib.EPI_BIAS_QGELU_BF16)


def _check_matrix(name, t, dtype, rows, cols, device):
    if t.dtype != dtype or t.dim() != 2 or t.device != device:
        raise _lib.ClipGuideError("gemm_bf16_tn: %s must be a 2-D %s tensor on %s, got %s %s on %s" % (name, dtype, device, t.dtype, tuple(t.shape), t.device))
    if t.shape[0] < rows or t.shape[1] < cols or t.stride(1) != 1:
        raise _lib.ClipGuideError("gemm_bf16_tn: %s must hold at least [%d, %d] with unit column stride, got %s stride %s"
                                  % (name, rows, cols, tuple(t.shape), t.stride()))


def gemm_bf16_tn(a, b, epilogue, bias=None, out=None, aux=None, pos=None, g2=0, m=None):
    """acc[M,N] = a[M,K] @ b[N,K]^T with a fused epilogue (see CG_EPI_* in the header).  a, b: bf16 row-major
    (row stride may exceed K).  ``out``/``aux`` must be preallocated for in-place / auxiliary epilogues; the kernel
    addresses ``aux`` with ``out``'s row stride, so both must have the same one."""
    _lib.require_cuda(a, b, bias, out, aux, pos)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.stride(-1) == 1 and b.stride(-1) == 1
    M = a.shape[0] if m is None else m
    K = a.shape[1]
    N = b.shape[0]
    assert b.shape[1] == K
    out_dtype = torch.float32 if epilogue in _F32_OUT else torch.bfloat16
    if out is None:
        assert epilogue != _lib.EPI_PATCH_POS_F32, "the patch epilogue writes into a preallocated token buffer"
        out = torch.empty(M, N, device=a.device, dtype=out_dtype)
    if epilogue == _lib.EPI_BIAS_QGELU_BF16 and aux is None:
        aux = torch.empty(M, N, device=a.device, dtype=torch.bfloat16)
    out_rows = M // g2 * (g2 + 1) if epilogue == _lib.EPI_PATCH_POS_F32 and g2 > 0 else M
    _check_matrix("out", out, out_dtype, out_rows, N, a.device)
    if epilogue in _AUX_DTYPE:
        if aux is None:
            raise _lib.ClipGuideError("gemm_bf16_tn: epilogue %d needs aux" % epilogue)
        _check_matrix("aux", aux, _AUX_DTYPE[epilogue], M, N, a.device)
        if aux.stride(0) != out.stride(0):
            raise _lib.ClipGuideError("gemm_bf16_tn: aux row stride %d != out row stride %d" % (aux.stride(0), out.stride(0)))
    if epilogue in _NEEDS_BIAS:
        if bias is None or bias.dtype != torch.float32 or not bias.is_contiguous() or bias.shape != (N,) or bias.device != a.device:
            raise _lib.ClipGuideError("gemm_bf16_tn: epilogue %d needs a contiguous fp32 bias of length %d on %s" % (epilogue, N, a.device))
    if epilogue == _lib.EPI_PATCH_POS_F32 and (pos is None or pos.dtype != torch.float32 or not pos.is_contiguous()
                                               or pos.numel() < (g2 + 1) * N or pos.device != a.device):
        raise _lib.ClipGuideError("gemm_bf16_tn: the patch epilogue needs a contiguous fp32 pos of [g2 + 1, %d] on %s" % (N, a.device))
    _lib.call(
        "cg_gemm_bf16_tn", _lib.ptr(a), _lib.ptr(b), M, N, K, a.stride(0), b.stride(0), epilogue, _lib.ptr(bias), _lib.ptr(out),
        _lib.ptr(aux), out.stride(0), _lib.ptr(pos), g2,
    )
    return (out, aux) if epilogue == _lib.EPI_BIAS_QGELU_BF16 else out


_RELU_EPILOGUES = (_lib.EPI_BIAS_RELU_BF16, _lib.EPI_BIAS_RESID_RELU_BF16, _lib.EPI_DRELU_BF16, _lib.EPI_RESID_DRELU)


def gemm_bf16_tn_relu(a, b, epilogue, bias=None, resid=None, mask=None, out=None, out_bf16=None):
    """cg_gemm_bf16_tn_relu: acc[M,N] = a[M,K] @ b[N,K]^T with one of the ReLU-network epilogues (CG_EPI_BIAS_RELU_BF16 ..
    CG_EPI_RESID_DRELU in the header).  ``out`` (fp32 for RESID_DRELU, bf16 otherwise), ``resid``, ``mask`` and ``out_bf16`` share one
    row stride; resid may be ``out`` itself (RESID_DRELU)."""
    _lib.require_cuda(a, b, bias, resid, mask, out, out_bf16)
    if epilogue not in _RELU_EPILOGUES:
        raise _lib.ClipGuideError("gemm_bf16_tn_relu: %d is not a ReLU epilogue" % epilogue)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.stride(-1) == 1 and b.stride(-1) == 1
    M, K, N = a.shape[0], a.shape[1], b.shape[0]
    assert b.shape[1] == K
    f32 = epilogue == _lib.EPI_RESID_DRELU
    _check_matrix("out", out, torch.float32 if f32 else torch.bfloat16, M, N, a.device)
    for name, t in (("resid", resid), ("mask", mask), ("out_bf16", out_bf16)):
        if t is None:
            continue
        dtype = torch.float32 if (f32 and name == "resid") else torch.bfloat16
        _check_matrix(name, t, dtype, M, N, a.device)
        if t.stride(0) != out.stride(0):
            raise _lib.ClipGuideError("gemm_bf16_tn_relu: %s row stride %d != out row stride %d" % (name, t.stride(0), out.stride(0)))
    if epilogue in (_lib.EPI_BIAS_RELU_BF16, _lib.EPI_BIAS_RESID_RELU_BF16):
        if bias is None or bias.dtype != torch.float32 or not bias.is_contiguous() or bias.shape != (N,) or bias.device != a.device:
            raise _lib.ClipGuideError("gemm_bf16_tn_relu: epilogue %d needs a contiguous fp32 bias of length %d on %s" % (epilogue, N, a.device))
    _lib.call("cg_gemm_bf16_tn_relu", _lib.ptr(a), _lib.ptr(b), M, N, K, a.stride(0), b.stride(0), epilogue, _lib.ptr(bias), _lib.ptr(resid),
              _lib.ptr(mask), _lib.ptr(out), _lib.ptr(out_bf16), out.stride(0))
    return out
