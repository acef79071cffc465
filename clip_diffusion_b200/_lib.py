"""ctypes binding of csrc/libclipguide_b200.so (C ABI declared in include/clipguide_b200.h).

There is NO fallback: if the shared library has not been built (``python -c "import
__graft_entry__ as g; g.build()"`` or ``make -C clip_diffusion_b200/csrc``) every op raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CLIPGUIDE_B200_LIB") or os.path.join(_HERE, "csrc", "libclipguide_b200.so")  # the override is for developer builds (make trace)

CG_FMT_F32_NCHW = 0
CG_FMT_BF16_PATCH = 1
CG_FMT_F32_PATCH = 2

EPI_BIAS_BF16 = 0
EPI_BIAS_RESID_F32 = 1
EPI_BIAS_QGELU_BF16 = 2
EPI_DQGELU_BF16 = 3
EPI_F32 = 4
EPI_BF16 = 5
EPI_PATCH_POS_F32 = 6
# the ReLU-network epilogues, run through cg_gemm_bf16_tn_relu
EPI_BIAS_RELU_BF16 = 7
EPI_BIAS_RESID_RELU_BF16 = 8
EPI_DRELU_BF16 = 9
EPI_RESID_DRELU = 10

GEMM_TILE_128x256 = 0
GEMM_TILE_128x128 = 1
GEMM_TILE_PAIR_256x256 = 2


class CgCut(C.Structure):
    _fields_ = [("y0", C.c_int32), ("x0", C.c_int32), ("size", C.c_int32), ("flags", C.c_int32)]


class CgAug(C.Structure):
    _fields_ = [
        ("flip", C.c_int32),
        ("gray", C.c_int32),
        ("perm", C.c_int32 * 4),
        ("theta", C.c_float * 6),
        ("theta_fwd", C.c_float * 6),
        ("brightness", C.c_float),
        ("contrast", C.c_float),
        ("saturation", C.c_float),
        ("hue", C.c_float),
        ("augment", C.c_int32),
        ("normalize", C.c_int32),
        ("mean", C.c_float * 3),
        ("stdv", C.c_float * 3),
        ("noise_seed", C.c_uint64),
        ("cut_index0", C.c_uint64),
        ("noise_std", C.c_float),
        ("input01", C.c_int32),
        ("noise_mode", C.c_int32),
        ("noise_threads", C.c_uint32),
        ("noise_offset", C.c_uint64 * 3),
        ("noise_total", C.c_uint64),
    ]


_P = C.c_void_p
_I = C.c_int
_L = C.c_int64
_F = C.c_float

_SIGNATURES = {
    "cg_last_error": (C.c_char_p, []),
    "cg_abi_version": (_I, []),
    "cg_check_device": (_I, []),
    "cg_tv_loss_fwd_bwd": (_I, [_P, _I, _I, _I, _I, _F, _I, _P, _P, _P]),
    "cg_range_loss_fwd_bwd": (_I, [_P, _I, _I, _I, _I, _F, _I, _P, _P, _P]),
    "cg_randn_like_torch_geometry": (C.c_uint32, [_L, C.POINTER(C.c_uint64)]),
    "cg_randn_like_torch": (_I, [_P, _L, C.c_uint64, C.c_uint64, _P]),
    "cg_ms_ssim_workspace_bytes": (C.c_size_t, [_I, _I, _I]),
    "cg_ms_ssim_dissimilarity_fwd_bwd": (_I, [_P, _P, _I, _I, _I, _F, _I, _P, _P, _P, _P]),
    "cg_image_losses_fwd_bwd": (_I, [_P, _I, _I, _I, _I, _F, _F, _I, _P, _P, _P, _P]),
    "cg_spherical_dist_fwd": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "cg_spherical_dist_bwd": (_I, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "cg_spherical_loss_fwd_bwd": (_I, [_P, _P, _P, _I, _I, _I, _F, _P, _P, _P]),
    "cg_cutouts_workspace_bytes": (C.c_size_t, [_I, _I, _I]),
    "cg_cutouts_fwd": (_I, [_P, _I, _I, C.POINTER(CgCut), _I, _I, C.POINTER(CgAug), _P, _P, _I, _I, _I, _P, _P]),
    "cg_cutouts_bwd": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _F, _I, _I, _P, _P, _P]),
    "cg_layernorm_fwd": (_I, [_P, _P, _P, _I, _I, _L, _P, _P, _P, _P, _P]),
    "cg_layernorm_bwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _L, _I, _P, _P, _P]),
    "cg_gemm_bf16_tn": (_I, [_P, _P, _I, _I, _I, _L, _L, _I, _P, _P, _P, _L, _P, _I, _P]),
    "cg_gemm_tile_variant": (_I, [_I, _I, _I, _I]),
    "cg_gemm_bf16_tn_relu": (_I, [_P, _P, _I, _I, _I, _L, _L, _I, _P, _P, _P, _P, _P, _L, _P]),
    "cg_im2col3x3_nhwc": (_I, [_P, _I, _I, _I, _I, _L, _I, _I, _P, _P]),
    "cg_conv3x3s2_dgrad": (_I, [_P, _I, _I, _I, _I, _L, _P, _I, _I, _P, _P]),
    "cg_avgpool2x2_nhwc_fwd": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "cg_avgpool2x2_nhwc_bwd": (_I, [_P, _I, _P, _I, _I, _I, _I, _P, _I, _P]),
    "cg_resnet_attnpool_fwd": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "cg_resnet_attnpool_bwd": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "cg_resnet_attnpool_dctx": (_I, [_P, _I, _I, _I, _P, _P]),
    "cg_attention_fwd": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "cg_attention_bwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _P, _P, _P]),
    "cg_attention_causal_fwd": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "cg_text_embed_fwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "cg_text_pool_fwd": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _P]),
    "cg_vit_set_cls_rows": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "cg_vit_proj_fwd": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "cg_vit_proj_bwd": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "cg_vit_tokens_to_bf16": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "cg_patchify_fwd": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "cg_patchify_bwd": (_I, [_P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "cg_grad_finalize": (_I, [_P, _L, _F, _F, _P, _P, _P, _P]),
    "cg_any_nan": (_I, [_P, _L, _P, _P]),
    "cg_dynamic_threshold_workspace_bytes": (C.c_size_t, [_I]),
    "cg_dynamic_threshold": (_I, [_P, _I, _L, _F, _F, _P, _P, _P, _P]),
    "cg_groupnorm_nhwc_workspace_bytes": (C.c_size_t, [_I, _I, _I]),
    "cg_groupnorm_nhwc_geometry": (_I, [_I, _I, _I, C.POINTER(C.c_int)]),
    "cg_groupnorm_nhwc_fwd": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _F, _I, _I, _P, _P, _P, _P, _P]),
    "cg_bias_residual_add_stats_nhwc": (_I, [_P, _P, _P, _I, _I, _I, _P, _P, _P]),
    "cg_concat2_stats_nhwc": (_I, [_P, _I, _P, _I, _I, _I, _P, _P, _P]),
    "cg_groupnorm_nhwc_bwd": (_I, [_P, _I, _P, _I, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P]),
    "cg_bias_residual_add_nhwc": (_I, [_P, _P, _P, _L, _I, _P, _P]),
    "cg_resample2x_nhwc": (_I, [_P, _I, _I, _I, _I, _I, _F, _P, _P]),
    "cg_concat2_nhwc": (_I, [_P, _I, _P, _I, _L, _P, _I, _P]),
}

_lib = None
launch_count = 0     # C-ABI calls made through this module
kernel_launches = 0  # CUDA kernels those calls launched (bench.py reports it as gpu_launches)
# kernels launched per entry point (csrc/*.cu); 1 unless listed
_KERNELS_PER_CALL = {"cg_cutouts_fwd": 4, "cg_cutouts_bwd": 4, "cg_ms_ssim_dissimilarity_fwd_bwd": 17, "cg_attention_bwd": 3, "cg_grad_finalize": 2, "cg_any_nan": 2, "cg_dynamic_threshold": 5, "cg_groupnorm_nhwc_fwd": 3, "cg_groupnorm_nhwc_bwd": 3}
# longest sequence of the tcgen05 attention kernels (ATTN_TC_MAX_T in csrc/tcgen05.cuh); cg_attention_fwd / _bwd run longer ones
# on the mma.sync kernels, and cg_attention_causal_fwd refuses them
ATTN_TC_MAX_T = 272


class ClipGuideError(RuntimeError):
    pass


def exported_symbols():
    return sorted(_SIGNATURES)


def load():
    """Load the library (once).  Raises if it is missing: the product has no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ClipGuideError(
            "%s not found: build it with `make -C clip_diffusion_b200/csrc` (or __graft_entry__.build()). "
            "clip_diffusion_b200 has no CPU or eager fallback." % LIB_PATH
        )
    lib = C.CDLL(LIB_PATH)
    missing = []
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            missing.append(name)  # stale build: calling it raises below, loudly
            continue
        fn.restype = res
        fn.argtypes = args
    lib._cg_missing = missing
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().cg_last_error().decode("utf-8", "replace")
        raise ClipGuideError("%s failed (rc=%d): %s" % (what or "clipguide_b200 call", rc, msg))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# bench.py sets this to a list to time C-ABI calls with CUDA events on the launching stream: entries are
# (entry point name, args, start_event, end_event).  PROFILE_NAMES restricts it to the entry points of interest.
PROFILE = None
PROFILE_NAMES = ()


def call(name, *args):
    """Call an int-returning entry point on the current stream (appended as last argument)."""
    global launch_count, kernel_launches
    lib = load()
    if name in lib._cg_missing:
        raise ClipGuideError("%s is not exported by %s: rebuild the library (stale build)" % (name, LIB_PATH))
    prof = PROFILE is not None and name in PROFILE_NAMES
    if prof:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    rc = getattr(lib, name)(*args, stream_ptr())
    if prof:
        ev1.record()
        PROFILE.append((name, args, ev0, ev1))
    launch_count += 1
    if name == "cg_attention_bwd" and args[5] <= ATTN_TC_MAX_T:
        kernel_launches += 1  # one persistent tcgen05 kernel (delta included); the mma.sync path beyond T = 272 is delta + dQ + dK/dV
    else:
        kernel_launches += _KERNELS_PER_CALL.get(name, 1)
    check(rc, name)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise ClipGuideError("clip_diffusion_b200 ops need CUDA tensors (no CPU fallback); got a %s tensor" % t.device)
