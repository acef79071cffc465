"""Hot-path helpers of clip_diffusion/utils/functional.py (:16-18 CLIP_NORMALIZE, :74-76 L2_norm,
:97-102 embed_image, :105-111 set_seed) with the same names and argument meaning."""
import random

import numpy as np
import torch
from torch.nn import functional as F

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)


def CLIP_NORMALIZE(image):
    """(x - mean) / std per channel (functional.py:16-18), as a plain differentiable torch op for callers that
    need the normalised tensor itself; embed_image fuses it into the patch kernel instead."""
    mean = torch.tensor(CLIP_MEAN, device=image.device, dtype=image.dtype).view(1, 3, 1, 1)
    std = torch.tensor(CLIP_STD, device=image.device, dtype=image.dtype).view(1, 3, 1, 1)
    return (image - mean) / std


def L2_norm(input, dim=-1):
    """functional.py:74-76"""
    return F.normalize(input, dim=dim)


def embed_image(clip_model, image, clip_normalize=True, L2_normalize=False):
    """functional.py:97-102: [N,3,res,res] image -> [N,E] fp32 embedding, differentiable w.r.t. ``image``."""
    fused = getattr(clip_model, "encode_image_normalized_input", None)
    if clip_normalize and fused is not None:
        image_embedding = fused(image)
    else:
        if clip_normalize:
            image = CLIP_NORMALIZE(image)
        image_embedding = clip_model.encode_image(image).float()
    return image_embedding if not L2_normalize else L2_norm(image_embedding, dim=-1)


def embed_text(clip_model, text, L2_normalize=False):
    """functional.py:91-94: token ids [P, 77] (clip.tokenize output on the model's device) -> [P, E] fp32.  Runs once per job
    (preprocessing.py:11-24); the B200 models encode on the sm_100a kernels (CLIPModelB200.encode_text), without autograd."""
    text_embedding = clip_model.encode_text(text).float()
    return text_embedding if not L2_normalize else L2_norm(text_embedding, dim=-1)


def set_seed(seed):
    """functional.py:105-111 -- defines what "identical seeds" means for parity runs."""
    np.random.seed(seed)
    random.seed(seed)
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)
    torch.backends.cudnn.deterministic = True
