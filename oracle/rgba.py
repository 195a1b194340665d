"""Reference of an RGBA call (``MZ_FLAG_RGBA``): the definition the kernels implement.  TEST INFRASTRUCTURE ONLY.

An RGBA image (B, 4, H, W) holds colour 0..2, then a straight (not premultiplied) alpha.  The colour goes through the
network exactly as a 3-channel image does; the network never reads the alpha.  The alpha is the global skip's
resampling alone -- ``bicubic_upsample_ref`` (Keys cubic, A = -0.75, half-pixel centres, clamped taps) -- clamped to
[0, 1] where ``upscale`` clamps.  See ``MZ_FLAG_RGBA`` in include/mewzoom_b200.h for the contract this restates.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor

from .mewzoom_oracle import OracleMewZoom, bicubic_upsample_ref


@torch.inference_mode()
def upscale_rgba_ref(model: OracleMewZoom, x: Tensor, c: Optional[Tensor] = None, clamp: bool = True) -> Tensor:
    """x (B,4,H,W) -> (B,4,rH,rW): the model on x[:, :3] (``upscale`` with clamp=True, ``forward`` without), then
    bicubic_upsample_ref of x[:, 3:], clamped to [0, 1] when clamp is set."""
    assert x.dim() == 4 and x.shape[1] == 4, f"Expected an RGBA image (B, 4, H, W), got {tuple(x.shape)}."
    x = x.float()
    colour = model.upscale(x[:, :3], c) if clamp else model.forward(x[:, :3], c)
    alpha = bicubic_upsample_ref(x[:, 3:], model.upscale_ratio)
    return torch.cat([colour, alpha.clamp(0, 1) if clamp else alpha], dim=1)
