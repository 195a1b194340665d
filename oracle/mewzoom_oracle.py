"""fp32 CPU restatement of the MewZoom (0.2.x-style) inference forward pass.

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.

Parity status
-------------
* bicubic / stem / InvertedBottleneck / ResidualConnection / SubpixelConv2d /
  clamp: restated from ``/root/reference/src/ultrazoom/model.py`` and PINNED by
  ``tests/golden/*.npz`` -- fixtures produced by ``oracle/make_golden.py`` from
  the reference's own importable leaf classes (the reference's ``MewZoom``
  itself cannot be constructed: ``model.py:356-358`` raises ``NameError``).
* control module (``src/ultrazoom/control.py``): ABSENT from the reference
  snapshot.  Its form here (per-layer FiLM: ``Linear(F, 2*hC)`` -> (1+gamma)*h +
  beta, applied between conv1 and SiLU) is OUR specification (SURVEY.md
  Appendix C).  **Parity unpinned** for that one piece; the fixtures pin our
  restatement of it, not the upstream's.

Reference call sites followed (file:line relative to /root/reference):
  MewZoom.forward            src/ultrazoom/model.py:149-164
  MewZoom.upscale            src/ultrazoom/model.py:166-179   (clamp :177)
  Upsample(bicubic)          src/ultrazoom/model.py:71,156
  FanOutProjection           src/ultrazoom/model.py:212-242   (1x1 conv + bias :224)
  InvertedBottleneck         src/ultrazoom/model.py:731-778   (3x3, pad 1, bias=False)
  ResidualConnection         src/ultrazoom/model.py:781-792
  SubpixelConv2d             src/ultrazoom/model.py:885-930   (3x3 conv -> PixelShuffle)
  ControlVector usage        README.md:94,118-122,181-185; validate.py:73-94
"""
from __future__ import annotations

import math
from typing import Optional

import torch
from torch import Tensor, nn
from torch.nn import functional as F

# README.md:35-42 -- the published model table (channels, encoder layers).
MODEL_CONFIGS = {
    "MewZoom-2X": dict(upscale_ratio=2, num_channels=48, hidden_ratio=2, num_encoder_layers=20, control_features=0),
    "MewZoom-3X": dict(upscale_ratio=3, num_channels=54, hidden_ratio=2, num_encoder_layers=30, control_features=0),
    "MewZoom-4X": dict(upscale_ratio=4, num_channels=96, hidden_ratio=2, num_encoder_layers=40, control_features=0),
    "MewZoom-2X-Ctrl": dict(upscale_ratio=2, num_channels=48, hidden_ratio=2, num_encoder_layers=20, control_features=3),
    "MewZoom-3X-Ctrl": dict(upscale_ratio=3, num_channels=54, hidden_ratio=2, num_encoder_layers=30, control_features=3),
    "MewZoom-4X-Ctrl": dict(upscale_ratio=4, num_channels=96, hidden_ratio=2, num_encoder_layers=40, control_features=3),
}


class OracleControlVector:
    """README.md:94,118-122 -- three floats in [0, 1]; order README.md:181-185."""

    def __init__(self, gaussian_blur: float = 0.0, gaussian_noise: float = 0.0, jpeg_compression: float = 0.0):
        for name, v in (("gaussian_blur", gaussian_blur), ("gaussian_noise", gaussian_noise),
                        ("jpeg_compression", jpeg_compression)):
            assert 0.0 <= v <= 1.0, f"{name} must be between 0 and 1, {v} given."
        self.gaussian_blur = float(gaussian_blur)
        self.gaussian_noise = float(gaussian_noise)
        self.jpeg_compression = float(jpeg_compression)

    def to_tensor(self) -> Tensor:
        return torch.tensor([self.gaussian_blur, self.gaussian_noise, self.jpeg_compression], dtype=torch.float32)


# --------------------------------------------------------------------------- #
# Closed-form leaf operators (no torch.nn) -- used to cross-check torch's own  #
# kernels in the CPU tests and as the known-answer reference for the CUDA      #
# bicubic / pixel-shuffle kernels.                                             #
# --------------------------------------------------------------------------- #

_CUBIC_A = -0.75  # aten upsample_bicubic2d; Upsample(mode="bicubic") model.py:71


def _cubic_weights(t: float) -> list[float]:
    a = _CUBIC_A
    def near(x):  # |x| <= 1
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0
    def far(x):   # 1 < |x| < 2
        return ((a * x - 5.0 * a) * x + 8.0 * a) * x - 4.0 * a
    return [far(t + 1.0), near(t), near(1.0 - t), far(2.0 - t)]


def bicubic_phase_table(r: int) -> list[tuple[int, list[float]]]:
    """Per output phase p = ox mod r: (base tap offset ix - ox//r, 4 weights).
    align_corners=False, src = (ox + 0.5)/r - 0.5 (SURVEY.md Appendix A.1)."""
    out = []
    for p in range(r):
        src = (p + 0.5) / r - 0.5
        ix = math.floor(src)
        t = src - ix
        out.append((ix, _cubic_weights(t)))
    return out


def bicubic_upsample_ref(x: Tensor, r: int) -> Tensor:
    """Pure index-arithmetic bicubic zoom (float64 accumulate), clamped tap
    indices, no antialias, no output clamp.  x: (B,3,H,W), on any device (the result stays there)."""
    B, C, H, W = x.shape
    dev = x.device
    tab = bicubic_phase_table(r)
    xd = x.double()
    # horizontal pass
    ox = torch.arange(W * r, device=dev)
    base_x = ox // r + torch.tensor([tab[p][0] for p in range(r)], device=dev)[ox % r]
    wx = torch.tensor([tab[p][1] for p in range(r)], dtype=torch.float64, device=dev)[ox % r]  # (Wr,4)
    tmp = torch.zeros(B, C, H, W * r, dtype=torch.float64, device=dev)
    for k in range(4):
        idx = (base_x - 1 + k).clamp(0, W - 1)
        tmp += xd[..., idx] * wx[:, k]
    oy = torch.arange(H * r, device=dev)
    base_y = oy // r + torch.tensor([tab[p][0] for p in range(r)], device=dev)[oy % r]
    wy = torch.tensor([tab[p][1] for p in range(r)], dtype=torch.float64, device=dev)[oy % r]
    out = torch.zeros(B, C, H * r, W * r, dtype=torch.float64, device=dev)
    for k in range(4):
        idx = (base_y - 1 + k).clamp(0, H - 1)
        out += tmp[:, :, idx, :] * wy[:, k][None, None, :, None]
    return out.float()


def pixel_shuffle_ref(z: Tensor, r: int) -> Tensor:
    """out[b,c,h*r+i,w*r+j] = in[b, c*r*r + i*r + j, h, w]  (model.py:911,928)."""
    B, N, H, W = z.shape
    C = N // (r * r)
    return z.view(B, C, r, r, H, W).permute(0, 1, 4, 2, 5, 3).reshape(B, C, H * r, W * r)


# --------------------------------------------------------------------------- #
# The module                                                                   #
# --------------------------------------------------------------------------- #


class _Stem(nn.Module):  # FanOutProjection model.py:212-242
    def __init__(self, cin: int, cout: int):
        super().__init__()
        assert cin > 0, "Input channels must be greater than 0."
        assert cin < cout, "Output channels must be greater than input channels."
        self.conv = nn.Conv2d(cin, cout, kernel_size=1)


class _ConvNet(nn.Module):  # InvertedBottleneck model.py:731-778
    def __init__(self, c: int, h: int):
        super().__init__()
        assert c > 0, "Number of channels must be greater than 0."
        assert h in {1, 2, 4}, "Hidden ratio must be either 1, 2, or 4."
        self.conv1 = nn.Conv2d(c, h * c, kernel_size=3, padding=1, bias=False)
        self.conv2 = nn.Conv2d(h * c, c, kernel_size=3, padding=1, bias=False)


class _Control(nn.Module):  # OUR spec (control.py absent) -- SURVEY.md Appendix C
    def __init__(self, features: int, hidden_channels: int):
        super().__init__()
        self.linear = nn.Linear(features, 2 * hidden_channels, bias=True)


class _Block(nn.Module):  # EncoderBlock model.py:487-511 with plain ResidualConnection
    def __init__(self, c: int, h: int, features: int):
        super().__init__()
        self.convnet = _ConvNet(c, h)
        if features > 0:
            self.control = _Control(features, h * c)


class _Head(nn.Module):  # SubpixelConv2d model.py:885-930
    def __init__(self, cin: int, cout: int, r: int):
        super().__init__()
        assert r in {2, 3, 4}, "Upscale ratio must be either 2, 3, or 4."
        self.conv = nn.Conv2d(cin, cout * r * r, kernel_size=3, stride=1, padding=1, bias=False)


class OracleMewZoom(nn.Module):
    """forward(x[, c]) / upscale(x[, c]) exactly as SURVEY.md Appendix C."""

    AVAILABLE_UPSCALE_RATIOS = {2, 3, 4}

    def __init__(self, upscale_ratio: int, num_channels: int, hidden_ratio: int,
                 num_encoder_layers: int, control_features: int = 0):
        super().__init__()
        assert upscale_ratio in self.AVAILABLE_UPSCALE_RATIOS, (
            f"Upscale ratio must be one of {self.AVAILABLE_UPSCALE_RATIOS}, but got {upscale_ratio}.")
        assert num_encoder_layers > 0, "Number of encoder layers must be greater than 0."
        assert control_features >= 0
        self.upscale_ratio = upscale_ratio
        self.num_channels = num_channels
        self.hidden_ratio = hidden_ratio
        self.num_encoder_layers = num_encoder_layers
        self.control_features = control_features
        self.stem = _Stem(3, num_channels)
        self.encoder = nn.ModuleList(
            [_Block(num_channels, hidden_ratio, control_features) for _ in range(num_encoder_layers)])
        self.head = _Head(num_channels, 3, upscale_ratio)

    def _check_c(self, x: Tensor, c: Optional[Tensor]) -> Optional[Tensor]:
        if self.control_features == 0:
            assert c is None, "This model has no control modules; c must be None."
            return None
        assert c is not None, "Control vector c is required for control models."
        if c.dim() == 1:
            c = c.unsqueeze(0)
        assert c.shape[-1] == self.control_features, (
            f"Expected {self.control_features} control features, got {c.shape[-1]}.")
        assert c.shape[0] in (1, x.shape[0]), "Batch size of c must match x."
        return c.expand(x.shape[0], -1).to(torch.float32)

    def forward(self, x: Tensor, c: Optional[Tensor] = None) -> Tensor:
        c = self._check_c(x, c)
        r = self.upscale_ratio
        s = F.interpolate(x, scale_factor=r, mode="bicubic")                 # model.py:71,156
        z = F.conv2d(x, self.stem.conv.weight, self.stem.conv.bias)          # model.py:224
        for blk in self.encoder:
            h = F.conv2d(z, blk.convnet.conv1.weight, padding=1)             # model.py:742-744
            if c is not None:
                g = F.linear(c, blk.control.linear.weight, blk.control.linear.bias)
                hc = h.shape[1]
                h = (1.0 + g[:, :hc])[:, :, None, None] * h + g[:, hc:][:, :, None, None]
            h = F.silu(h)                                                    # model.py:750,775
            d = F.conv2d(h, blk.convnet.conv2.weight, padding=1)             # model.py:746-748
            assert z.shape == d.shape, "Input and residual must have the same shape."
            z = z + d                                                        # model.py:789-792
        u = F.pixel_shuffle(F.conv2d(z, self.head.conv.weight, padding=1), r)  # model.py:926-930
        assert s.shape == u.shape, "Input and residual must have the same shape."
        return s + u                                                         # model.py:162

    @torch.inference_mode()
    def upscale(self, x: Tensor, c: Optional[Tensor] = None) -> Tensor:
        return torch.clamp(self.forward(x, c), 0, 1)                         # model.py:177

    @torch.inference_mode()
    def residual(self, x: Tensor, c: Optional[Tensor] = None) -> Tensor:
        """forward() minus the bicubic skip -- the degeneracy guard uses its rms."""
        return self.forward(x, c) - F.interpolate(x, scale_factor=self.upscale_ratio, mode="bicubic")


def make_oracle(name_or_cfg, seed: int = 0) -> OracleMewZoom:
    """Deterministic random-init oracle: torch.manual_seed(seed) then construct
    (PyTorch default Conv2d/Linear init -- NOT initialize_weights(), SURVEY.md 0.4)."""
    cfg = MODEL_CONFIGS[name_or_cfg] if isinstance(name_or_cfg, str) else dict(name_or_cfg)
    gen_state = torch.random.get_rng_state()
    try:
        torch.manual_seed(seed)
        m = OracleMewZoom(**cfg)
        if cfg.get("control_features", 0) > 0:
            # The default Linear init on fan_in=3 gives |gamma|,|beta| up to 0.58 -- keep it:
            # it makes the control path numerically visible in parity tests.
            pass
    finally:
        torch.random.set_rng_state(gen_state)
    return m.eval()


def psnr(a: Tensor, b: Tensor) -> float:
    """10*log10(1/MSE) on [0,1] data (PeakSignalNoiseRatio(data_range=1.0), pretrain.py:209)."""
    mse = torch.mean((a.double() - b.double()) ** 2).item()
    return float("inf") if mse == 0 else 10.0 * math.log10(1.0 / mse)


def max_abs_err(a: Tensor, b: Tensor) -> float:
    return (a.double() - b.double()).abs().max().item()


def residual_rms(model: OracleMewZoom, x: Tensor, c: Optional[Tensor] = None) -> float:
    return model.residual(x, c).double().pow(2).mean().sqrt().item()
