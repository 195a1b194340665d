"""CPU: the RGBA reference (oracle/rgba.py) states the MZ_FLAG_RGBA contract -- colour through the network on x[:, :3],
the alpha its bicubic resampling alone, clamped where upscale clamps."""
import torch
import torch.nn.functional as F

from oracle import bicubic_upsample_ref
from oracle.rgba import upscale_rgba_ref
from tests.helpers import load_case, oracle_from_case


def _rgba(x):
    """x (B,3,H,W) plus a hard-edged alpha (0 / 1 columns): its bicubic resampling over- and undershoots."""
    B, _, H, W = x.shape
    a = torch.zeros(B, 1, H, W)
    a[..., W // 3: 2 * W // 3] = 1.0
    return torch.cat([x, a], dim=1)


def test_rgba_reference_definition():
    cfg, sd, x, c, _ = load_case("ctrl_2x_c48_l2")
    m = oracle_from_case(cfg, sd)
    r = cfg["upscale_ratio"]
    x4 = _rgba(x)
    y = upscale_rgba_ref(m, x4, c)
    yf = upscale_rgba_ref(m, x4, c, clamp=False)
    assert y.shape == (x.shape[0], 4, x.shape[2] * r, x.shape[3] * r)
    assert torch.equal(y[:, :3], m.upscale(x, c)) and torch.equal(yf[:, :3], m.forward(x, c))
    alpha = bicubic_upsample_ref(x4[:, 3:], r)
    assert torch.equal(yf[:, 3:], alpha) and torch.equal(y[:, 3:], alpha.clamp(0, 1))
    assert yf[:, 3].min() < 0 and yf[:, 3].max() > 1, "hard edges over- and undershoot unclamped"
    # the alpha's resampling is the network's own global skip (F.interpolate bicubic, reference model.py:71,156)
    skip = F.interpolate(x4[:, 3:], scale_factor=r, mode="bicubic")
    assert (yf[:, 3:] - skip).abs().max().item() <= 1e-5


def test_rgba_reference_ignores_the_alpha_for_the_colour():
    cfg, sd, x, c, _ = load_case("ctrl_2x_c48_l2")
    m = oracle_from_case(cfg, sd)
    x4 = _rgba(x)
    x4n = x4.clone()
    x4n[:, 3] = float("nan")
    assert torch.equal(upscale_rgba_ref(m, x4n, c)[:, :3], upscale_rgba_ref(m, x4, c)[:, :3])
