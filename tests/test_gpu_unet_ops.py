"""GPU: the 0.3.0 U-Net operators (ultrazoom_b200.unet -> csrc/unet_tc.cu, unet_ops.cu + the tcgen05 convolutions) against
the fixtures computed by the reference's OWN leaf classes (tests/golden/unet_ops.npz; SURVEY.md 8(f) rank 3) and against
the pinned oracle at further shapes.  Operators with fp32 arithmetic end to end (shuffle, crop, assessor, and the fp32
twins of mix and crush) match to 1e-5; the default mix / crush run their GEMM on tcgen05 with tf32 operands (fp32 words
truncated to a 10-bit mantissa, fp32 accumulation) and are held to 3e-3 x the output scale; blocks that contain 3x3
convolutions run those on fp16 tensor-core operands and are held to 6e-3 x the output scale (the same budget per
convolution as the flat path's stated tolerances)."""
import numpy as np
import pytest
import torch

from oracle import unet_oracle as U
from tests.helpers import GOLDEN
from tests.test_gpu_fp16_range import same16

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def gold():
    z = np.load(GOLDEN + "/unet_ops.npz")
    return {k: torch.from_numpy(z[k]) for k in z.files}


def _sd(gold, prefix):
    return {k[len(prefix) + 3:]: v for k, v in gold.items() if k.startswith(prefix + "/w:")}


TF32_TOL = 3e-3      # x the output scale: K <= 1536 products of operands truncated to 10 mantissa bits


def _close(got_nhwc, want_nchw, tol):
    from ultrazoom_b200.unet import to_nchw

    got = to_nchw(got_nhwc).cpu()
    assert got.shape == want_nchw.shape, (got.shape, want_nchw.shape)
    err = (got - want_nchw).abs().max().item()
    assert err <= tol, err


def test_mix_crush_shuffle_crop_assessor_match_reference_fixtures(dev, gold):
    from ultrazoom_b200 import unet as N

    m = N.AdaptiveResidualMix(16)
    m.load_state_dict(_sd(gold, "mix"))
    for math, tol in (("tf32", TF32_TOL * gold["mix/out"].abs().max().item()), ("fp32", 1e-5)):
        m.math = math
        _close(m.forward(N.to_nhwc(gold["mix/in0"]).to(dev), N.to_nhwc(gold["mix/in1"]).to(dev)), gold["mix/out"], tol)
    for f in (2, 3, 4):
        c = N.PixelCrush(16, 32, f)
        c.load_state_dict(_sd(gold, f"crush{f}"))
        for math, tol in (("tf32", TF32_TOL * gold[f"crush{f}/out"].abs().max().item()), ("fp32", 1e-5)):
            c.math = math
            _close(c.forward(N.to_nhwc(gold[f"crush{f}/in0"]).to(dev)), gold[f"crush{f}/out"], tol)
    for name in ("crop_smaller", "crop_larger", "crop_mixed"):
        size = tuple(int(v) for v in gold[name + "/size"])
        _close(N.crop_feature_maps(N.to_nhwc(gold[name + "/in0"]).to(dev), size), gold[name + "/out"], 0.0)
    q = N.QualityAssessor(32, 3)
    q.load_state_dict(_sd(gold, "quality"))
    got = q.forward(N.to_nhwc(gold["quality/in0"]).to(dev)).cpu()
    assert got.shape == (2, 3) and (got - gold["quality/out"]).abs().max().item() <= 1e-5
    z = np.load(GOLDEN + "/leaf_ops.npz")                                 # PixelShuffle known answers, r = 2, 3, 4
    for r in (2, 3, 4):
        x = torch.from_numpy(z[f"shuffle_in_r{r}"])
        _close(N.pixel_shuffle_nhwc(N.to_nhwc(x).to(dev), r), torch.from_numpy(z[f"shuffle_out_r{r}"]), 0.0)


def test_blocks_with_convolutions_match_reference_fixtures(dev, gold):
    from ultrazoom_b200 import unet as N

    up = N.SubpixelConv2d(32, 16, 2)
    up.load_state_dict(_sd(gold, "subpixel"))
    _close(up.forward(N.to_nhwc(gold["subpixel/in0"]).to(dev)), gold["subpixel/out"], 6e-3 * gold["subpixel/out"].abs().max().item())
    blk = N.EncoderBlock(16, 2)
    blk.load_state_dict(_sd(gold, "encoder_block"))
    _close(blk.forward(N.to_nhwc(gold["encoder_block/in0"]).to(dev)), gold["encoder_block/out"],
           6e-3 * gold["encoder_block/out"].abs().max().item())
    sr = N.SR2XBlock(16, 2, 16)
    sr.load_state_dict(_sd(gold, "sr2x"))
    _close(sr.forward(N.to_nhwc(gold["sr2x/in0"]).to(dev)), gold["sr2x/out"], 6e-3 * gold["sr2x/out"].abs().max().item())
    head = N.SuperResolver(16, 2, 4)
    head.load_state_dict(_sd(gold, "super_resolver"))
    got = head.forward(N.to_nhwc(gold["super_resolver/in0"]).to(dev))
    assert tuple(got.shape) == (1, 20, 28, 3)
    _close(got, gold["super_resolver/out"], 1.2e-2 * gold["super_resolver/out"].abs().max().item())


@pytest.mark.parametrize("C,shape", [(16, (1, 1, 1)), (48, (2, 37, 61)), (96, (1, 20, 130)), (32, (3, 5, 257)),
                                     (20, (1, 9, 70)), (192, (1, 12, 140)), (384, (1, 6, 40))])
def test_mix_and_crush_against_the_oracle_at_other_shapes(dev, C, shape):
    """Ragged rows (tiles of 128 pixels with a tail, warps past the end of a row), channel counts that are not a multiple
    of the 32-channel chunk (zero-filled by the TMA), weight matrices too large to stay resident (192 / 384 channels: the
    output channels are sliced over CTAs), both arithmetic forms."""
    from ultrazoom_b200 import unet as N

    g = torch.Generator().manual_seed(C + sum(shape))
    B, H, W = shape
    x, z = torch.randn(B, C, H, W, generator=g), torch.randn(B, C, H, W, generator=g)
    w = torch.randn(C, 2 * C, 1, 1, generator=g) / (2 * C) ** 0.5
    for a in (-2.0, 0.0, 1.5):
        alpha = torch.tensor(a)
        want = U.adaptive_residual_mix(x, z, w, alpha)
        for math, tol in (("tf32", TF32_TOL * want.abs().max().item()), ("fp32", 2e-5)):
            _close(N.adaptive_residual_mix(N.to_nhwc(x).to(dev), N.to_nhwc(z).to(dev), w, alpha, math), want, tol)
    for f in (2, 3, 4):
        if H < f or W < f:
            with pytest.raises(AssertionError):
                N.pixel_crush(N.to_nhwc(x).to(dev), torch.randn(C, C, f, f), f)
            continue
        wc = torch.randn(2 * C, C, f, f, generator=g) / (f * f * C) ** 0.5
        want = U.pixel_crush(x, wc, f)
        for math, tol in (("tf32", TF32_TOL * want.abs().max().item()), ("fp32", 2e-5)):
            _close(N.pixel_crush(N.to_nhwc(x).to(dev), wc, f, math), want, tol)
    wq, bq = torch.randn(3, C, 3, 3, generator=g) / (9 * C) ** 0.5, torch.randn(3, generator=g)
    got = N.quality_assessor(N.to_nhwc(x).to(dev), wq, bq).cpu()
    assert (got - U.quality_assessor(x, wq, bq)).abs().max().item() <= 2e-5
    for size in ((H + 3, W - 1 if W > 1 else 1), (max(1, H - 2), W + 4)):
        _close(N.crop_feature_maps(N.to_nhwc(x).to(dev), size), U.crop_feature_maps(x, size), 0.0)


@pytest.mark.parametrize("math", ["tf32", "fp32"])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_sixteen_bit_shadow_is_the_rounded_output(dev, math, dt):
    """Both operators (and the pixel shuffle) can also write the 16-bit copy the tcgen05 convolutions read: exactly
    round16(out), i.e. ``out.to(dt)`` -- beyond the fp16 range too, where that is +-inf (the shadow replaces the cast, it
    does not clip); NaN compared by NaN-ness.  Many tiles per CTA (more tiles than SMs) and a deterministic result."""
    from ultrazoom_b200 import unet as N

    g = torch.Generator().manual_seed(11)
    C = 48
    x, z = torch.randn(2, 150, 301, C, generator=g).to(dev), torch.randn(2, 150, 301, C, generator=g).to(dev)
    w = torch.randn(C, 2 * C, 1, 1, generator=g) / (2 * C) ** 0.5
    out, sh = N.adaptive_residual_mix(x, z, w, torch.tensor(0.3), math, shadow=dt)
    assert sh.dtype == dt and torch.equal(sh, out.to(dt))
    assert torch.equal(out, N.adaptive_residual_mix(x, z, w, torch.tensor(0.3), math))
    want = U.adaptive_residual_mix(N.to_nchw(x).cpu(), N.to_nchw(z).cpu(), w, torch.tensor(0.3))
    _close(out, want, TF32_TOL * want.abs().max().item() if math == "tf32" else 2e-5)
    wc = torch.randn(96, C, 2, 2, generator=g) / (4 * C) ** 0.5
    out, sh = N.pixel_crush(x, wc, 2, math, shadow=dt)
    assert tuple(out.shape) == (2, 75, 150, 96) and torch.equal(sh, out.to(dt))
    want = U.pixel_crush(N.to_nchw(x).cpu(), wc, 2)
    _close(out, want, TF32_TOL * want.abs().max().item() if math == "tf32" else 2e-5)
    # beyond the fp16 range: outputs up to ~1e5, a few inputs at the edge, inf and NaN
    xw, zw = x * 3e4, z * 3e4
    xw[0, 7, 11, :8] = torch.tensor([float("inf"), -float("inf"), float("nan"), 1e5, -65519.99, 65520.0, 3e38, 2.0**-25])
    out, sh = N.adaptive_residual_mix(xw, zw, w, torch.tensor(0.3), math, shadow=dt)
    assert float(out.abs().nan_to_num(0, 0, 0).max()) > 65520
    same16(sh, out.to(dt))
    out, sh = N.pixel_crush(xw, wc, 2, math, shadow=dt)
    assert float(out.abs().nan_to_num(0, 0, 0).max()) > 65520
    same16(sh, out.to(dt))
    out = N.pixel_shuffle_nhwc(xw, 2, shadow=dt)
    same16(out._mz16[0], out.to(dt))


@pytest.mark.parametrize("C,hidden_ratio,shape", [(96, 2, (1, 24, 150)), (192, 2, (1, 10, 140)), (384, 2, (1, 6, 40)), (64, 4, (2, 9, 70))])
def test_blocks_at_the_widths_of_the_default_unet(dev, C, hidden_ratio, shape):
    """The stage widths of the reference's default U-Net (48 / 96 / 192 / 384 channels): convolutions wider than one launch
    (more than 256 hidden channels, more than 128 output channels -- e.g. SubpixelConv2d's C -> 4C) run as slices of output
    channels; blocks against the pinned oracle on the same weights."""
    from ultrazoom_b200 import unet as N

    torch.manual_seed(C + hidden_ratio)
    B, H, W = shape
    x = torch.randn(B, C, H, W)
    blk = N.SR2XBlock(C, hidden_ratio, C // 2)
    sd = {k: v.detach().clone() for k, v in blk.state_dict().items()}
    want = U.sr2x_block(x, sd)
    got = blk.to(dev).forward(N.to_nhwc(x).to(dev))
    assert tuple(got.shape) == (B, 2 * H, 2 * W, C // 2)
    _close(got, want, 8e-3 * want.abs().max().item())
    ib = N.InvertedBottleneck(C, hidden_ratio)
    want = U.inverted_bottleneck(x, ib.conv1.weight.detach(), ib.conv2.weight.detach())
    _close(ib.to(dev).forward(N.to_nhwc(x).to(dev)), want, 6e-3 * want.abs().max().item())
    # the block's output carries its 16-bit copy for the next convolution; an in-place edit retires it
    y = blk.refiner.forward(N.to_nhwc(x).to(dev))
    assert torch.equal(N._operand(y, torch.float16), y.to(torch.float16)) and N._operand(y, torch.float16) is y._mz16[0]
    y.mul_(0.5)
    assert N._operand(y, torch.float16) is not y._mz16[0] and torch.equal(N._operand(y, torch.float16), y.to(torch.float16))
    again = ib.forward(N.to_nhwc(x).to(dev))                              # packed banks come from the cache now
    assert torch.equal(again, ib.forward(N.to_nhwc(x).to(dev)))
    with torch.no_grad():
        ib.conv2.weight.mul_(2.0)                                        # ... and are re-packed when a weight changes
    _close(ib.forward(N.to_nhwc(x).to(dev)), 2.0 * want, 6e-3 * 2.0 * want.abs().max().item())


@pytest.mark.parametrize("how", ["stream", "resident"])
def test_streamed_and_resident_weights_agree(dev, how, monkeypatch):
    """The weight slice either stays in shared memory or its chunks travel with the activation chunks (deep K): the same
    UMMAs in the same order, so the two forms are bit-identical."""
    from ultrazoom_b200 import unet as N

    g = torch.Generator().manual_seed(3)
    x, z = torch.randn(1, 33, 200, 64, generator=g).to(dev), torch.randn(1, 33, 200, 64, generator=g).to(dev)
    w = torch.randn(64, 128, 1, 1, generator=g) / 128 ** 0.5
    wc = torch.randn(80, 64, 3, 3, generator=g) / (9 * 64) ** 0.5
    base_mix, base_crush = N.adaptive_residual_mix(x, z, w, torch.tensor(0.1)), N.pixel_crush(x, wc, 3)
    monkeypatch.setenv("MZ_SG_WEIGHTS", how)
    assert torch.equal(N.adaptive_residual_mix(x, z, w, torch.tensor(0.1)), base_mix)
    assert torch.equal(N.pixel_crush(x, wc, 3), base_crush)
    want = U.pixel_crush(N.to_nchw(x).cpu(), wc, 3)
    _close(base_crush, want, TF32_TOL * want.abs().max().item())


@pytest.mark.parametrize("math", ["tf32", "fp32"])
def test_padded_channel_pitch_through_the_c_abi(dev, math):
    """Feature maps whose channel pitch exceeds the channel count (the C ABI's pitch arguments): the crush then reads one
    K segment per (i, j) tap instead of one per input row; the mix reads and writes the logical channels only."""
    from ultrazoom_b200 import _native
    from ultrazoom_b200 import unet as N

    lib = _native.load()
    g = torch.Generator().manual_seed(17)
    B, H, W, C, P, Co, Po = 2, 21, 150, 40, 48, 72, 80
    code = _native.MATH_TF32 if math == "tf32" else _native.MATH_FP32
    xp = torch.randn(B, H, W, P, generator=g).to(dev)
    zp = torch.randn(B, H, W, P, generator=g).to(dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for f in (2, 3):
        wc = torch.randn(Co, C, f, f, generator=g) / (f * f * C) ** 0.5
        wt = wc.permute(0, 2, 3, 1).reshape(Co, f * f * C).contiguous().to(dev)
        out = torch.full((B, H // f, W // f, Po), 7.0, device=dev)
        _native.check(lib.mz_pixel_crush(xp.data_ptr(), wt.data_ptr(), out.data_ptr(), None, B, H, W, C, Co, f, P, Po,
                                         _native.DTYPE_F16, code, stream))
        want = U.pixel_crush(N.to_nchw(xp[..., :C].contiguous()).cpu(), wc, f)
        _close(out[..., :Co].contiguous(), want, TF32_TOL * want.abs().max().item() if math == "tf32" else 2e-5)
        assert bool((out[..., Co:] == 7.0).all())                       # the padding channels are left alone
    w = torch.randn(C, 2 * C, 1, 1, generator=g) / (2 * C) ** 0.5
    out = torch.full((B, H, W, P), 7.0, device=dev)
    _native.check(lib.mz_adaptive_mix(xp.data_ptr(), zp.data_ptr(), w.reshape(C, 2 * C).contiguous().to(dev).data_ptr(), 0.4,
                                      out.data_ptr(), None, B * H * W, C, P, _native.DTYPE_F16, code, stream))
    want = U.adaptive_residual_mix(N.to_nchw(xp[..., :C].contiguous()).cpu(), N.to_nchw(zp[..., :C].contiguous()).cpu(), w,
                                   torch.tensor(0.4))
    _close(out[..., :C].contiguous(), want, TF32_TOL * want.abs().max().item() if math == "tf32" else 2e-5)
    assert bool((out[..., C:] == 7.0).all())


def test_argument_checks_and_no_cpu_fallback(dev):
    from ultrazoom_b200 import unet as N

    with pytest.raises(AssertionError, match="Crush factor"):
        N.PixelCrush(16, 32, 5)                                          # reference model.py:853-857
    with pytest.raises(AssertionError, match="Upscale ratio"):
        N.SuperResolver(16, 2, 3)                                        # model.py:939-943
    with pytest.raises(AssertionError, match="Hidden ratio"):
        N.InvertedBottleneck(16, 3)                                      # model.py:738
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        N.adaptive_residual_mix(torch.rand(1, 2, 2, 16), torch.rand(1, 2, 2, 16), torch.rand(16, 32, 1, 1), torch.tensor(0.0))
    with pytest.raises(AssertionError):
        N.adaptive_residual_mix(torch.rand(1, 2, 2, 16, device=dev), torch.rand(1, 2, 3, 16, device=dev),
                                torch.rand(16, 32, 1, 1), torch.tensor(0.0))
