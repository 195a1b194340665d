"""GPU: every kernel behind the C ABI against a CPU fp32 reference computed on the SAME bf16-rounded operands
(torch.nn.functional on the host), including the reference's edge cases: ragged widths (W not a multiple of the
128-pixel tile), heights not a multiple of the patch rows, single-row images, padded channel counts (54 -> 64,
108 -> 112), batch > 1, every upscale ratio, both halo modes, SIMT twin vs tcgen05 kernel."""
import numpy as np
import pytest
import torch
from torch.nn import functional as F

from tests.helpers import GOLDEN

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _ops():
    from ultrazoom_b200 import _native, ops

    assert _native.load().mz_device_count() >= 1, "no sm_100 device: the CUDA path cannot run"
    return ops, _native


# Upsample(bicubic): r = 2, 4 have dyadic weights (bit-level agreement with ATen); for r = 3 ATen evaluates
# t = fp32((ox + 0.5) / 3 - 0.5) per pixel, whose rounding error grows with ox (ulp(W) * slope), while the kernel
# uses the exact 3-phase table -> tolerance 1e-4 (SURVEY.md Appendix A.1).
@pytest.mark.parametrize("r,tol", [(2, 2e-6), (3, 1e-4), (4, 2e-6)])
@pytest.mark.parametrize("shape", [(1, 3, 1, 1), (1, 3, 5, 7), (2, 3, 33, 61), (1, 3, 128, 256), (1, 1, 2, 300)])
def test_bicubic_matches_torch(dev, r, tol, shape):
    ops, _ = _ops()
    x = torch.rand(shape, generator=torch.Generator().manual_seed(sum(shape) + r))
    ref = F.interpolate(x, scale_factor=r, mode="bicubic")
    got = ops.bicubic(x.to(dev), r).cpu()
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= tol


@pytest.mark.parametrize("r,tol", [(2, 2e-6), (3, 2e-6), (4, 2e-6)])
def test_bicubic_matches_reference_fixture(dev, r, tol):
    ops, _ = _ops()
    z = np.load(GOLDEN + "/leaf_ops.npz")
    got = ops.bicubic(torch.from_numpy(z["x"]).to(dev), r).cpu()
    assert (got - torch.from_numpy(z[f"bicubic_r{r}"])).abs().max().item() <= tol


def test_bicubic_rejects_bad_ratio(dev):
    ops, _ = _ops()
    with pytest.raises(AssertionError, match="Upscale ratio"):
        ops.bicubic(torch.rand(1, 3, 4, 4, device=dev), 5)


@pytest.mark.parametrize("C", [16, 48, 54, 96])
def test_stem_pack(dev, C):
    ops, _ = _ops()
    g = torch.Generator().manual_seed(C)
    x = torch.rand(2, 3, 9, 11, generator=g)
    w = torch.randn(C, 3, 1, 1, generator=g) * 0.5
    b = torch.randn(C, generator=g) * 0.1
    ref = F.conv2d(x, w, b).permute(0, 2, 3, 1)
    for dt in (torch.float16, torch.bfloat16):
        zf, zb = ops.stem_pack(x.to(dev), w, b, dtype=dt)
        zf, zb = zf.cpu(), zb.cpu()
        assert (zf[..., :C] - ref).abs().max().item() <= 1e-5
        assert torch.equal(zb, zf.to(dt))                          # shadow copy is exactly round16(zf)
        if zf.shape[-1] > C:
            assert zf[..., C:].abs().max().item() == 0.0           # padded channels stay zero


def test_stem_pack_with_padded_shadow_pitch(dev):
    """48-channel models keep zb at a 64-channel pitch (one 128-byte TMA row per pixel); the pad must be zero."""
    ops, native = _ops()
    assert native.load().mz_zb_pitch(48) in (48, 64) and native.load().mz_zb_pitch(96) == 96
    g = torch.Generator().manual_seed(5)
    x = torch.rand(1, 3, 6, 7, generator=g)
    w, b = torch.randn(48, 3, 1, 1, generator=g) * 0.5, torch.randn(48, generator=g) * 0.1
    ref = F.conv2d(x, w, b).permute(0, 2, 3, 1)
    zf, zb = ops.stem_pack(x.to(dev), w, b, zb_pitch=64)
    assert tuple(zf.shape) == (1, 6, 7, 48) and tuple(zb.shape) == (1, 6, 7, 64)
    assert (zf.cpu() - ref).abs().max().item() <= 1e-5
    assert torch.equal(zb.cpu()[..., :48], zf.cpu().to(torch.float16)) and zb.cpu()[..., 48:].abs().max().item() == 0.0


def test_conv2_writes_shadow_at_padded_pitch(dev):
    ops, native = _ops()
    inp, w, _, zf0, acc = _conv_operands(96, 48, (2, 9, 140), 21, ops, torch.float16)
    wp = ops.pack_conv_weight(w, dev)
    for use_tc in (True, False):
        zf = zf0.to(dev).contiguous()
        zb = ops.conv3x3(inp.to(dev), wp, 1, None, zf, use_tc=use_tc, out_pitch=64).cpu()
        assert tuple(zb.shape) == (2, 9, 140, 64)
        assert torch.equal(zb[..., :48], zf.cpu().to(torch.float16)) and zb[..., 48:].abs().max().item() == 0.0
        assert (zf.cpu() - (zf0 + acc)).abs().max().item() <= 1e-4


def test_control_film(dev):
    ops, _ = _ops()
    g = torch.Generator().manual_seed(4)
    L, B, Fc, hC = 3, 2, 3, 108
    w, bb, c = torch.randn(L, 2 * hC, Fc, generator=g), torch.randn(L, 2 * hC, generator=g), torch.rand(B, Fc, generator=g)
    gl = torch.einsum("bf,lnf->lbn", c, w) + bb[:, None, :]
    for cc in (c, c[:1]):                                           # per-image and broadcast control vectors
        film = ops.control_film(cc.to(dev), w.to(dev), bb.to(dev), B).cpu()
        ref = gl if cc.shape[0] == B else gl[:, :1].expand(-1, B, -1)
        assert (film[:, :, 0, :hC] - (1 + ref[..., :hC])).abs().max().item() <= 1e-5
        assert (film[:, :, 1, :hC] - ref[..., hC:]).abs().max().item() <= 1e-5
        assert bool((film[:, :, 0, hC:] == 1).all()) and bool((film[:, :, 1, hC:] == 0).all())
    with pytest.raises(AssertionError, match="Batch size"):
        ops.control_film(torch.rand(3, Fc, device=dev), w.to(dev), bb.to(dev), B)


DTYPES = [torch.float16, torch.bfloat16]


def _ulp(dt):
    return 2.0 ** -11 if dt == torch.float16 else 2.0 ** -8     # half an ulp relative to the value


def _conv_operands(cin, cout, shape, seed, ops, dt):
    g = torch.Generator().manual_seed(seed)
    B, H, W = shape
    cin_p, cout_p = ops.padded_channels(cin), ops.padded_channels(cout)
    inp = torch.zeros(B, H, W, cin_p, dtype=dt)
    inp[..., :cin] = torch.randn(B, H, W, cin, generator=g).to(dt)
    w = torch.randn(cout, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    film = torch.ones(B, 2, cout_p)
    film[:, 0, :cout] = 1 + 0.3 * torch.randn(B, cout, generator=g)
    film[:, 1] = 0
    film[:, 1, :cout] = 0.3 * torch.randn(B, cout, generator=g)
    zf0 = torch.zeros(B, H, W, cout_p)
    zf0[..., :cout] = torch.randn(B, H, W, cout, generator=g)
    acc = F.conv2d(inp.float().permute(0, 3, 1, 2)[:, :cin], w.to(dt).float(), padding=1).permute(0, 2, 3, 1)
    return inp, w, film, zf0, acc


CONV_CASES = [
    # cin, cout, shape (B,H,W), tune
    (16, 16, (1, 1, 128), dict(rows=1, acc_stages=1)),
    (16, 32, (1, 1, 1), {}),
    (32, 32, (1, 5, 130), dict(rows=1)),
    (64, 64, (1, 5, 130), dict(rows=2)),
    (48, 96, (2, 13, 150), {}),
    (96, 192, (1, 21, 300), {}),
    (54, 108, (1, 10, 70), {}),
    (96, 192, (2, 30, 260), dict(max_ctas=3)),
    (96, 192, (1, 9, 257), dict(kc=16, b_stages=2)),
    (96, 192, (2, 30, 260), dict(max_ctas=3, cluster=1)),
    (96, 192, (2, 30, 260), dict(cluster=4)),
    (48, 96, (2, 13, 150), dict(cluster=4, max_ctas=6)),
    (64, 64, (1, 3, 100), dict(cluster=4)),
    (96, 192, (1, 21, 300), dict(pair=1)),
    (96, 192, (2, 30, 260), dict(pair=1, max_ctas=4)),
    (64, 64, (1, 5, 130), dict(pair=1)),
    (64, 128, (1, 1, 100), dict(pair=1)),
    (48, 96, (2, 33, 300), dict(pair=1, max_ctas=4)),
    # filter bank resident in shared memory (the default when it fits) vs streamed per patch
    (48, 96, (2, 13, 150), dict(resident=1)),
    (48, 96, (2, 13, 150), dict(resident=2)),
    (48, 96, (2, 40, 300), dict(resident=1, max_ctas=3)),
    (64, 128, (1, 9, 257), dict(resident=1, max_ctas=2)),
    (64, 128, (1, 9, 257), dict(resident=2)),
    (96, 192, (2, 30, 260), dict(pair=1, resident=1, max_ctas=4)),
    (96, 192, (1, 21, 300), dict(pair=1, resident=2)),
    # filter rows fused along N (one UMMA per input row; the default where it applies) vs one UMMA per (row, tap)
    (48, 96, (2, 13, 150), dict(fuse=1)),
    (48, 96, (2, 13, 150), dict(fuse=2)),
    (48, 96, (2, 41, 300), dict(fuse=1, max_ctas=3)),
    (64, 128, (1, 9, 257), dict(fuse=1, max_ctas=2)),
    (32, 48, (1, 7, 130), dict(fuse=1, rows=4)),
    (32, 48, (2, 9, 100), dict(fuse=1, rows=2, max_ctas=2)),
    (16, 64, (1, 6, 64), dict(fuse=1)),
    # four epilogue warps (one per TMEM lane quarter) instead of the default eight
    (48, 96, (2, 13, 150), dict(epi_warps=4)),
    (96, 192, (1, 21, 300), dict(epi_warps=4, resident=2)),
    (64, 64, (1, 5, 130), dict(epi_warps=4, rows=1)),
]


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("halo_mode", [0, 1])
@pytest.mark.parametrize("cin,cout,shape,tune", CONV_CASES)
def test_conv1_film_silu(dev, cin, cout, shape, tune, halo_mode, dt):
    ops, native = _ops()
    if halo_mode == 1 and (tune.get("resident") == 1 or tune.get("fuse") == 1):
        pytest.skip("the resident filter bank is a shared-halo (halo_mode 0) configuration")
    inp, w, film, _, acc = _conv_operands(cin, cout, shape, 7, ops, dt)
    ref = F.silu(acc * film[:, 0][:, None, None, :cout] + film[:, 1][:, None, None, :cout])
    wp = ops.pack_conv_weight(w, dev, dtype=dt)
    got = ops.conv3x3(inp.to(dev), wp, 0, film.to(dev), use_tc=True, tune=native.tune(halo_mode=halo_mode, **tune))
    simt = ops.conv3x3(inp.to(dev), wp, 0, film.to(dev), use_tc=False)
    got, simt = got.cpu().float(), simt.cpu().float()
    # rounding of the stored 16-bit result + tanh.approx SiLU (abs err ~|x| * 2.5e-4) + accumulate order
    tol = (2 * _ulp(dt) + 5e-4) * max(1.0, ref.abs().max().item())
    assert (got[..., :cout] - ref).abs().max().item() <= tol
    assert (simt[..., :cout] - ref).abs().max().item() <= tol
    assert got[..., cout:].abs().max().item() == 0.0 if got.shape[-1] > cout else True
    nofilm = ops.conv3x3(inp.to(dev), wp, 0, None, use_tc=True, tune=native.tune(halo_mode=halo_mode, **tune)).cpu().float()
    assert (nofilm[..., :cout] - F.silu(acc)).abs().max().item() <= tol


@pytest.mark.parametrize("halo_mode", [0, 1])
@pytest.mark.parametrize("cin,cout,shape,tune", [
    (96, 48, (2, 13, 150), {}), (192, 96, (1, 21, 300), {}), (108, 54, (1, 10, 70), {}),
    (192, 96, (2, 30, 260), dict(max_ctas=3)), (32, 16, (1, 1, 5), {}), (192, 96, (1, 7, 129), dict(rows=1, acc_stages=1)),
    (192, 96, (2, 30, 260), dict(cluster=4)), (192, 96, (2, 30, 260), dict(cluster=1)), (96, 48, (1, 5, 700), dict(cluster=2, max_ctas=5)),
    (192, 96, (1, 21, 300), dict(pair=1)), (192, 96, (2, 30, 260), dict(pair=1, max_ctas=4)), (128, 64, (1, 3, 129), dict(pair=1)),
    (96, 48, (2, 13, 150), dict(resident=1)), (96, 48, (2, 40, 300), dict(resident=1, max_ctas=3)), (96, 48, (2, 13, 150), dict(resident=2)),
    (128, 64, (1, 9, 257), dict(resident=1, max_ctas=2)), (192, 96, (1, 21, 300), dict(resident=2)),
    (96, 48, (2, 13, 150), dict(fuse=1)), (96, 48, (2, 41, 300), dict(fuse=1, max_ctas=3)), (96, 48, (2, 13, 150), dict(fuse=2)),
    (96, 48, (1, 7, 129), dict(fuse=1, rows=4, epi_warps=4)), (64, 64, (1, 9, 257), dict(fuse=1, max_ctas=2)), (64, 32, (2, 9, 100), dict(fuse=1, rows=2)),
    (96, 48, (2, 13, 150), dict(epi_warps=4)), (192, 96, (1, 21, 300), dict(epi_warps=4)), (96, 48, (2, 40, 300), dict(epi_warps=4, rows=4, max_ctas=3)),
    (96, 48, (2, 40, 300), dict(rows=4, resident=2, max_ctas=3)), (96, 48, (1, 7, 129), dict(rows=1)),
])
@pytest.mark.parametrize("dt", DTYPES)
def test_conv2_residual(dev, cin, cout, shape, tune, halo_mode, dt):
    ops, native = _ops()
    if halo_mode == 1 and (tune.get("resident") == 1 or tune.get("fuse") == 1):
        pytest.skip("the resident filter bank is a shared-halo (halo_mode 0) configuration")
    inp, w, _, zf0, acc = _conv_operands(cin, cout, shape, 8, ops, dt)
    zref = zf0[..., :cout] + acc
    wp = ops.pack_conv_weight(w, dev, dtype=dt)
    for use_tc in (True, False):
        zf = zf0.to(dev).contiguous()
        zb = ops.conv3x3(inp.to(dev), wp, 1, None, zf, use_tc=use_tc, tune=native.tune(halo_mode=halo_mode, **tune))
        zf, zb = zf.cpu(), zb.cpu()
        assert (zf[..., :cout] - zref).abs().max().item() <= 1e-4     # fp32 residual stream: accumulate-order noise only
        assert torch.equal(zb, zf.to(dt))                             # shadow copy is exactly round16(zf)
        if zf.shape[-1] > cout:
            assert zf[..., cout:].abs().max().item() == 0.0


@pytest.mark.parametrize("use_tc", [True, False])
@pytest.mark.parametrize("r,tol", [(2, 1e-4), (3, 2e-4), (4, 1e-4)])
@pytest.mark.parametrize("cin,shape", [(48, (2, 7, 190)), (96, (1, 9, 129)), (54, (1, 1, 3))])
@pytest.mark.parametrize("dt", DTYPES)
def test_head_shuffle_skip_clamp(dev, r, tol, cin, shape, use_tc, dt):
    ops, native = _ops()
    g = torch.Generator().manual_seed(9 + r)
    B, H, W = shape
    cin_p = ops.padded_channels(cin)
    zb = torch.zeros(B, H, W, cin_p, dtype=dt)
    zb[..., :cin] = torch.randn(B, H, W, cin, generator=g).to(dt)
    w = torch.randn(3 * r * r, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    x = torch.rand(B, 3, H, W, generator=g)
    wp = ops.pack_conv_weight(w, dev, dtype=dt)
    u = F.pixel_shuffle(F.conv2d(zb.float().permute(0, 3, 1, 2)[:, :cin], w.to(dt).float(), padding=1), r)
    s = F.interpolate(x, scale_factor=r, mode="bicubic")
    # skip recomputed in the epilogue, clamped (upscale) and un-clamped (forward)
    got = ops.head_shuffle_add(zb.to(dev), wp, r, x=x.to(dev), skip_mode=2, clamp01=True, use_tc=use_tc).cpu()
    assert (got - (u + s).clamp(0, 1)).abs().max().item() <= tol
    got = ops.head_shuffle_add(zb.to(dev), wp, r, x=x.to(dev), skip_mode=2, clamp01=False, use_tc=use_tc).cpu()
    assert (got - (u + s)).abs().max().item() <= tol
    # skip read from a precomputed bicubic buffer
    y = ops.bicubic(x.to(dev), r)
    got = ops.head_shuffle_add(zb.to(dev), wp, r, x=None, y=y, skip_mode=1, clamp01=False, use_tc=use_tc).cpu()
    assert (got - (u + s)).abs().max().item() <= tol
    # pixel shuffle only
    got = ops.head_shuffle_add(zb.to(dev), wp, r, skip_mode=0, use_tc=use_tc).cpu()
    assert (got - u).abs().max().item() <= tol


@pytest.mark.parametrize("r,tol", [(2, 1e-4), (3, 2e-4), (4, 1e-4)])
@pytest.mark.parametrize("cin,shape", [(48, (2, 7, 190)), (96, (1, 9, 129)), (54, (1, 4, 131)), (48, (1, 13, 300))])
def test_head_with_stacked_taps(dev, r, tol, cin, shape):
    """The head with its vertical filter taps stacked along N (`VAR 2`, four-row patches; the default, forced here): one UMMA per input
    row and filter column feeds up to three output rows.  Heights that are not multiples of four exercise the re-zeroing
    of accumulator rows below the image; both skip forms, clamp, and the plain shuffle match the PyTorch reference."""
    ops, native = _ops()
    g = torch.Generator().manual_seed(19 + r)
    B, H, W = shape
    dt = torch.float16
    cin_p = ops.padded_channels(cin)
    zb = torch.zeros(B, H, W, cin_p, dtype=dt)
    zb[..., :cin] = torch.randn(B, H, W, cin, generator=g).to(dt)
    w = torch.randn(3 * r * r, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    x = torch.rand(B, 3, H, W, generator=g)
    wp = ops.pack_conv_weight(w, dev, dtype=dt)
    u = F.pixel_shuffle(F.conv2d(zb.float().permute(0, 3, 1, 2)[:, :cin], w.to(dt).float(), padding=1), r)
    s = F.interpolate(x, scale_factor=r, mode="bicubic")
    t = native.tune(fuse=1)
    for _ in range(2):   # (twice: the second launch finds the accumulators as the first one left them)
        got = ops.head_shuffle_add(zb.to(dev), wp, r, x=x.to(dev), skip_mode=2, clamp01=True, tune=t).cpu()
        assert (got - (u + s).clamp(0, 1)).abs().max().item() <= tol
    got = ops.head_shuffle_add(zb.to(dev), wp, r, skip_mode=0, tune=t).cpu()
    assert (got - u).abs().max().item() <= tol
    y = ops.bicubic(x.to(dev), r)
    got = ops.head_shuffle_add(zb.to(dev), wp, r, x=None, y=y, skip_mode=1, clamp01=False, tune=t).cpu()
    assert (got - (u + s)).abs().max().item() <= tol


def test_2x_pair_form_equals_row_form(dev):
    """The 2X head finishes two vertically adjacent LR rows per epilogue warp (pair form: four-row patches, eight epilogue
    warps) unless told to go row by row (tune dbg 128).  Every value is the same FMA chain in both, so they agree bit for
    bit, in every element type and layout pair, RGB and RGBA, with the skip recomputed: on a width that is not a multiple
    of 128 (clamped edge warps) and an odd height (a pair whose second row is below the image).  Eight epilogue warps are
    required (the launch fails rather than take four) and the head kernel's name shows its four-row patches, so the pair
    form is what ran."""
    from torch.profiler import ProfilerActivity, profile

    from tests.test_gpu_memory_contract import bits
    from tests.test_gpu_rgba_io import CL, _build, _cl, _is_cl, _rand4, _types

    m = _build("2x-fused-f16", dev)
    x, c = _rand4((2, 4, 9, 131), 31, dev)
    try:
        m.set_conv_tune(2, dev, epi_warps=8)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m.upscale(x, c)
            torch.cuda.synchronize()
        heads = {e.key for e in prof.key_averages() if "conv_tc_kernel<2," in e.key}
        assert heads and all(", 4, 2, 8>" in k for k in heads), heads   # <2, K, ROWS = 4, VAR 2, LAY 8 (RGBA)>
        for ch in (3, 4):
            for tag, xx, trunc in _types(x[:, :ch].contiguous()):
                m.u8_truncate = trunc
                for x_in in (xx, _cl(xx)):
                    for fmt in (torch.contiguous_format, CL):
                        m.set_conv_tune(2, dev, epi_warps=8)
                        pair = m.upscale(x_in, c, memory_format=fmt)
                        m.set_conv_tune(2, dev, epi_warps=8, dbg=128)
                        row = m.upscale(x_in, c, memory_format=fmt)
                        assert torch.equal(bits(pair), bits(row)), (ch, tag, _is_cl(x_in), fmt)
    finally:
        m.set_conv_tune(2, dev)
        m.u8_truncate = False

def test_shifted_umma_descriptor_probe(dev):
    """The hardware property the shared-halo conv relies on (DESIGN.md): a K-major swizzled A descriptor may
    start at ANY row of a TMA-written tile when base_offset stays 0."""
    ops, _ = _ops()
    for kc in (64, 32, 16):
        for shift in (0, 1, 2, 7, 130, 131, 132, 256):
            assert ops.probe_umma(kc, shift, 0) == 0.0


def test_conv1_and_head_read_the_first_channels_of_a_wider_tensor(dev):
    """in_pitch: a convolution whose input tensor is wider than its cin_p reads only the first cin_p channels."""
    ops, native = _ops()
    inp, w, film, _, acc = _conv_operands(48, 96, (2, 13, 150), 19, ops, torch.float16)
    junk = torch.randn(inp.shape).to(torch.float16)
    z16 = torch.cat([inp, junk], dim=-1).contiguous()
    wp = ops.pack_conv_weight(w, dev)
    for use_tc in (True, False):
        a = ops.conv3x3(inp.to(dev), wp, 0, film.to(dev), use_tc=use_tc).cpu()
        b = ops.conv3x3(z16.to(dev), wp, 0, film.to(dev), use_tc=use_tc).cpu()
        assert torch.equal(a, b)
    g = torch.Generator().manual_seed(20)
    wh = ops.pack_conv_weight(torch.randn(12, 48, 3, 3, generator=g) / 20, dev)
    x = torch.rand(2, 3, 13, 150, generator=g)
    ya = ops.head_shuffle_add(inp.to(dev), wh, 2, x=x.to(dev), skip_mode=2).cpu()
    yb = ops.head_shuffle_add(z16.to(dev), wh, 2, x=x.to(dev), skip_mode=2).cpu()
    assert torch.equal(ya, yb)
