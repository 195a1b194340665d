"""GPU: 16-bit images in and out of the stem and head kernels (MZ_FLAG_IO_U16).

The property is exact: the stem reads x16 / 65535 as the IEEE quotient and so does the head's bicubic skip, so a 16-bit
call equals the fp32 call on ``x16.float() / 65535`` bit for bit before quantisation, and its output is that result
quantised once as the kernel does it: ``floor(fl32(65535 y + 0.5))`` (one fmaf, then truncation).  One input holds every
code 0..65535 exactly once per colour, so every code passes through both quotients.

torch's uint16 support is partial (no reductions; CUDA kernels beyond copies are not relied on): images are made on the
CPU, and results are compared as int16 bit patterns widened to int32.
"""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from tests.test_gpu_memory_contract import Guarded, _ctrl, _model, assert_guards, assert_unchanged
from tests.test_gpu_nhwc_io import MODELS, SHAPES, _build, _call_args

gpu = pytest.mark.gpu
CL, NCHW = torch.channels_last, torch.contiguous_format


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _codes(t):
    """uint16 -> int32 codes 0..65535 (any device, any strides)."""
    return t.view(torch.int16).to(torch.int32) & 0xFFFF


def _cl(t):
    """channels-last copy (through an int16 view for uint16)"""
    if t.dtype == torch.uint16:
        return t.view(torch.int16).contiguous(memory_format=CL).view(torch.uint16)
    return t.contiguous(memory_format=CL)


def _is_cl(t):
    return t.permute(0, 2, 3, 1).is_contiguous() and not t.is_contiguous()


def q16(y):
    """The head's quantisation of a [0, 1] fp32 result: 65535 y + 0.5 rounded once to fp32 (fmaf), then floored."""
    return torch.floor((y.double() * 65535.0 + 0.5).float()).to(torch.int32)


def _image(shape, seed, dev):
    """A random uint16 image, its value as fp32 (x16 / 65535, computed on the CPU) and a control vector."""
    g = torch.Generator().manual_seed(seed)
    x16 = torch.randint(0, 65536, shape, generator=g, dtype=torch.int32).to(torch.uint16)
    c = torch.rand(shape[0], 3, generator=g)
    return x16.to(dev), (x16.float() / 65535.0).to(dev), c.to(dev)


def _every_code(dev, seed=7):
    """(1, 3, 256, 256): each colour plane holds every code 0..65535 exactly once, in its own permuted order."""
    g = torch.Generator().manual_seed(seed)
    x16 = torch.stack([torch.randperm(65536, generator=g) for _ in range(3)]).view(1, 3, 256, 256).to(torch.uint16)
    c = torch.rand(1, 3, generator=g)
    return x16.to(dev), (x16.float() / 65535.0).to(dev), c.to(dev)


# ---------------------------------------------------------------------------------------------------------------------
# 0. CPU: the head's quotient (reciprocal multiply + one FMA correction, kernels.cuh lr_px) is exact for every code
# ---------------------------------------------------------------------------------------------------------------------
def _rn32(v: Fraction) -> float:
    """A positive rational rounded to the nearest float32, ties to even (normal range)."""
    e = v.numerator.bit_length() - v.denominator.bit_length()
    e += 1 if Fraction(2) ** (e + 1) <= v else (-1 if Fraction(2) ** e > v else 0)
    m = v / Fraction(2) ** (e - 23)
    n, rem = divmod(m.numerator, m.denominator)
    n += 1 if 2 * rem > m.denominator or (2 * rem == m.denominator and n % 2) else 0
    return float(n * Fraction(2) ** (e - 23))


def test_head_quotient_is_exact_for_every_code():
    """q = fl(x rcp), q' = fmaf(fmaf(-q, 65535, x), rcp, q) equals fl(x / 65535) for x = 0..65535.  The first fmaf is
    exact in float64 (Sterbenz: 65535 q is within a factor 2 of x), then rounded once to float32.  The second is
    evaluated in float64 and rounded to float32; that double rounding can only differ from fmaf's single rounding when
    the float64 value sits exactly on a float32 midpoint, and those codes are redone in exact rational arithmetic."""
    f32 = np.float32
    rcp = f32(1.0) / f32(65535.0)
    x = np.arange(65536, dtype=np.float32)
    q = x * rcp
    r = (np.float64(x) - np.float64(q) * 65535.0).astype(np.float32)
    d = np.float64(r) * np.float64(rcp) + np.float64(q)
    got = d.astype(np.float32)
    mid = d.astype(np.float32).astype(np.float64)
    ulp = np.spacing(got).astype(np.float64)
    on_mid = (np.abs(d - mid) * 2 == ulp) & (d != mid)
    for i in np.nonzero(on_mid)[0]:
        got[i] = _rn32(Fraction(float(r[i])) * Fraction(float(rcp)) + Fraction(float(q[i])))
    want = x / f32(65535.0)                                      # IEEE division, as the stem's __fdiv_rn
    assert np.array_equal(got, want), int(np.count_nonzero(got != want))
    assert np.count_nonzero(q != want) > 0                       # (the product alone is not exact: the test has teeth)


# ---------------------------------------------------------------------------------------------------------------------
# 1. bit-exact against the fp32 path, every model, every layout combination
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_u16_equals_quantised_fp32(dev, name):
    m = _build(name, dev)
    r = m.upscale_ratio
    inputs = [_image(shape, sum(shape) + 40, dev) for shape in SHAPES]
    inputs.append(_every_code(dev))
    for x16, xf, c in inputs:
        want = q16(m.upscale(xf, c))
        B, _, H, W = x16.shape
        for x_in in (x16, _cl(x16)):
            for fmt in (NCHW, CL):
                y = m.upscale(x_in, c, memory_format=fmt)
                tag = (name, tuple(x16.shape), _is_cl(x_in), fmt)
                assert y.dtype == torch.uint16 and tuple(y.shape) == (B, 3, H * r, W * r), tag
                assert _is_cl(y) if fmt == CL else y.is_contiguous(), tag
                d = (_codes(y) - want).abs()
                assert int(d.max()) == 0, (tag, int(d.max()), int((d != 0).sum()))


@gpu
def test_u16_layouts_alternate_through_the_prepared_launch(dev):
    """fp32, uint8 and uint16 calls in both layouts alternating on one model and shape: each call's head runs with its
    own element type and layouts, never those of the previous call."""
    m = _build("2x-fused-f16", dev)
    x16, xf, c = _image((2, 3, 11, 131), 41, dev)
    x8 = (xf * 255).to(torch.uint8)
    want16, wantf, want8 = q16(m.upscale(xf, c)), m.upscale(xf, c), m.upscale(x8, c)
    seq = [(x16, NCHW), (xf, NCHW), (_cl(x16), CL), (x8, CL), (x16, CL), (_cl(xf), NCHW), (_cl(x16), NCHW), (x8, NCHW)]
    for i, (x_in, fmt) in enumerate(seq):
        y = m.upscale(x_in, c, memory_format=fmt)
        if x_in.dtype == torch.uint16:
            assert torch.equal(_codes(y), want16), (i, fmt)
        else:
            assert torch.equal(y, wantf if x_in.dtype == torch.float32 else want8), (i, x_in.dtype, fmt)


# ---------------------------------------------------------------------------------------------------------------------
# 2. against the oracle, once per ratio
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["MewZoom-2X-Ctrl", "MewZoom-3X-Ctrl", "MewZoom-4X-Ctrl"])
def test_u16_against_the_oracle(dev, name):
    """Within the fp32 path's max-abs tolerance (tests/test_gpu_parity.py), in 16-bit steps, plus one for rounding."""
    from oracle import make_oracle
    from tests.test_gpu_parity import TOL, _model_from

    o = make_oracle(name, seed=4)
    m = _model_from(dict(upscale_ratio=o.upscale_ratio, num_channels=o.num_channels, hidden_ratio=o.hidden_ratio,
                         num_encoder_layers=o.num_encoder_layers, control_features=o.control_features),
                    o.state_dict(), dev)
    x16, _, c = _image((1, 3, 20, 70), 42, dev)
    xc = x16.cpu()
    with torch.inference_mode():
        ref = q16(o.upscale(xc.float() / 65535.0, c.cpu()))
    got = _codes(m.upscale(x16, c)).cpu()
    steps = math.ceil(TOL[name.replace("-Ctrl", "")][0] * 65535) + 1
    d = (got - ref).abs()
    assert int(d.max()) <= steps, (name, int(d.max()), steps)


# ---------------------------------------------------------------------------------------------------------------------
# 3. entry points: each equals upscale(x16) bit for bit
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_upscale_host_u16(dev):
    m = _build("2x-fused-f16", dev)
    B, H, W = 3, 9, 131
    r = m.upscale_ratio
    x16, _, c = _image((B, 3, H, W), 43, dev)
    want = _codes(m.upscale(x16, c)).cpu()
    xp = x16.cpu().pin_memory()
    xn = x16.cpu().permute(0, 2, 3, 1).contiguous().pin_memory().permute(0, 3, 1, 2)     # pinned (B,H,W,3) frames
    ch = c.cpu()
    for x_in in (xp, xn):
        y = m.upscale_host(x_in, ch)
        assert y.dtype == torch.uint16 and y.is_contiguous() and torch.equal(_codes(y), want)
        y = m.upscale_host(x_in, ch, memory_format=CL)
        assert _is_cl(y) and torch.equal(_codes(y), want)
        for lane in (None, 0, 1):
            for out in (torch.full((B, 3, H * r, W * r), 7, dtype=torch.uint16).pin_memory(),
                        torch.full((B, H * r, W * r, 3), 7, dtype=torch.uint16).pin_memory().permute(0, 3, 1, 2)):
                got = m.upscale_host(x_in, ch, out=out, lane=lane)       # a caller's out sets the layout
                if lane is not None:
                    m.host_wait(lane)
                assert got is out and torch.equal(_codes(out), want), (_is_cl(x_in), lane, _is_cl(out))


@gpu
def test_graph_u16(dev):
    m = _build("2x-fused-f16", dev)
    x16, _, c = _image((2, 3, 17, 131), 44, dev)
    x2, _, c2 = _image((2, 3, 17, 131), 45, dev)
    want, want2 = _codes(m.upscale(x16, c)), _codes(m.upscale(x2, c2))
    g = m.capture(x16, c)
    assert g.x.dtype == g.y.dtype == torch.uint16
    assert torch.equal(_codes(g.replay()), want)
    assert torch.equal(_codes(g(x2, c2)), want2)
    with pytest.raises(AssertionError):
        g(x2.view(torch.int16).to(torch.int32).float() / 65535.0, c2)   # captured for uint16: no other element type
    gi = m.capture(_cl(x16), c, memory_format=CL)
    assert _is_cl(gi.x) and _is_cl(gi.y) and torch.equal(_codes(gi.replay()), want)
    assert torch.equal(_codes(gi(_cl(x2), c2)), want2)


@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
def test_windows_assemble_u16_frames(dev, name):
    """upscale_into: four windows of a tile written into planar and interleaved uint16 frames that are views with padded
    row and image pitches assemble the whole output; the padding keeps its fill."""
    m = _build(name, dev)
    r = m.upscale_ratio
    B, H, W = 2, 13, 131
    x16, _, c = _image((B, 3, H, W), 46, dev)
    want = _codes(m.upscale(x16, c))
    fill = 0x1234
    bw = (W * r + 5 + 3) // 4 * 4                                      # rows of 8-byte multiples
    for nhwc in (False, True):
        if nhwc:
            buf = torch.full((B, H * r + 3, bw, 3), fill, dtype=torch.int16, device=dev)
            frame16 = buf[:, 1:1 + H * r, 4:4 + W * r, :].permute(0, 3, 1, 2)
        else:
            buf = torch.full((B, 3, H * r + 3, bw), fill, dtype=torch.int16, device=dev)
            frame16 = buf[:, :, 1:1 + H * r, 4:4 + W * r]
        frame = frame16.view(torch.uint16)
        for x_in in (x16, _cl(x16)):
            buf.fill_(fill)
            for (y0, y1) in ((0, 6), (6, H)):
                for (x0, x1) in ((0, 64), (64, W)):
                    m.upscale_into(x_in, c, frame, (y0, y1, x0, x1), (y0 * r, x0 * r))
            assert torch.equal(_codes(frame), want), (name, nhwc, _is_cl(x_in))
            inside = torch.zeros(buf.shape, dtype=torch.bool, device=dev)
            if nhwc:
                inside[:, 1:1 + H * r, 4:4 + W * r, :] = True
            else:
                inside[:, :, 1:1 + H * r, 4:4 + W * r] = True
            assert bool((buf[~inside] == fill).all()), (name, nhwc, "the padding was written")


@gpu
def test_tiles_into_u16_frame(dev):
    """run_tile_into and upscale_tiled_refresh (one process) assemble a uint16 frame equal to the un-tiled result."""
    from ultrazoom_b200.sharding import close_refresh_state, halo_radius, plan_tiles, run_tile_into, upscale_tiled_refresh

    L = 4
    m = _model(_ctrl("MewZoom-2X-Ctrl", L), dev, seed=17)
    r = m.upscale_ratio
    x16, _, c = _image((1, 3, 50, 300), 47, dev)
    want = _codes(m.upscale(x16, c))
    for x_in, fmt in ((x16, NCHW), (_cl(x16), CL)):
        frame = torch.full((1, 3, 50 * r, 300 * r), -1, dtype=torch.int16, device=dev).contiguous(memory_format=fmt)
        frame = frame.view(torch.uint16)
        for t in plan_tiles(50, 300, 2, 2, halo_radius(L), align_w=128):
            run_tile_into(m, x_in, c, t, r, frame)
        assert torch.equal(_codes(frame), want), fmt
        frame.view(torch.int16).fill_(-1)
        state = upscale_tiled_refresh(m, x_in, c, r, L, 2, 2, 2, frame, align_w=128)
        try:
            assert torch.equal(_codes(frame), want), fmt
        finally:
            torch.cuda.synchronize()
            close_refresh_state(state)


# ---------------------------------------------------------------------------------------------------------------------
# 4. guarded C ABI calls (guard bands, see test_gpu_memory_contract.py)
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
def test_guarded_u16_calls(dev, name):
    """mz_upscale in every layout and mz_upscale_window into a larger frame, on guarded uint16 buffers: each call made
    twice, the output prefilled with 0x0000 and then 0xFFFF (integer outputs have no NaN to find unwritten elements);
    both results equal the expected image, guards unchanged, inputs byte-identical, pixels outside the window kept."""
    m = _build(name, dev)
    r = m.upscale_ratio
    B, H, W = 2, 9, 131
    x16, _, c = _image((B, 3, H, W), 48, dev)
    want = _codes(m.upscale(x16, c))
    N, eng, ws_ptr, ws_bytes, s = _call_args(m, dev, B, H, W)
    base = N.FLAG_CLAMP01 | N.FLAG_IO_U16
    gxp = Guarded((B, 3, H, W), torch.uint16, dev, row=W, src=True)
    gxn = Guarded((B, H, W, 3), torch.uint16, dev, row=3 * W, src=True)
    gxp.view.view(torch.int16).copy_(x16.view(torch.int16))
    gxn.view.view(torch.int16).copy_(x16.view(torch.int16).permute(0, 2, 3, 1))
    snaps = {id(g): g.snapshot() for g in (gxp, gxn)}
    for xn in (False, True):
        gx = gxn if xn else gxp
        for yn in (False, True):
            flags = base | (N.FLAG_X_NHWC if xn else 0) | (N.FLAG_Y_NHWC if yn else 0)
            shape = (B, H * r, W * r, 3) if yn else (B, 3, H * r, W * r)
            for f in (0, -1):
                gy = Guarded(shape, torch.uint16, dev, row=shape[2] * shape[3])
                gy.view.view(torch.int16).fill_(f)
                N.check(eng.lib.mz_upscale(eng.handle, gx.ptr(), c.data_ptr(), B, gy.ptr(), B, H, W, ws_ptr, ws_bytes,
                                           flags, s))
                torch.cuda.synchronize()
                got = gy.view.permute(0, 3, 1, 2) if yn else gy.view
                assert torch.equal(_codes(got), want), (name, xn, yn, f)
                assert_guards(("y", gy))
                assert_unchanged(("x", gx, snaps[id(gx)]))
            # windowed into a frame larger than the window: LR window rows 2..7, columns 33..100
            wy0, wy1, wx0, wx1, fy, fx = 2, 7, 33, 100, 3, 4
            FH, FW = (wy1 - wy0) * r + 7, ((wx1 - wx0) * r + 11 + 3) // 4 * 4   # (8-byte aligned rows and origin)
            hh, ww = (wy1 - wy0) * r, (wx1 - wx0) * r
            for f in (0, -1):
                if yn:
                    gf = Guarded((B, FH, FW, 3), torch.uint16, dev, row=3 * FW)
                    dst, rp, ip = gf.ptr((fy * FW + fx) * 3), 3 * FW, 3 * FH * FW
                else:
                    gf = Guarded((B, 3, FH, FW), torch.uint16, dev, row=FW)
                    dst, rp, ip = gf.ptr(fy * FW + fx), FW, FH * FW
                gf.view.view(torch.int16).fill_(f)
                N.check(eng.lib.mz_upscale_window(eng.handle, gx.ptr(), c.data_ptr(), B, dst, rp, ip, B, H, W, wy0, wy1,
                                                  wx0, wx1, ws_ptr, ws_bytes, flags, s))
                torch.cuda.synchronize()
                fr = _codes(gf.view.permute(0, 3, 1, 2) if yn else gf.view)
                assert torch.equal(fr[:, :, fy:fy + hh, fx:fx + ww], want[:, :, wy0 * r:wy1 * r, wx0 * r:wx1 * r]), (
                    name, xn, yn, f)
                outside = torch.ones(fr.shape, dtype=torch.bool, device=dev)
                outside[:, :, fy:fy + hh, fx:fx + ww] = False
                assert bool((fr[outside] == (f & 0xFFFF)).all()), (name, xn, yn, f, "window overwritten outside")
                assert_guards(("frame", gf))
                assert_unchanged(("x", gx, snaps[id(gx)]))


# ---------------------------------------------------------------------------------------------------------------------
# 5. fp16 range guard
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_u16_fp16_range_guard(dev):
    """On a checkpoint whose hidden tensor overflows fp16 (built as tests/test_gpu_fp16_range.py builds it): a uint16
    upscale on a "float16" model returns and the next call raises, upscale_host raises itself; "auto" returns the bf16
    model's uint16 result bit for bit."""
    from oracle import make_oracle
    from tests.test_gpu_fp16_range import CFG, _m
    from tests.test_gpu_robustness import _scaled_block

    sd = _scaled_block(make_oracle(CFG, seed=5), 3.0e5)
    x16, _, c = _image((1, 3, 24, 136), 49, dev)
    raises = pytest.raises(RuntimeError, match="fp16 range")
    m = _m(sd, dev)
    m.upscale(x16, c)
    torch.cuda.synchronize()
    with raises:
        m.upscale(x16, c)
    assert m.saturated(reset=True)
    with raises:
        m.upscale_host(x16.cpu(), c.cpu())
    assert m.saturated(reset=True)
    mb = _m(sd, dev, "bfloat16")
    a = _m(sd, dev, "auto")
    assert torch.equal(_codes(a.upscale(x16, c)), _codes(mb.upscale(x16, c))) and a._auto_dtype == "bfloat16"
    a = _m(sd, dev, "auto")
    assert torch.equal(_codes(a.upscale_host(x16.cpu(), c.cpu())), _codes(mb.upscale_host(x16.cpu(), c.cpu())))
    assert a._auto_dtype == "bfloat16"


# ---------------------------------------------------------------------------------------------------------------------
# 6. errors, refused on the host before any launch
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_invalid_u16_calls(dev):
    m = _build("4x", dev)
    r = m.upscale_ratio
    B, H, W = 1, 8, 40
    x16, xf, c = _image((B, 3, H, W), 50, dev)
    N, eng, ws_ptr, ws_bytes, s = _call_args(m, dev, B, H, W)
    y = torch.full((B, 3, H * r, W * r), 0x2345, dtype=torch.int16, device=dev)
    U16 = N.FLAG_IO_U16
    xh, ch, yh = x16.cpu(), c.cpu(), torch.zeros(B, 3, H * r, W * r, dtype=torch.int16)
    for flags in (N.FLAG_CLAMP01 | U16 | N.FLAG_IO_U8, N.FLAG_CLAMP01 | U16 | N.FLAG_U8_TRUNC,
                  N.FLAG_CLAMP01 | U16 | N.FLAG_SKIP_FROM_BUFFER, U16):
        rc = eng.lib.mz_upscale(eng.handle, x16.data_ptr(), c.data_ptr(), B, y.data_ptr(), B, H, W, ws_ptr, ws_bytes,
                                flags, s)
        assert rc == N.MZ_ERR_INVALID, flags
        for lane in (None, 0):
            rc = (eng.lib.mz_upscale_host(eng.handle, xh.data_ptr(), ch.data_ptr(), B, yh.data_ptr(), B, H, W, flags)
                  if lane is None else
                  eng.lib.mz_upscale_host_async(eng.handle, lane, xh.data_ptr(), ch.data_ptr(), B, yh.data_ptr(), B, H, W,
                                                flags))
            assert rc == N.MZ_ERR_INVALID, (flags, lane)
    torch.cuda.synchronize()
    assert bool((y == 0x2345).all())                                   # nothing was launched
    # windows: 8-byte stores at r = 4 (4 pixels x 2 bytes), planar and interleaved
    for yn in (False, True):
        if yn:
            f = torch.empty(B, H * r, W * r + 8, 3, dtype=torch.int16, device=dev)
            rp, ip = 3 * (W * r + 8), 3 * (W * r + 8) * H * r
        else:
            f = torch.empty(B, 3, H * r, W * r + 8, dtype=torch.int16, device=dev)
            rp, ip = W * r + 8, (W * r + 8) * H * r
        flags = N.FLAG_CLAMP01 | U16 | (N.FLAG_Y_NHWC if yn else 0)

        def window(dst, row, img):
            return eng.lib.mz_upscale_window(eng.handle, x16.data_ptr(), c.data_ptr(), B, dst, row, img, B, H, W, 0, H, 0,
                                             W, ws_ptr, ws_bytes, flags, s)

        assert window(f.data_ptr(), rp, ip) == N.MZ_OK
        assert window(f.data_ptr() + 2, rp, ip) == N.MZ_ERR_INVALID   # 2 B: not 8-byte aligned
        assert window(f.data_ptr() + 4, rp, ip) == N.MZ_ERR_INVALID   # 4 B: not 8-byte aligned
        assert window(f.data_ptr(), rp + 2, ip) == N.MZ_ERR_INVALID   # row pitch 4 B off alignment
        assert window(f.data_ptr(), rp, ip + 1) == N.MZ_ERR_INVALID   # image pitch 2 B off alignment
    torch.cuda.synchronize()
    # Python
    with pytest.raises(AssertionError):
        m.forward(x16, c)
    with pytest.raises(AssertionError):
        m.upscale_host(x16.cpu(), c.cpu(), out=torch.empty(B, 3, H * r, W * r))                      # fp32 out
    with pytest.raises(AssertionError):
        m.upscale_host(x16.cpu(), c.cpu(), out=torch.empty(B, 3, H * r, W * r, dtype=torch.uint8))   # uint8 out
    with pytest.raises(AssertionError):
        m.upscale_host(xf.cpu(), c.cpu(), out=torch.empty(B, 3, H * r, W * r, dtype=torch.uint16))   # uint16 out, fp32 in
    with pytest.raises(AssertionError):
        m.upscale_into(x16, c, torch.empty(B, 3, H * r, W * r, device=dev), (0, H, 0, W), (0, 0))
    with pytest.raises(AssertionError):
        m.upscale_into(xf, c, torch.empty(B, 3, H * r, W * r, dtype=torch.uint16, device=dev), (0, H, 0, W), (0, 0))
