"""GPU: RGBA images in and out (MZ_FLAG_RGBA): colour through the network, a straight alpha resampled in the head.

The contract (include/mewzoom_b200.h, MZ_FLAG_RGBA):
  * colour: y[:, :3] equals the 3-channel call on x[:, :3] bit for bit, for every element type, layout and entry point --
    the stem never reads the alpha, the network is unchanged;
  * alpha: y[:, 3] = Q(clamp?(bicubic_r(x[:, 3]))), computed with a colour skip's FMAs in the same order, started from 0
    instead of from the accumulator -- so with all head weights zero an alpha equal to a colour plane gives a
    bit-identical channel (fp32 compared as values: 0 + (-0) is +0).
All comparisons are bit for bit unless stated.
"""
import pytest
import torch

from oracle.mewzoom_oracle import bicubic_upsample_ref
from tests.test_gpu_memory_contract import Guarded, _ctrl, _model, _no_nan, assert_guards, assert_unchanged, bits
from tests.test_gpu_nhwc_io import MODELS, SHAPES, _build

gpu = pytest.mark.gpu
CL = torch.channels_last
SHAPES4 = [(b, 4, h, w) for (b, _, h, w) in SHAPES]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _cl(t):
    return t.contiguous(memory_format=CL)


def _is_cl(t):
    return t.permute(0, 2, 3, 1).is_contiguous() and not t.is_contiguous()


def _rand4(shape, seed, dev):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(shape, generator=g)
    c = torch.rand(shape[0], 3, generator=g)
    return x.to(dev), c.to(dev)


def _types(x):
    """(tag, image, u8_truncate) for fp32, uint8, uint8 truncating and uint16 images holding the same values."""
    return [("f32", x, False), ("u8", (x * 255).round().to(torch.uint8), False),
            ("u8-trunc", (x * 255).round().to(torch.uint8), True), ("u16", (x * 65535).round().to(torch.uint16), False)]


def _zero_head(m):
    with torch.no_grad():
        m.head.conv.weight.zero_()
    m._invalidate_params()


# ---------------------------------------------------------------------------------------------------------------------
# 1. colour equals the RGB call, in every type and layout pair
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_colour_equals_rgb_call(dev, name):
    m = _build(name, dev)
    for shape in SHAPES4:
        x, c = _rand4(shape, sum(shape), dev)
        for tag, xx, trunc in _types(x):
            m.u8_truncate = trunc
            fns = [("upscale", m.upscale)] + ([("forward", m.forward)] if tag == "f32" else [])
            for what, fn in fns:
                want = fn(xx[:, :3].contiguous(), c)
                for x_in in (xx, _cl(xx)):
                    for fmt in (torch.contiguous_format, CL):
                        y = fn(x_in, c, memory_format=fmt)
                        key = (name, shape, tag, what, _is_cl(x_in), fmt)
                        assert y.shape == (shape[0], 4) + want.shape[2:] and y.dtype == want.dtype, key
                        assert y.is_contiguous(memory_format=fmt), key
                        assert torch.equal(y[:, :3], want), (key, (y[:, :3].float() - want.float()).abs().max())
                        if tag == "f32":
                            _no_nan(str(key), y)
        m.u8_truncate = False


# ---------------------------------------------------------------------------------------------------------------------
# 2. the alpha is the skip's resampling
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "2x-two-kernels", "3x", "4x", "2x-simt"])
def test_alpha_is_the_colour_skip(dev, name):
    """Head weights zero and x[:, 3] = x[:, 1]: the alpha channel equals the green channel (the skip alone) for every
    type and layout; with the real head weights the alpha does not change."""
    m = _build(name, dev)
    x, c = _rand4((2, 4, 9, 131), 21, dev)
    x[:, 3] = x[:, 1]
    real = {}
    for tag, xx, trunc in _types(x):
        m.u8_truncate = trunc
        for x_in in (xx, _cl(xx)):
            for fmt in (torch.contiguous_format, CL):
                for what in ("upscale", "forward") if tag == "f32" else ("upscale",):
                    real[(tag, _is_cl(x_in), fmt, what)] = getattr(m, what)(x_in, c, memory_format=fmt)[:, 3].clone()
    _zero_head(m)
    for tag, xx, trunc in _types(x):
        m.u8_truncate = trunc
        for x_in in (xx, _cl(xx)):
            for fmt in (torch.contiguous_format, CL):
                for what in ("upscale", "forward") if tag == "f32" else ("upscale",):
                    y = getattr(m, what)(x_in, c, memory_format=fmt)
                    key = (name, tag, _is_cl(x_in), fmt, what)
                    if tag == "f32":
                        assert bool((y[:, 3] == y[:, 1]).all()), key
                        assert torch.equal(y[:, 3].abs(), real[(tag, _is_cl(x_in), fmt, what)].abs()), key
                    else:
                        assert torch.equal(y[:, 3], y[:, 1]), key
                        assert torch.equal(y[:, 3], real[(tag, _is_cl(x_in), fmt, what)]), key
    m.u8_truncate = False


# ---------------------------------------------------------------------------------------------------------------------
# 3. the alpha against a float64 bicubic
# ---------------------------------------------------------------------------------------------------------------------
def _alpha_planes(H, W, dev):
    """Alpha planes (B=3, H, W) in [0, 1]: every 8-bit code, every 16-bit code (as code / 65535), hard 0/1 edges."""
    n = H * W
    a8 = (torch.arange(n) % 256).float().div(255).view(H, W)
    a16 = (torch.arange(n) % 65536).float().div(65535).view(H, W)
    edge = torch.zeros(H, W)
    edge[:, W // 3: 2 * W // 3] = 1.0
    edge[H // 2:, :] = 1.0 - edge[H // 2:, :]
    return torch.stack([a8, a16, edge]).to(dev)


@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
def test_alpha_against_float64(dev, name):
    m = _build(name, dev)
    r = m.upscale_ratio
    H, W = 128, 512                                          # 65536 pixels: every 16-bit code once
    x, c = _rand4((3, 4, H, W), 22, dev)
    x[:, 3] = _alpha_planes(H, W, dev)
    for tag, xx, trunc in _types(x):
        if tag == "u8-trunc":
            continue
        scale = {"f32": 1.0, "u8": 255.0, "u16": 65535.0}[tag]
        exact = xx[:, 3:].double() / scale                    # the values the kernel reads (x / 255, x / 65535)
        ref = bicubic_upsample_ref(exact, r)[:, 0].double()
        for fmt in (torch.contiguous_format, CL):
            y = m.upscale(_cl(xx) if fmt == CL else xx, c, memory_format=fmt)[:, 3]
            if tag == "f32":
                assert (y.double() - ref.clamp(0, 1)).abs().max().item() <= 1e-6, (name, fmt)
                yf = m.forward(xx, c, memory_format=fmt)[:, 3]
                # (unclamped, the hard edges' overshoot shows the fp32 phase weights: at r = 3 they are not dyadic and
                # the bound is the stand-alone bicubic kernel's, test_gpu_memory_contract.test_bicubic)
                assert (yf.double() - ref).abs().max().item() <= (1e-4 if r == 3 else 1e-6), (name, fmt, "forward")
                assert yf.min().item() < 0 and yf.max().item() > 1, "hard edges over- and undershoot"
                assert y.min().item() == 0 and y.max().item() == 1, "upscale clamps them"
            else:
                want = (ref.clamp(0, 1) * scale + 0.5).floor()
                assert (y.double() - want).abs().max().item() <= 1, (name, tag, fmt)


# ---------------------------------------------------------------------------------------------------------------------
# 4. the network never reads the alpha
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "2x-two-kernels", "3x", "4x", "2x-c160-sliced"])
def test_network_never_reads_alpha(dev, name):
    m = _build(name, dev)
    x, c = _rand4((2, 4, 11, 131), 23, dev)
    xp = x.clone()
    xp[:, 3] = float("nan")
    for fn in (m.upscale, m.forward):
        for x_in, xp_in in ((x, xp), (_cl(x), _cl(xp))):
            want = fn(x_in, c)[:, :3]
            got = fn(xp_in, c)
            assert torch.equal(got[:, :3], want), (name, fn.__name__, _is_cl(x_in))
            if fn == m.forward:                                        # (upscale's clamp maps NaN to 0)
                assert bool(torch.isnan(got[:, 3]).all()), "the alpha is its own resampling"


# ---------------------------------------------------------------------------------------------------------------------
# 5. prepared launches alternate between RGB and RGBA
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
def test_rgb_rgba_alternate(dev, name):
    m = _build(name, dev)
    x, c = _rand4((2, 4, 11, 131), 24, dev)
    x3 = x[:, :3].contiguous()
    w3, w4 = m.upscale(x3, c), m.upscale(x, c)
    w4cl = m.upscale(_cl(x), c, memory_format=CL)
    for i, (xi, fmt, want) in enumerate([(x3, None, w3), (x, None, w4), (x3, None, w3), (_cl(x), CL, w4cl), (x3, None, w3),
                                         (x, None, w4), (_cl(x3), CL, w3), (_cl(x), CL, w4cl)]):
        y = m.upscale(xi, c, memory_format=fmt or torch.contiguous_format)
        assert torch.equal(y, want.contiguous(memory_format=fmt or torch.contiguous_format)), (name, i)


# ---------------------------------------------------------------------------------------------------------------------
# 6. host path
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_upscale_host_rgba(dev):
    m = _build("2x-fused-f16", dev)
    B, H, W = 3, 9, 131
    r = m.upscale_ratio
    x, c = _rand4((B, 4, H, W), 25, dev)
    ch = c.cpu()
    m.upscale_host(x[:, :3].contiguous().cpu().pin_memory(), ch)      # an RGB call first: the lanes' buffers must grow
    for tag, xx, trunc in _types(x):
        m.u8_truncate = trunc
        want = m.upscale(xx, c).cpu()
        for nhwc in (False, True):
            xh = (xx.permute(0, 2, 3, 1).contiguous().cpu().pin_memory().permute(0, 3, 1, 2) if nhwc
                  else xx.cpu().pin_memory())
            y = m.upscale_host(xh, ch)
            assert y.shape == want.shape and torch.equal(y, want), (tag, nhwc)
            for lane in (None, 0, 1, 0):
                for ocl in (False, True):
                    out = (torch.full((B, H * r, W * r, 4), 7, dtype=want.dtype).pin_memory().permute(0, 3, 1, 2) if ocl
                           else torch.full(want.shape, 7, dtype=want.dtype).pin_memory())
                    got = m.upscale_host(xh, ch, out=out, lane=lane)
                    if lane is not None:
                        m.host_wait(lane)
                    assert got is out and torch.equal(out, want), (tag, nhwc, lane, ocl)
    m.u8_truncate = False


# ---------------------------------------------------------------------------------------------------------------------
# 7. graphs
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_graph_rgba(dev):
    m = _build("2x-fused-f16", dev)
    x, c = _rand4((2, 4, 17, 131), 26, dev)
    x2, c2 = _rand4((2, 4, 17, 131), 27, dev)
    for xx, xx2 in ((x, x2), ((x * 255).round().to(torch.uint8), (x2 * 255).round().to(torch.uint8))):
        want2 = m.upscale(xx2, c2)
        g = m.capture(xx, c)
        assert torch.equal(g(xx2, c2), want2)
        g2 = m.capture(_cl(xx), c, memory_format=CL)
        assert torch.equal(g2(_cl(xx2), c2), want2)
        with pytest.raises(AssertionError):                            # a 3-channel frame into a 4-channel graph
            g(xx2[:, :3].contiguous(), c2)
    gf = m.capture(x, c, clamp=False)
    assert torch.equal(gf(x2, c2), m.forward(x2, c2))


# ---------------------------------------------------------------------------------------------------------------------
# 8. windows and stages
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
def test_windows_assemble_an_rgba_frame(dev, name):
    m = _build(name, dev)
    r = m.upscale_ratio
    B, H, W = 2, 13, 131
    x, c = _rand4((B, 4, H, W), 28, dev)
    for tag, xx, trunc in _types(x):
        if tag == "u8-trunc":
            continue
        want = m.upscale(xx, c)
        fill = 77 if xx.dtype != torch.float32 else -1.0
        bw = (W * r + 5 + 3) // 4 * 4                                  # rows of bw pixels: 16-byte multiples
        for interleaved in (False, True):
            if interleaved:
                buf = torch.full((B, H * r + 3, bw, 4), fill, dtype=want.dtype, device=dev)
                frame = buf[:, 1:1 + H * r, 4:4 + W * r, :].permute(0, 3, 1, 2)
                inside = (slice(None), slice(1, 1 + H * r), slice(4, 4 + W * r), slice(None))
            else:
                buf = torch.full((B, 4, H * r + 3, bw), fill, dtype=want.dtype, device=dev)
                frame = buf[:, :, 1:1 + H * r, 4:4 + W * r]
                inside = (slice(None), slice(None), slice(1, 1 + H * r), slice(4, 4 + W * r))
            for x_in in (xx, _cl(xx)):
                buf.fill_(fill)
                for (y0, y1) in ((0, 6), (6, H)):
                    for (x0, x1) in ((0, 64), (64, W)):
                        m.upscale_into(x_in, c, frame, (y0, y1, x0, x1), (y0 * r, x0 * r))
                assert torch.equal(frame, want), (name, tag, interleaved, _is_cl(x_in))
                outside = torch.ones(buf.shape, dtype=torch.bool, device=dev)
                outside[inside] = False
                vals = buf.to(torch.int32) if buf.dtype == torch.uint16 else buf   # (few uint16 ops exist on CUDA)
                assert bool(((vals == fill) | ~outside).all()), (name, tag, interleaved, "the padding was written")


@gpu
def test_tiles_into_rgba_frame(dev):
    from ultrazoom_b200.sharding import close_refresh_state, halo_radius, plan_tiles, run_tile_into, upscale_tiled, \
        upscale_tiled_refresh

    L = 4
    m = _model(_ctrl("MewZoom-2X-Ctrl", L), dev, seed=17)
    r = m.upscale_ratio
    x, c = _rand4((1, 4, 50, 300), 29, dev)
    full = m.upscale(x, c)
    assert torch.equal(upscale_tiled(m.upscale, x, c, r, L, 2, 2), full)
    for xin, fmt in ((x, torch.contiguous_format), (_cl(x), CL)):
        frame = torch.full_like(full, -1.0, memory_format=fmt)
        for t in plan_tiles(50, 300, 2, 2, halo_radius(L), align_w=128):
            run_tile_into(m, xin, c, t, r, frame)
        assert torch.equal(frame, full), fmt
        frame.fill_(-1.0)
        state = upscale_tiled_refresh(m, xin, c, r, L, 2, 2, 2, frame, align_w=128)
        try:
            assert torch.equal(frame, full), fmt
        finally:
            torch.cuda.synchronize()
            close_refresh_state(state)


# ---------------------------------------------------------------------------------------------------------------------
# 9. memory contract
# ---------------------------------------------------------------------------------------------------------------------
def _call_args(m, dev, B, H, W):
    from ultrazoom_b200 import _native

    eng = m._engine(dev)
    stream = torch.cuda.current_stream(dev)
    ws = eng.workspace(B, H, W, stream)
    ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
    return _native, eng, ws, ws_ptr, ws.numel() - (ws_ptr - ws.data_ptr()), stream.cuda_stream


@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
def test_guarded_rgba_calls(dev, name):
    """mz_upscale in every type and layout pair and mz_upscale_window into a wider frame, on guarded buffers with a
    NaN-poisoned workspace: guards intact, inputs byte-identical, every element outside the window untouched."""
    m = _build(name, dev)
    r = m.upscale_ratio
    B, H, W = 2, 9, 131
    x, c = _rand4((B, 4, H, W), 30, dev)
    for tag, xx, trunc in _types(x):
        if tag == "u8-trunc":
            continue
        want = m.upscale(xx, c)
        dt = want.dtype
        N, eng, ws, ws_ptr, ws_bytes, s = _call_args(m, dev, B, H, W)
        base = N.FLAG_CLAMP01 | N.FLAG_RGBA | {"f32": 0, "u8": N.FLAG_IO_U8, "u16": N.FLAG_IO_U16}[tag]
        gxp = Guarded((B, 4, H, W), xx.dtype, dev, row=W, fill=xx, src=True)
        gxn = Guarded((B, H, W, 4), xx.dtype, dev, row=4 * W, fill=xx.permute(0, 2, 3, 1), src=True)
        snaps = {id(g): g.snapshot() for g in (gxp, gxn)}
        for xn in (False, True):
            gx = gxn if xn else gxp
            for yn in (False, True):
                flags = base | (N.FLAG_X_NHWC if xn else 0) | (N.FLAG_Y_NHWC if yn else 0)
                shape = (B, H * r, W * r, 4) if yn else (B, 4, H * r, W * r)
                gy = Guarded(shape, dt, dev, row=shape[2] * shape[3])
                gy.poison()
                with torch.inference_mode():                           # (the engine's workspace is an inference tensor)
                    ws.fill_(0xFF)
                N.check(eng.lib.mz_upscale(eng.handle, gx.ptr(), c.data_ptr(), B, gy.ptr(), B, H, W, ws_ptr, ws_bytes,
                                           flags, s))
                torch.cuda.synchronize()
                got = gy.view.permute(0, 3, 1, 2) if yn else gy.view
                assert torch.equal(got, want), (name, tag, xn, yn)
                assert_guards(("y", gy))
                assert_unchanged(("x", gx, snaps[id(gx)]))
                # windowed into a frame larger than the window: LR rows 2..7, columns 33..100
                wy0, wy1, wx0, wx1, fy, fx = 2, 7, 33, 100, 3, 4
                FH, FW = (wy1 - wy0) * r + 7, ((wx1 - wx0) * r + 11 + 3) // 4 * 4
                if yn:
                    gf = Guarded((B, FH, FW, 4), dt, dev, row=4 * FW)
                    dst, rp, ip = gf.ptr((fy * FW + fx) * 4), 4 * FW, 4 * FH * FW
                else:
                    gf = Guarded((B, 4, FH, FW), dt, dev, row=FW)
                    dst, rp, ip = gf.ptr(fy * FW + fx), FW, FH * FW
                gf.poison()
                N.check(eng.lib.mz_upscale_window(eng.handle, gx.ptr(), c.data_ptr(), B, dst, rp, ip, B, H, W, wy0, wy1,
                                                  wx0, wx1, ws_ptr, ws_bytes, flags, s))
                torch.cuda.synchronize()
                fr = gf.view.permute(0, 3, 1, 2) if yn else gf.view
                hh, ww = (wy1 - wy0) * r, (wx1 - wx0) * r
                assert torch.equal(fr[:, :, fy:fy + hh, fx:fx + ww], want[:, :, wy0 * r:wy1 * r, wx0 * r:wx1 * r]), \
                    (name, tag, xn, yn)
                outside = torch.ones(fr.shape, dtype=torch.bool, device=dev)
                outside[:, :, fy:fy + hh, fx:fx + ww] = False
                poison = (fr == 255) if dt == torch.uint8 else (bits(fr) == -1)
                assert bool((poison | ~outside).all()), (name, tag, xn, yn, "window overwritten outside")
                assert_guards(("frame", gf))
                assert_unchanged(("x", gx, snaps[id(gx)]))


# ---------------------------------------------------------------------------------------------------------------------
# 10. the SIMT twin
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("ratio", [2, 3, 4])
def test_simt_twin_rgba(dev, ratio):
    from ultrazoom_b200 import _native

    m = _model(_ctrl({2: "MewZoom-2X-Ctrl", 3: "MewZoom-3X-Ctrl", 4: "MewZoom-4X-Ctrl"}[ratio], 1), dev, seed=31)
    x, c = _rand4((2, 4, 7, 70), 32, dev)
    for tag, xx, trunc in _types(x):
        m.u8_truncate = trunc
        for x_in in (xx, _cl(xx)):
            for fmt in (torch.contiguous_format, CL):
                m._flags_extra = 0
                tc = m.upscale(x_in, c, memory_format=fmt)
                m._flags_extra = _native.FLAG_SIMT_CONV
                simt = m.upscale(x_in, c, memory_format=fmt)
                simt3 = m.upscale(x_in[:, :3].contiguous(), c)
                m._flags_extra = 0
                key = (ratio, tag, _is_cl(x_in), fmt)
                assert torch.equal(simt[:, :3], simt3), key
                assert torch.equal(simt[:, 3], tc[:, 3]), key
    m.u8_truncate = False


# ---------------------------------------------------------------------------------------------------------------------
# 11. refusals
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_invalid_rgba_calls(dev):
    from ultrazoom_b200 import Yuv420

    m = _build("4x", dev)
    r = m.upscale_ratio
    B, H, W = 1, 8, 40
    x, c = _rand4((B, 4, H, W), 33, dev)
    N, eng, ws, ws_ptr, ws_bytes, s = _call_args(m, dev, B, H, W)
    y = torch.full((B, 4, H * r, W * r), -1.0, device=dev)
    y8 = torch.full((B, 4, H * r, W * r), 7, dtype=torch.uint8, device=dev)
    x8 = (x * 255).to(torch.uint8)
    for xp, yp, flags in ((x8, y8, N.FLAG_RGBA | N.FLAG_CLAMP01 | N.FLAG_IO_U8 | N.FLAG_YUV420),
                          (x, y, N.FLAG_RGBA | N.FLAG_CLAMP01 | N.FLAG_SKIP_FROM_BUFFER)):
        rc = eng.lib.mz_upscale(eng.handle, xp.data_ptr(), c.data_ptr(), B, yp.data_ptr(), B, H, W, ws_ptr, ws_bytes, flags, s)
        assert rc == N.MZ_ERR_INVALID, flags
        rc = eng.lib.mz_upscale_host(eng.handle, xp.cpu().data_ptr(), c.cpu().data_ptr(), B, yp.cpu().data_ptr(), B, H, W,
                                     flags)
        assert rc == N.MZ_ERR_INVALID, flags
    torch.cuda.synchronize()
    assert bool((y == -1.0).all()) and bool((y8 == 7).all()), "a refused call wrote its output"
    with pytest.raises(AssertionError):                                # 5 channels
        m.upscale(torch.rand(B, 5, H, W, device=dev), c)
    with pytest.raises(AssertionError):                                # RGBA with 4:2:0 frames
        m.upscale(x8, c, yuv=Yuv420())
    # a frame / out whose channel count differs from x
    for xx, frame in ((x, torch.full((B, 3, H * r, W * r), -1.0, device=dev)),
                      (x[:, :3].contiguous(), torch.full((B, 4, H * r, W * r), -1.0, device=dev))):
        with pytest.raises(AssertionError):
            m.upscale_into(xx, c, frame, (0, H, 0, W), (0, 0))
        with pytest.raises(AssertionError):
            m.upscale_stage(xx, c, frame, (0, H, 0, W), (0, 0), 0, 2, m.stage_workspace(xx.shape, dev))
        with pytest.raises(AssertionError):
            m.upscale_host(xx.cpu(), c.cpu(), out=torch.empty(frame.shape))
        assert bool((frame == -1.0).all())
    # misaligned interleaved RGBA windows: fp32 rows of 4r values leave in 16-byte stores
    f = torch.full((B, H * r, W * r + 8, 4), -1.0, device=dev)
    flags = N.FLAG_CLAMP01 | N.FLAG_RGBA | N.FLAG_Y_NHWC
    rp, ip = 4 * (W * r + 8), 4 * (W * r + 8) * H * r

    def window(dst, row, img):
        return eng.lib.mz_upscale_window(eng.handle, x.data_ptr(), c.data_ptr(), B, dst, row, img, B, H, W, 0, H, 0, W,
                                         ws_ptr, ws_bytes, flags, s)

    def stage(dst, row, img):                                          # the same window, stored by a stage's head
        return eng.lib.mz_upscale_stage(eng.handle, x.data_ptr(), c.data_ptr(), B, dst, row, img, B, H, W, 0, H, 0, W,
                                        ws_ptr, ws_bytes, flags, s, 0, m.num_encoder_layers)

    for call in (window, stage):
        assert call(f.data_ptr() + 8, rp, ip) == N.MZ_ERR_INVALID       # 8 B: not 16-byte aligned
        assert call(f.data_ptr(), rp - 2, ip) == N.MZ_ERR_INVALID       # row pitch 8 B off
        assert call(f.data_ptr(), rp, ip - 2) == N.MZ_ERR_INVALID       # image pitch 8 B off
        assert call(f.data_ptr(), 3 * r * W, ip) == N.MZ_ERR_INVALID    # an RGB row pitch is too small for RGBA
    torch.cuda.synchronize()
    assert bool((f == -1.0).all()), "a refused window wrote its frame"
    assert window(f.data_ptr(), rp, ip) == N.MZ_OK
    torch.cuda.synchronize()
    assert torch.equal(f[:, :, :W * r].permute(0, 3, 1, 2), m.upscale(x, c))


# ---------------------------------------------------------------------------------------------------------------------
# 12. against the reference (oracle/rgba.py) on a committed checkpoint
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_rgba_against_reference(dev):
    """upscale / forward of an RGBA image against oracle.rgba.upscale_rgba_ref on the ctrl_2x_c48_l2 fixture: the colour
    within the fp32 oracle bound smoke() uses, the alpha (the skip alone, no 16-bit rounding) within 1e-6."""
    from oracle.rgba import upscale_rgba_ref
    from tests.helpers import load_case, oracle_from_case
    from ultrazoom_b200 import MewZoom

    cfg, sd, x, c, _ = load_case("ctrl_2x_c48_l2")
    ref_model = oracle_from_case(cfg, sd)
    m = MewZoom(**cfg)
    m.load_state_dict(sd)
    m = m.to(dev).eval()
    B, _, H, W = x.shape
    a = torch.zeros(B, 1, H, W)
    a[..., W // 3: 2 * W // 3] = 1.0
    x4 = torch.cat([x, a], dim=1)
    for clamp in (True, False):
        want = upscale_rgba_ref(ref_model, x4, c, clamp=clamp)
        for x_in, fmt in ((x4, torch.contiguous_format), (_cl(x4), CL)):
            fn = m.upscale if clamp else m.forward
            y = fn(x_in.to(dev), c.to(dev), memory_format=fmt).cpu()
            assert (y[:, :3] - want[:, :3]).abs().max().item() <= 2e-2, (clamp, fmt)
            assert (y[:, 3] - want[:, 3]).abs().max().item() <= 1e-6, (clamp, fmt)

