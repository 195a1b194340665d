"""GPU: interleaved (channels-last) images in and out of the stem and head kernels (MZ_FLAG_X_NHWC / MZ_FLAG_Y_NHWC).

The property is exact: every call with an interleaved input and / or output equals the planar call on the same data, bit
for bit -- the stem stages the same values, the head's bicubic skip runs the same FMAs in the same order per colour, only
the addresses differ.  Shapes include ragged widths (W = 1, 3, 5, 131: the clamped neighbourhood branches), odd H, H = 1
and batches whose stem blocks cross image boundaries.
"""
import pytest
import torch

from tests.test_gpu_memory_contract import Guarded, _ctrl, _model, _no_nan, assert_guards, assert_unchanged, is_poison

gpu = pytest.mark.gpu
CL = torch.channels_last


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _cl(t):
    return t.contiguous(memory_format=CL)


def _is_cl(t):
    return t.permute(0, 2, 3, 1).is_contiguous() and not t.is_contiguous()


def _rand(shape, seed, dev):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(shape, generator=g)
    c = torch.rand(shape[0], 3, generator=g)
    return x.to(dev), c.to(dev)


# ---------------------------------------------------------------------------------------------------------------------
# 1. model level: every layout combination equals the planar call
# ---------------------------------------------------------------------------------------------------------------------
MODELS = {
    "2x-fused-f16": (lambda: _ctrl("MewZoom-2X-Ctrl", 2), "float16", {}),
    "2x-fused-bf16": (lambda: _ctrl("MewZoom-2X-Ctrl", 2), "bfloat16", {}),
    "2x-two-kernels": (lambda: _ctrl("MewZoom-2X-Ctrl", 2), "float16", dict(block=2)),
    "3x": (lambda: _ctrl("MewZoom-3X-Ctrl", 2), "float16", {}),
    "4x": (lambda: _ctrl("MewZoom-4X-Ctrl", 2), "float16", {}),
    "2x-c160-sliced": (lambda: dict(upscale_ratio=2, num_channels=160, hidden_ratio=2, num_encoder_layers=2,
                                    control_features=3), "float16", {}),
    "2x-simt": (lambda: _ctrl("MewZoom-2X-Ctrl", 1), "float16", "simt"),
}
SHAPES = [(2, 3, 7, 131), (3, 3, 5, 1), (2, 3, 1, 3), (1, 3, 9, 5)]


def _build(name, dev, seed=3):
    from ultrazoom_b200 import _native

    make_cfg, odt, how = MODELS[name]
    m = _model(make_cfg(), dev, seed=seed, operand_dtype=odt)
    if isinstance(how, dict) and how:
        m.set_conv_tune(0, dev, **how)
    if how == "simt":
        m._flags_extra = _native.FLAG_SIMT_CONV
    return m


@gpu
@pytest.mark.parametrize("name", list(MODELS))
def test_every_layout_equals_planar(dev, name):
    m = _build(name, dev)
    for shape in SHAPES:
        x, c = _rand(shape, sum(shape), dev)
        x8 = (x * 255).to(torch.uint8)
        cases = [("forward", m.forward, x, False), ("upscale", m.upscale, x, False), ("upscale u8", m.upscale, x8, False),
                 ("upscale u8 trunc", m.upscale, x8, True)]
        for what, fn, xx, trunc in cases:
            m.u8_truncate = trunc
            want = fn(xx, c)
            if xx.dtype != torch.uint8:
                _no_nan(what, want)
            for x_in in (xx, _cl(xx)):
                for fmt in (torch.contiguous_format, CL):
                    y = fn(x_in, c, memory_format=fmt)
                    tag = (name, shape, what, _is_cl(x_in), fmt)
                    assert y.dtype == want.dtype and y.shape == want.shape, tag
                    if fmt == CL:
                        assert y.permute(0, 2, 3, 1).is_contiguous(), tag
                    else:
                        assert y.is_contiguous(), tag          # (the default stays NCHW for a channels-last input)
                    assert torch.equal(y, want.contiguous(memory_format=fmt)), (tag, (y.float() - want.float()).abs().max())
        m.u8_truncate = False


# ---------------------------------------------------------------------------------------------------------------------
# 2. stem state
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "2x-c160-sliced"])
def test_stem_state_is_byte_identical(dev, name):
    """upscale_stage(..., 0, 0) runs the stem only: zf and the 16-bit shadow from an interleaved input are byte-identical
    to those from the planar one (fp32 and uint8 inputs; three images of 35 pixels, so stem blocks cross images)."""
    m = _build(name, dev)
    B, H, W = 3, 5, 7
    r = m.upscale_ratio
    x, c = _rand((B, 3, H, W), 11, dev)
    frame = torch.empty(B, 3, H * r, W * r, device=dev)
    for xx in (x, (x * 255).to(torch.uint8)):
        got = []
        for x_in in (xx, _cl(xx)):
            ws = m.stage_workspace(xx.shape, dev)
            ws.fill_(0xFF)
            m.upscale_stage(x_in, c, frame, (0, H, 0, W), (0, 0), 0, 0, ws)
            torch.cuda.synchronize()
            zf, z16 = m.stage_views(ws, xx.shape, 0)
            got.append((zf.view(torch.int32).clone(), z16.view(torch.int16).clone()))
        assert torch.equal(got[0][0], got[1][0]), (name, xx.dtype, "zf")
        assert torch.equal(got[0][1], got[1][1]), (name, xx.dtype, "16-bit shadow")


# ---------------------------------------------------------------------------------------------------------------------
# 3. prepared-launch cache
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "4x"])
def test_layouts_alternate_through_the_prepared_launch(dev, name):
    """One model, one shape, layouts alternating call after call: the head's prepared launch is replayed with each call's
    layouts, never with the previous call's."""
    m = _build(name, dev)
    x, c = _rand((2, 3, 11, 131), 12, dev)
    want = m.upscale(x, c)
    seq = [(x, torch.contiguous_format), (_cl(x), CL), (x, torch.contiguous_format), (_cl(x), CL),
           (_cl(x), torch.contiguous_format), (x, CL), (x, torch.contiguous_format), (x, CL), (_cl(x), CL)]
    for i, (x_in, fmt) in enumerate(seq):
        y = m.upscale(x_in, c, memory_format=fmt)
        assert torch.equal(y, want.contiguous(memory_format=fmt)), (name, i, _is_cl(x_in), fmt)


# ---------------------------------------------------------------------------------------------------------------------
# 4. host path and graphs
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("u8", [False, True])
def test_upscale_host_interleaved(dev, u8):
    m = _build("2x-fused-f16", dev)
    B, H, W = 3, 9, 131
    r = m.upscale_ratio
    x, c = _rand((B, 3, H, W), 13, dev)
    if u8:
        x = (x * 255).to(torch.uint8)
    want = m.upscale(x, c)
    xh = x.permute(0, 2, 3, 1).contiguous().cpu().pin_memory().permute(0, 3, 1, 2)   # pinned (B,H,W,3) frames
    ch = c.cpu()
    assert _is_cl(xh)
    y = m.upscale_host(xh, ch, memory_format=CL)                       # library-allocated channels-last output
    assert _is_cl(y) and torch.equal(y, want.cpu())
    y = m.upscale_host(xh, ch)                                          # default: NCHW
    assert y.is_contiguous() and torch.equal(y, want.cpu())
    for lane in (None, 0, 1):
        out = torch.full((B, H * r, W * r, 3), 7, dtype=want.dtype).pin_memory().permute(0, 3, 1, 2)
        got = m.upscale_host(xh, ch, out=out, lane=lane)                # a caller's out sets the layout
        if lane is not None:
            m.host_wait(lane)
        assert got is out and torch.equal(out, want.cpu()), lane
    planar_out = torch.empty(want.shape, dtype=want.dtype).pin_memory()
    m.upscale_host(xh, ch, out=planar_out, memory_format=CL)            # (out wins over memory_format)
    assert torch.equal(planar_out, want.cpu())


@gpu
def test_graph_interleaved(dev):
    m = _build("2x-fused-f16", dev)
    x, c = _rand((2, 3, 17, 131), 14, dev)
    x2, c2 = _rand((2, 3, 17, 131), 15, dev)
    want, want2 = m.upscale(x, c), m.upscale(x2, c2)
    g = m.capture(_cl(x), c, memory_format=CL)
    assert _is_cl(g.x) and _is_cl(g.y)
    assert torch.equal(g.replay(), want)
    assert torch.equal(g(_cl(x2), c2), want2)
    assert torch.equal(g(x, c), want)                                   # a planar x is copied into the interleaved buffer
    g2 = m.capture(_cl(x), c)                                           # interleaved in, default NCHW out
    assert g2.y.is_contiguous() and torch.equal(g2(x2, c2), want2)


# ---------------------------------------------------------------------------------------------------------------------
# 5. windows and tiles
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
def test_windows_assemble_an_interleaved_frame(dev, name):
    """upscale_into: four windows of the same tile written into a channels-last frame that is a view with a padded row
    pitch (and a padded image pitch) assemble the whole interleaved output; the padding is never written.  (The padding
    keeps the pointers and pitches aligned to the head's 16-byte stores.)"""
    m = _build(name, dev)
    r = m.upscale_ratio
    B, H, W = 2, 13, 131
    x, c = _rand((B, 3, H, W), 16, dev)
    for xx in (x, (x * 255).to(torch.uint8)):
        want = m.upscale(xx, c)
        fill = 77 if xx.dtype == torch.uint8 else -1.0
        bw = (W * r + 5 + 3) // 4 * 4                                  # row of bw pixels: 12 bw bytes, a multiple of 16
        buf = torch.full((B, H * r + 3, bw, 3), fill, dtype=want.dtype, device=dev)
        frame = buf[:, 1:1 + H * r, 4:4 + W * r, :].permute(0, 3, 1, 2)
        for x_in in (xx, _cl(xx)):
            buf.fill_(fill)
            for (y0, y1) in ((0, 6), (6, H)):
                for (x0, x1) in ((0, 64), (64, W)):
                    m.upscale_into(x_in, c, frame, (y0, y1, x0, x1), (y0 * r, x0 * r))
            assert torch.equal(frame, want), (name, xx.dtype, _is_cl(x_in))
            outside = torch.ones(buf.shape, dtype=torch.bool, device=dev)
            outside[:, 1:1 + H * r, 4:4 + W * r, :] = False
            assert bool((buf[outside] == fill).all()), (name, xx.dtype, "the padding was written")


@gpu
def test_tiles_into_interleaved_frame(dev):
    """run_tile_into (halo-padded tiles of a channels-last frame) and upscale_tiled_refresh on one GPU: the channels-last
    frame they assemble equals the un-tiled result bit for bit."""
    from ultrazoom_b200.sharding import close_refresh_state, halo_radius, plan_tiles, run_tile_into, upscale_tiled_refresh

    L = 4
    m = _model(_ctrl("MewZoom-2X-Ctrl", L), dev, seed=17)
    r = m.upscale_ratio
    x, c = _rand((1, 3, 50, 300), 18, dev)
    full = m.upscale(x, c)
    xc = _cl(x)
    frame = torch.full_like(full, -1.0, memory_format=CL)
    for t in plan_tiles(50, 300, 2, 2, halo_radius(L), align_w=128):
        run_tile_into(m, xc, c, t, r, frame)
    assert _is_cl(frame) and torch.equal(frame, full)
    frame.fill_(-1.0)
    state = upscale_tiled_refresh(m, xc, c, r, L, 2, 2, 2, frame, align_w=128)
    try:
        assert torch.equal(frame, full)
    finally:
        torch.cuda.synchronize()
        close_refresh_state(state)


# ---------------------------------------------------------------------------------------------------------------------
# 6. memory contract of the C ABI with interleaved images (guard bands, see test_gpu_memory_contract.py)
# ---------------------------------------------------------------------------------------------------------------------
def _call_args(m, dev, B, H, W):
    from ultrazoom_b200 import _native

    eng = m._engine(dev)
    stream = torch.cuda.current_stream(dev)
    ws = eng.workspace(B, H, W, stream)
    ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
    return _native, eng, ws_ptr, ws.numel() - (ws_ptr - ws.data_ptr()), stream.cuda_stream


@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x"])
@pytest.mark.parametrize("u8", [False, True])
def test_guarded_interleaved_calls(dev, name, u8):
    """mz_upscale with each NHWC flag combination and mz_upscale_window into an interleaved frame, on guarded buffers:
    guards unchanged, inputs byte-identical, no NaN left, every pixel outside the window untouched."""
    m = _build(name, dev)
    r = m.upscale_ratio
    B, H, W = 2, 9, 131
    x, c = _rand((B, 3, H, W), 19, dev)
    if u8:
        x = (x * 255).to(torch.uint8)
    want = m.upscale(x, c)
    dt = want.dtype
    N, eng, ws_ptr, ws_bytes, s = _call_args(m, dev, B, H, W)
    base = N.FLAG_CLAMP01 | (N.FLAG_IO_U8 if u8 else 0)
    gxp = Guarded((B, 3, H, W), x.dtype, dev, row=W, fill=x, src=True)
    gxn = Guarded((B, H, W, 3), x.dtype, dev, row=3 * W, fill=x.permute(0, 2, 3, 1), src=True)
    snaps = {id(g): g.snapshot() for g in (gxp, gxn)}
    for xn in (False, True):
        gx = gxn if xn else gxp
        for yn in (False, True):
            if not (xn or yn):
                continue
            shape = (B, H * r, W * r, 3) if yn else (B, 3, H * r, W * r)
            fills = (0x00, 0xFF) if u8 else (None,)
            for f in fills:
                gy = Guarded(shape, dt, dev, row=shape[2] * shape[3])
                if u8:
                    gy.view.fill_(f)
                else:
                    gy.poison()
                flags = base | (N.FLAG_X_NHWC if xn else 0) | (N.FLAG_Y_NHWC if yn else 0)
                N.check(eng.lib.mz_upscale(eng.handle, gx.ptr(), c.data_ptr(), B, gy.ptr(), B, H, W, ws_ptr, ws_bytes,
                                           flags, s))
                torch.cuda.synchronize()
                got = gy.view.permute(0, 3, 1, 2) if yn else gy.view
                assert torch.equal(got, want), (name, u8, xn, yn, f)
                if not u8:
                    _no_nan("y", gy.view)
                assert_guards(("y", gy))
                assert_unchanged(("x", gx, snaps[id(gx)]))
            # windowed into an interleaved frame larger than the window: LR window rows 2..7, columns 33..100
            wy0, wy1, wx0, wx1, fy, fx = 2, 7, 33, 100, 3, 4
            FH, FW = (wy1 - wy0) * r + 7, ((wx1 - wx0) * r + 11 + 3) // 4 * 4   # (16-byte aligned rows and origin)
            if yn:
                gf = Guarded((B, FH, FW, 3), dt, dev, row=3 * FW)
                dst, rp, ip = gf.ptr((fy * FW + fx) * 3), 3 * FW, 3 * FH * FW
            else:
                gf = Guarded((B, 3, FH, FW), dt, dev, row=FW)
                dst, rp, ip = gf.ptr(fy * FW + fx), FW, FH * FW
            if u8:
                gf.view.fill_(0xA5)
            else:
                gf.poison()
            N.check(eng.lib.mz_upscale_window(eng.handle, gx.ptr(), c.data_ptr(), B, dst, rp, ip, B, H, W, wy0, wy1, wx0,
                                              wx1, ws_ptr, ws_bytes, flags, s))
            torch.cuda.synchronize()
            fr = gf.view.permute(0, 3, 1, 2) if yn else gf.view
            hh, ww = (wy1 - wy0) * r, (wx1 - wx0) * r
            assert torch.equal(fr[:, :, fy:fy + hh, fx:fx + ww], want[:, :, wy0 * r:wy1 * r, wx0 * r:wx1 * r]), (name, xn, yn)
            outside = torch.ones(fr.shape, dtype=torch.bool, device=dev)
            outside[:, :, fy:fy + hh, fx:fx + ww] = False
            if u8:
                assert bool((fr[outside] == 0xA5).all()), (name, xn, yn, "window overwritten outside")
            else:
                assert is_poison(fr[outside]), (name, xn, yn, "window overwritten outside")
            assert_guards(("frame", gf))
            assert_unchanged(("x", gx, snaps[id(gx)]))


# ---------------------------------------------------------------------------------------------------------------------
# 7. errors
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_invalid_interleaved_calls(dev):
    m = _build("4x", dev)
    r = m.upscale_ratio
    B, H, W = 1, 8, 40
    x, c = _rand((B, 3, H, W), 20, dev)
    N, eng, ws_ptr, ws_bytes, s = _call_args(m, dev, B, H, W)
    y = torch.empty(B, 3, H * r, W * r, device=dev)
    for nf in (N.FLAG_X_NHWC, N.FLAG_Y_NHWC):                         # the skip-from-buffer bicubic is planar only
        rc = eng.lib.mz_upscale(eng.handle, x.data_ptr(), c.data_ptr(), B, y.data_ptr(), B, H, W, ws_ptr, ws_bytes,
                                N.FLAG_CLAMP01 | N.FLAG_SKIP_FROM_BUFFER | nf, s)
        assert rc == N.MZ_ERR_INVALID, nf
    f = torch.empty(B, H * r, W * r + 8, 3, device=dev)              # interleaved frame, float4 stores at r = 4
    flags = N.FLAG_CLAMP01 | N.FLAG_Y_NHWC
    rp, ip = 3 * (W * r + 8), 3 * (W * r + 8) * H * r

    def window(dst, row, img, x1=W):
        return eng.lib.mz_upscale_window(eng.handle, x.data_ptr(), c.data_ptr(), B, dst, row, img, B, H, W, 0, H, 0, x1,
                                         ws_ptr, ws_bytes, flags, s)

    def stage(dst, row, img):                                          # the same window, stored by a stage's head
        return eng.lib.mz_upscale_stage(eng.handle, x.data_ptr(), c.data_ptr(), B, dst, row, img, B, H, W, 0, H, 0, W,
                                        ws_ptr, ws_bytes, flags, s, 0, m.num_encoder_layers)

    assert window(f.data_ptr(), rp, ip) == N.MZ_OK
    for call in (window, stage):
        assert call(f.data_ptr() + 8, rp, ip) == N.MZ_ERR_INVALID      # 8 B: not 16-byte aligned
        assert call(f.data_ptr(), rp - 2, ip) == N.MZ_ERR_INVALID      # row pitch 8 B off alignment
        assert call(f.data_ptr(), rp, ip - 2) == N.MZ_ERR_INVALID      # image pitch 8 B off alignment
        assert call(f.data_ptr(), 3 * r * W - 4, ip) == N.MZ_ERR_INVALID  # row pitch smaller than the window's 3 r w
        assert call(f.data_ptr(), r * W, ip) == N.MZ_ERR_INVALID       # a planar row pitch is too small interleaved
    torch.cuda.synchronize()
    # Python: frames in neither layout
    bad = [torch.empty(B, 3, H * r, 2 * W * r, device=dev)[..., ::2],                    # stride(3) == 2
           torch.empty(B, 4, H * r, W * r, device=dev)[:, :3],                            # planes not evenly spaced
           torch.empty(B, H * r, W * r, 4, device=dev)[..., :3].permute(0, 3, 1, 2)]      # 4 channels per pixel
    for frame in bad:
        with pytest.raises(AssertionError):
            m.upscale_into(x, c, frame, (0, H, 0, W), (0, 0))
    ws = m.stage_workspace(x.shape, dev)
    with pytest.raises(AssertionError):
        m.upscale_stage(x, c, bad[0], (0, H, 0, W), (0, 0), 0, 2, ws)
    with pytest.raises(AssertionError):
        m.upscale(x, c, memory_format=torch.preserve_format)
    with pytest.raises(AssertionError):
        m.upscale_host(x.cpu(), c.cpu(), out=torch.empty(B, 3, H * r, 2 * W * r)[..., ::2])
