"""GPU: 4:2:0 video frames (NV12, P010) in and out of ``upscale`` (MZ_FLAG_YUV420).

The conversion kernels are held to the float64 reference (oracle/yuv420.py) within one code.  The whole call is defined as
decode -> the 16-bit planar upscale -> encode, so it must equal that composition of the public pieces bit for bit, on every
entry point (device, host lanes, graphs).  The new kernels touch only the elements they own (guard bands as in
test_gpu_memory_contract.py), and every invalid combination is refused.

torch's uint16 support is partial: frames are made with numpy and compared on the CPU."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import yuv420 as ref
from tests.test_gpu_memory_contract import Guarded, _ctrl, _model, assert_guards, assert_unchanged
from tests.test_gpu_nhwc_io import _build

gpu = pytest.mark.gpu
MATRICES = ("bt709", "bt601", "bt2020")
# (B, H, W): W not a multiple of 8 or 16, H = 2, a single quad, a frame wider than one 128-quad block row
SHAPES = [(2, 6, 20), (3, 2, 6), (1, 2, 2), (2, 4, 522), (1, 10, 34)]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _np(t):
    t = t.detach().cpu()
    return t.view(torch.int16).numpy().view(np.uint16) if t.dtype == torch.uint16 else t.numpy()


def _t(a, dev=None):
    a = np.ascontiguousarray(a)
    t = torch.from_numpy(a.view(np.int16)).view(torch.uint16) if a.dtype == np.uint16 else torch.from_numpy(a)
    return t.to(dev) if dev is not None else t


def _frames(B, H, W, dtype, seed, low_bits=False):
    """Random NV12 / P010 frames (codes over the whole range; P010 low bits zero unless ``low_bits``)."""
    rng = np.random.default_rng(seed)
    mx = 255 if dtype == np.uint8 else 1023
    f = ref.join_frames(rng.integers(0, mx + 1, (B, H, W)), rng.integers(0, mx + 1, (B, H // 2, W // 2)),
                        rng.integers(0, mx + 1, (B, H // 2, W // 2)), dtype)
    if low_bits:
        f = f | rng.integers(0, 64, f.shape).astype(np.uint16)
    return f


def _rgb16(B, H, W, seed):
    return np.random.default_rng(seed).integers(0, 65536, (B, 3, H, W)).astype(np.uint16)


def _yuv(matrix, full):
    from ultrazoom_b200 import Yuv420

    return Yuv420(matrix, full)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the conversion kernels against the float64 reference
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16], ids=["nv12", "p010"])
@pytest.mark.parametrize("matrix", MATRICES)
@pytest.mark.parametrize("full", [False, True], ids=["limited", "full"])
def test_kernels_against_reference(dev, dtype, matrix, full):
    from ultrazoom_b200 import ops

    f = _yuv(matrix, full)
    for i, (B, H, W) in enumerate(SHAPES):
        x = _frames(B, H, W, dtype, seed=10 + i)
        got = _np(ops.yuv420_to_rgb16(_t(x, dev), f)).astype(np.int64)
        want = ref.decode(x, matrix, full).astype(np.int64)
        assert got.shape == (B, 3, H, W)
        assert np.abs(got - want).max() <= 1, ((B, H, W), int(np.abs(got - want).max()))
        rgb = _rgb16(B, H, W, seed=20 + i)
        got = _np(ops.rgb16_to_yuv420(_t(rgb, dev), torch.uint8 if dtype == np.uint8 else torch.uint16, f))
        want = ref.encode(rgb, dtype, matrix, full)
        assert got.shape == (B, 3 * H // 2, W) and got.dtype == dtype
        d = np.abs(np.concatenate([c.ravel() for c in ref.split_frames(got)]) -
                   np.concatenate([c.ravel() for c in ref.split_frames(want)]))
        assert d.max() <= 1, ((B, H, W), int(d.max()))
        if dtype == np.uint16:
            assert not (got & 63).any(), "P010 output must have its low 6 bits zero"


@gpu
def test_p010_low_bits_are_ignored(dev):
    from ultrazoom_b200 import ops

    for B, H, W in SHAPES:
        noisy = _frames(B, H, W, np.uint16, seed=B + H + W, low_bits=True)
        clean = noisy & np.uint16(0xFFC0)
        assert (noisy != clean).any()
        assert np.array_equal(_np(ops.yuv420_to_rgb16(_t(noisy, dev))), _np(ops.yuv420_to_rgb16(_t(clean, dev))))


# ---------------------------------------------------------------------------------------------------------------------
# 2. upscale(yuv=) is exactly decode -> 16-bit upscale -> encode
# ---------------------------------------------------------------------------------------------------------------------
MODELS = ["2x-fused-f16", "2x-two-kernels", "3x", "4x", "2x-no-control"]


def _model_for(name, dev):
    if name == "2x-no-control":
        cfg = _ctrl("MewZoom-2X", 2)
        return _model(cfg, dev, seed=5), None
    return _build(name, dev), torch.rand(2, 3, generator=torch.Generator().manual_seed(1)).to(dev)


def _composed(m, x, c, f):
    from ultrazoom_b200 import ops

    return ops.rgb16_to_yuv420(m.upscale(ops.yuv420_to_rgb16(x, f), c), x.dtype, f)


@gpu
@pytest.mark.parametrize("name", MODELS)
def test_upscale_equals_the_composition(dev, name):
    m, c = _model_for(name, dev)
    r = m.upscale_ratio
    assert m.control_features == (0 if c is None else 3)
    cases = [(np.uint8, "bt709", False), (np.uint16, "bt2020", True), (np.uint8, "bt601", True), (np.uint16, "bt709", False)]
    for k, (dtype, matrix, full) in enumerate(cases):
        f = _yuv(matrix, full)
        for B, H, W in ((2, 10, 22), (1, 2, 2), (2, 4, 270)):
            x = _t(_frames(B, H, W, dtype, seed=k + W), dev)
            cc = None if c is None else c[:B]
            y = m.upscale(x, cc, yuv=f)
            assert y.dtype == x.dtype and tuple(y.shape) == (B, 3 * H * r // 2, W * r)
            assert np.array_equal(_np(y), _np(_composed(m, x, cc, f))), (name, dtype, matrix, full, (B, H, W))


@gpu
def test_host_lanes_and_graphs_equal_the_device_call(dev):
    m, c = _model_for("2x-fused-f16", dev)
    for dtype, f in ((np.uint8, _yuv("bt709", False)), (np.uint16, _yuv("bt2020", True))):
        B, H, W = 2, 12, 40
        x = _t(_frames(B, H, W, dtype, seed=3), dev)
        want = _np(m.upscale(x, c, yuv=f))
        xh, ch = x.cpu().pin_memory(), c.cpu()
        assert np.array_equal(_np(m.upscale_host(xh, ch, yuv=f)), want)
        outs = []
        for lane in (0, 1):
            out = torch.empty((B, 3 * H, 2 * W), dtype=x.dtype).pin_memory()
            outs.append(m.upscale_host(xh, ch, out=out, lane=lane, yuv=f))
        m.host_wait()
        for o in outs:
            assert np.array_equal(_np(o), want)
        g = m.capture(x, c, yuv=f)
        x2 = _t(_frames(B, H, W, dtype, seed=4), dev)
        want2 = _np(m.upscale(x2, c, yuv=f))
        assert np.array_equal(_np(g(x2, c)), want2)
        assert np.array_equal(_np(g(x, c)), want)
        m.upscale(x2, c, yuv=f)                                    # (an ordinary call in between leaves the graph's buffers)
        assert np.array_equal(_np(g.replay()), want)


@gpu
def test_auto_operands_follow_the_sixteen_bit_call(dev):
    """operand_dtype="auto" on an in-range checkpoint runs fp16 and gives the fp16 model's frames."""
    from ultrazoom_b200 import MewZoom

    m, c = _model_for("2x-fused-f16", dev)
    a = MewZoom(**_ctrl("MewZoom-2X-Ctrl", 2), operand_dtype="auto").to(dev).eval()
    a.load_state_dict(m.state_dict())
    x = _t(_frames(2, 8, 30, np.uint8, seed=6), dev)
    f = _yuv("bt709", False)
    assert np.array_equal(_np(a.upscale(x, c, yuv=f)), _np(m.upscale(x, c, yuv=f)))
    assert a._auto_dtype == "float16"


# ---------------------------------------------------------------------------------------------------------------------
# 3. memory contract
# ---------------------------------------------------------------------------------------------------------------------
def _refill_outside(g: Guarded, value: int):
    g.raw[:g.start].fill_(value)
    g.raw[g.end:].fill_(value)


@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16], ids=["nv12", "p010"])
def test_kernels_touch_only_their_own_elements(dev, dtype):
    from ultrazoom_b200 import _native

    lib = _native.load()
    tdt = torch.uint8 if dtype == np.uint8 else torch.uint16
    f = _yuv("bt601", False)
    flags = f.flags(tdt)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for B, H, W in SHAPES:
        x = _t(_frames(B, H, W, dtype, seed=W), dev)
        gx = Guarded(x.shape, tdt, dev, row=W, fill=x, src=True)
        gy = Guarded((B, 3, H, W), torch.uint16, dev, row=W)
        snap = gx.snapshot()
        _native.check(lib.mz_yuv420_to_rgb16(gx.ptr(), gy.ptr(), B, H, W, flags, stream))
        torch.cuda.synchronize(dev)
        assert_guards(("rgb16", gy))
        assert_unchanged(("yuv", gx, snap))
        rgb = gy.view.clone()
        _refill_outside(gx, 0x3C)
        gy.raw[gy.start:gy.end].fill_(0x77)
        _native.check(lib.mz_yuv420_to_rgb16(gx.ptr(), gy.ptr(), B, H, W, flags, stream))
        assert np.array_equal(_np(gy.view), _np(rgb)), "decode read outside its frame"

        gr = Guarded((B, 3, H, W), torch.uint16, dev, row=W, fill=rgb, src=True)
        go = Guarded(x.shape, tdt, dev, row=W)
        snap = gr.snapshot()
        _native.check(lib.mz_rgb16_to_yuv420(gr.ptr(), go.ptr(), B, H, W, flags, stream))
        torch.cuda.synchronize(dev)
        assert_guards(("yuv out", go))
        assert_unchanged(("rgb16 in", gr, snap))
        out = go.view.clone()
        _refill_outside(gr, 0x3C)
        go.raw[go.start:go.end].fill_(0x77)
        _native.check(lib.mz_rgb16_to_yuv420(gr.ptr(), go.ptr(), B, H, W, flags, stream))
        assert np.array_equal(_np(go.view), _np(out)), "encode read outside its image"


@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x"])
def test_guarded_upscale_call(dev, name):
    """mz_upscale with 4:2:0 frames on guarded buffers and a workspace filled with 0xFF: guards intact, input unchanged,
    the result the same as the ordinary call's and independent of the bytes around the input."""
    from ultrazoom_b200 import _native

    m, c = _model_for(name, dev)
    r = m.upscale_ratio
    B, H, W = 2, 8, 134
    for dtype, f in ((np.uint8, _yuv("bt709", False)), (np.uint16, _yuv("bt2020", False))):
        x = _t(_frames(B, H, W, dtype, seed=9), dev)
        want = _np(m.upscale(x, c, yuv=f))
        eng = m._engine(dev)
        stream = torch.cuda.current_stream(dev)
        flags = _native.FLAG_CLAMP01 | f.flags(x.dtype)
        ws = eng.workspace(B, H, W, stream, flags)
        ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
        gx = Guarded(x.shape, x.dtype, dev, row=W, fill=x, src=True)
        gy = Guarded((B, 3 * H * r // 2, W * r), x.dtype, dev, row=W * r)
        for fill in (0xA5, 0x3C):
            _refill_outside(gx, fill)
            snap = gx.snapshot()
            with torch.inference_mode():                           # (the engine's workspace is an inference tensor)
                ws.fill_(0xFF)
            gy.raw[gy.start:gy.end].fill_(0x77)
            _native.check(eng.lib.mz_upscale(eng.handle, gx.ptr(), c.data_ptr() if c is not None else None,
                                             B if c is not None else 0, gy.ptr(), B, H, W, ws_ptr,
                                             ws.numel() - (ws_ptr - ws.data_ptr()), flags, stream.cuda_stream))
            torch.cuda.synchronize(dev)
            assert_guards(("y", gy))
            assert_unchanged(("x", gx, snap))
            assert np.array_equal(_np(gy.view), want), (name, dtype, fill)


# ---------------------------------------------------------------------------------------------------------------------
# 4. refusals and the workspace
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_refusals(dev):
    from ultrazoom_b200 import _native

    m, c = _model_for("2x-fused-f16", dev)
    eng = m._engine(dev)
    lib, h = eng.lib, eng.handle
    stream = torch.cuda.current_stream(dev)
    B, H, W = 1, 8, 16
    ws = eng.workspace(B, H + 2, W + 2, stream, _native.FLAG_CLAMP01 | _native.FLAG_YUV420 | _native.FLAG_IO_U16)
    ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
    wsb = ws.numel() - (ws_ptr - ws.data_ptr())
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device=dev)
    out = torch.zeros(1 << 22, dtype=torch.uint8, device=dev)
    cp = c[:1].data_ptr()
    Y, U8, U16, CL = _native.FLAG_YUV420, _native.FLAG_IO_U8, _native.FLAG_IO_U16, _native.FLAG_CLAMP01

    def upscale(flags, h_=H, w_=W):
        return lib.mz_upscale(h, buf.data_ptr(), cp, 1, out.data_ptr(), B, h_, w_, ws_ptr, wsb, flags, stream.cuda_stream)

    assert upscale(CL | Y | U8) == 0 and upscale(CL | Y | U16) == 0
    refused = {
        "odd H": upscale(CL | Y | U8, h_=7), "odd W": upscale(CL | Y | U16, w_=15),
        "fp32": upscale(CL | Y), "both element types": upscale(CL | Y | U8 | U16), "no clamp": upscale(Y | U8),
        "x nhwc": upscale(CL | Y | U8 | _native.FLAG_X_NHWC), "y nhwc": upscale(CL | Y | U8 | _native.FLAG_Y_NHWC),
        "u8 trunc": upscale(CL | Y | U8 | _native.FLAG_U8_TRUNC),
        "skip from buffer": upscale(CL | Y | U16 | _native.FLAG_SKIP_FROM_BUFFER),
        "both matrices": upscale(CL | Y | U8 | _native.FLAG_YUV_BT601 | _native.FLAG_YUV_BT2020),
        "colour without yuv": upscale(CL | U8 | _native.FLAG_YUV_BT601),
        "range without yuv": upscale(CL | U16 | _native.FLAG_YUV_FULL_RANGE),
        "window": lib.mz_upscale_window(h, buf.data_ptr(), cp, 1, out.data_ptr(), 2 * W, 4 * H * W, B, H, W, 0, H, 0, W,
                                        ws_ptr, wsb, CL | Y | U8, stream.cuda_stream),
        "stage": lib.mz_upscale_stage(h, buf.data_ptr(), cp, 1, out.data_ptr(), 0, 0, B, H, W, 0, 0, 0, 0, ws_ptr, wsb,
                                      CL | Y | U8, stream.cuda_stream, 0, 2),
        "host odd W": lib.mz_upscale_host(h, buf.cpu().data_ptr(), c[:1].cpu().data_ptr(), 1, out.cpu().data_ptr(), B, H,
                                          W - 1, CL | Y | U8),
        "kernel both matrices": lib.mz_yuv420_to_rgb16(buf.data_ptr(), out.data_ptr(), B, H, W,
                                                       Y | U8 | _native.FLAG_YUV_BT601 | _native.FLAG_YUV_BT2020,
                                                       stream.cuda_stream),
        "kernel odd W": lib.mz_rgb16_to_yuv420(buf.data_ptr(), out.data_ptr(), B, H, W - 1, Y | U16, stream.cuda_stream),
        "kernel no element type": lib.mz_yuv420_to_rgb16(buf.data_ptr(), out.data_ptr(), B, H, W, Y, stream.cuda_stream),
        "kernel misaligned": lib.mz_yuv420_to_rgb16(buf.data_ptr() + 2, out.data_ptr(), B, H, W, Y | U16, stream.cuda_stream),
    }
    for what, rc in refused.items():
        assert rc == _native.MZ_ERR_INVALID, (what, rc)
    torch.cuda.synchronize(dev)

    f = _yuv("bt709", False)
    x = _t(_frames(1, 8, 16, np.uint8, seed=1), dev)
    xf = torch.rand(1, 12, 16, device=dev)
    frame = torch.zeros(1, 3, 16, 32, device=dev)
    with pytest.raises(AssertionError):
        m.forward(x, c[:1], yuv=f)
    with pytest.raises(AssertionError):
        m.upscale(xf, c[:1], yuv=f)                                   # fp32 frames
    with pytest.raises(AssertionError):
        m.upscale(x[:, :7], c[:1], yuv=f)                             # 3H/2 rows: H would not be an even integer
    with pytest.raises(AssertionError):
        m.upscale(x[:, :, :15].contiguous(), c[:1], yuv=f)            # odd W (refused by the library)
    with pytest.raises(AssertionError):
        m.upscale(x, c[:1])                                           # a 3-D tensor without yuv= is no image
    with pytest.raises(AssertionError):
        m.upscale(x, c[:1], yuv=f, memory_format=torch.channels_last)
    with pytest.raises(AssertionError):
        m.upscale_into(x, c[:1], frame, (0, 8, 0, 16), (0, 0), yuv=f)
    with pytest.raises(AssertionError):
        m.upscale_stage(x, c[:1], frame, (0, 8, 0, 16), (0, 0), 0, 2, ws, yuv=f)
    with pytest.raises(AssertionError):
        m.capture(x, c[:1], clamp=False, yuv=f)
    with pytest.raises(AssertionError):
        m.upscale_host(x[:, :, :15].cpu().contiguous(), c[:1].cpu(), yuv=f)
    with pytest.raises(AssertionError):
        _yuv("bt2100", False)


@gpu
@pytest.mark.parametrize("name", ["2x-fused-f16", "3x", "4x", "2x-no-control"])
def test_workspace_adds_exactly_the_two_intermediates(dev, name):
    from ultrazoom_b200 import _native

    m, _ = _model_for(name, dev)
    eng = m._engine(dev)
    r = m.upscale_ratio
    align = lambda n: -(-n // 1024) * 1024                           # noqa: E731
    for B, H, W in ((1, 2, 2), (16, 540, 960), (3, 10, 22)):
        base, zero, yuv8, yuv16 = (C.c_size_t() for _ in range(4))
        _native.check(eng.lib.mz_workspace_bytes(eng.handle, B, H, W, C.byref(base)))
        _native.check(eng.lib.mz_workspace_bytes_flags(eng.handle, B, H, W, 0, C.byref(zero)))
        _native.check(eng.lib.mz_workspace_bytes_flags(eng.handle, B, H, W, _native.FLAG_CLAMP01 | _native.FLAG_YUV420 |
                                                       _native.FLAG_IO_U8, C.byref(yuv8)))
        _native.check(eng.lib.mz_workspace_bytes_flags(eng.handle, B, H, W, _native.FLAG_CLAMP01 | _native.FLAG_YUV420 |
                                                       _native.FLAG_IO_U16 | _native.FLAG_YUV_BT2020, C.byref(yuv16)))
        extra = align(B * 3 * H * W * 2) + align(B * 3 * H * W * r * r * 2)
        assert base.value == zero.value and yuv8.value == yuv16.value == base.value + extra, (name, B, H, W)
