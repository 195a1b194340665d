"""GPU: every kernel reads and writes only the elements it owns.

The value tests elsewhere hand the kernels fresh, exact-size allocations, so a store past the end of a tensor lands in
the caching allocator's slack and an element the kernel forgets to write keeps whatever the allocator left there.
Here every tensor a kernel touches is a view inside a larger buffer whose bytes before and after the view (the guard
bands, at least 8 image rows and 64 KiB each) hold a known pattern: NaN bits for float and 16-bit tensors (0xFF bytes
around what a kernel writes, a different NaN around what it only reads, so that a stray store of a value read from an
input's guard is not mistaken for an intact band), 0xA5 for 8-bit ones.  The C ABI entry points are called directly so
that the test chooses every pointer, and for each call

  (a) the output is pre-filled with NaN and then matches a float64 reference computed on the same rounded operands,
      at the tolerances the value tests state for that kernel;
  (b) no NaN is left in the output;
  (c) both guard bands of every output are unchanged, byte for byte;
  (d) every input, guards included, is byte-identical after the call (for the in-place fp32 stream: its guards);
  (e) channels the header says are "left untouched" are pre-filled with NaN and still NaN bit for bit; channels it says
      are zero-filled are zero.

Inputs carry NaN guard bands too, so a read past the end that reaches the arithmetic turns the result into NaN instead
of silently reading a neighbour; channels beyond cin_p of a wider input (which the header says are not read) are NaN.

At the model level the workspace (zf, zb, hidden and FiLM regions of one buffer, reused across calls, graph replays and
staged tiles) is filled with 0xFF between calls: a result must not depend on what the workspace held before the call.
"""
import ctypes as C
import math

import pytest
import torch
from torch.nn import functional as F

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# guarded buffers
# ---------------------------------------------------------------------------------------------------------------------
_INT = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}


def bits(t):
    """The raw bits of a tensor (any strides) as a same-size integer view; an all-ones (0xFF..) element is -1."""
    return t.view(_INT[t.element_size()])


def is_poison(t) -> bool:
    """Every element of a float / 16-bit tensor still holds the 0xFF.. NaN pattern, bit for bit."""
    return bool((bits(t) == -1).all())


class Guarded:
    """A contiguous view of `shape` / `dtype` inside a larger flat byte buffer.  The view starts on a 1024-byte boundary
    (the alignment real allocations have: TMA needs 16 B, the model workspace 1024 B); the bytes before and after it
    form the guard bands, each at least 8 image rows (`row` elements per row) and 64 KiB, filled with a pattern:

      * tensors a kernel writes: 0xFF bytes -- NaN in fp32, fp16 and bf16;
      * tensors a kernel only reads (`src=True`): the bytes A5 FF repeated -- 0xFFA5 / 0xFFA5FFA5, NaN in the three types
        too, but a different NaN: a stray store that copies an input's guard into an output's guard is still seen;
      * uint8 tensors: 0xA5."""

    def __init__(self, shape, dtype, device, row: int = 1, fill=None, src: bool = False):
        self.shape, self.dtype = tuple(shape), dtype
        isz = torch.empty((), dtype=dtype).element_size()
        self.nbytes = math.prod(self.shape) * isz
        guard = -(-max(64 << 10, 8 * row * isz) // 1024) * 1024
        pattern = [0xA5] if dtype == torch.uint8 else [0xA5, 0xFF] if src else [0xFF]
        total = guard + self.nbytes + guard + 1024
        self.expect = torch.tensor(pattern, dtype=torch.uint8).repeat(total // len(pattern)).to(device)
        self.raw = self.expect.clone()
        self.start = guard + (-self.raw.data_ptr()) % 1024
        self.end = self.start + self.nbytes
        self.view = self.raw[self.start:self.end].view(dtype).view(self.shape)
        if fill is not None:
            self.view.copy_(fill)

    def ptr(self, elem_offset: int = 0) -> int:
        return self.view.data_ptr() + elem_offset * self.view.element_size()

    def poison(self) -> "Guarded":
        """Fill the view itself with 0xFF bytes (NaN for float and 16-bit types)."""
        self.raw[self.start:self.end].fill_(0xFF)
        return self

    def snapshot(self):
        return self.raw.clone()

    def stray(self):
        """None when both guard bands hold their pattern; else where they changed, as byte offsets from the view:
        negative before its first byte, positive after its end (one past the last byte = +0)."""
        msgs = []
        isz = self.view.element_size()
        for side, lo_, hi_, base in (("before", 0, self.start, -self.start), ("after", self.end, self.raw.numel(), 0)):
            bad = torch.nonzero(self.raw[lo_:hi_] != self.expect[lo_:hi_]).flatten()
            if bad.numel():
                lo, hi = int(bad[0]) + base, int(bad[-1]) + base
                near = hi if side == "before" else lo
                msgs.append(f"{bad.numel()} guard byte(s) changed {side} the view, nearest at byte {near:+d} "
                            f"(element {near // isz:+d}), span [{lo:+d}, {hi:+d}]")
        return "; ".join(msgs) or None


def assert_guards(*named):
    """(c): every guard band intact."""
    for name, g in named:
        s = g.stray()
        assert s is None, f"{name}: {s}"


def assert_unchanged(*named):
    """(d): inputs byte-identical, guards included."""
    for name, g, snap in named:
        if not torch.equal(g.raw, snap):
            diff = torch.nonzero(g.raw != snap).flatten()
            assert False, f"input {name} was modified: {diff.numel()} byte(s), first at byte {int(diff[0]) - g.start:+d} of the view"


def test_guard_checker_reports_each_band():
    """CPU self-test: the checker is not vacuous -- one element written into either guard through the backing buffer is
    reported on the right side; the view itself may change freely; the view is 1024-byte aligned and the bands large."""
    for dt, shape, row in ((torch.float32, (2, 3, 5, 7), 7), (torch.float16, (1, 4, 9, 64), 9 * 64),
                           (torch.bfloat16, (3, 33), 33), (torch.uint8, (1, 3, 10, 4000), 4000)):
        g = Guarded(shape, dt, "cpu", row=row)
        isz = g.view.element_size()
        assert g.view.data_ptr() % 1024 == 0 and g.view.is_contiguous() and tuple(g.view.shape) == shape
        assert g.start >= max(64 << 10, 8 * row * isz) and g.raw.numel() - g.end >= max(64 << 10, 8 * row * isz)
        assert g.stray() is None
        g.view.fill_(3)                                            # writes inside the view are not a stray store
        assert g.stray() is None
        if dt != torch.uint8:
            g.poison()
            assert is_poison(g.view) and torch.isnan(g.view.float()).all()
        snap = g.snapshot()
        g.raw[g.start - isz:g.start].view(dt).fill_(1)             # the element just before the view
        s = g.stray()
        assert s is not None and "before" in s and f"span [{-isz:+d}, -1]" in s and "after" not in s, s
        g.raw[g.start - isz:g.start] = g.expect[g.start - isz:g.start]
        assert g.stray() is None and torch.equal(g.raw, snap)
        far = g.raw.numel() - isz                                  # the last element of the trailing band
        g.raw[g.end:g.end + isz].view(dt).fill_(1)
        g.raw[far:far + isz].view(dt).fill_(1)
        s = g.stray()
        assert s is not None and "after" in s and "before" not in s and "byte +0" in s, s
        with pytest.raises(AssertionError, match="after"):
            assert_guards(("x", g))
        with pytest.raises(AssertionError, match="modified"):
            assert_unchanged(("x", g, snap))
        if dt != torch.uint8:                                     # both guard patterns are NaN, and they differ
            src, out = Guarded(shape, dt, "cpu", row=row, src=True), Guarded(shape, dt, "cpu", row=row)
            for t in (src, out):
                assert torch.isnan(t.raw[:t.start - t.start % isz].view(dt).float()).all()
            out.raw[out.end:out.end + 1024] = src.raw[src.end:src.end + 1024]   # a store that copies an input's guard
            assert "after" in (out.stray() or ""), "a NaN copied from an input's guard band went unseen"


# ---------------------------------------------------------------------------------------------------------------------
# GPU plumbing
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _lib():
    from ultrazoom_b200 import _native

    lib = _native.load()
    assert lib.mz_device_count() >= 1, "no sm_100 device: the CUDA path cannot run"
    return _native, lib


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _pad(c):
    return _lib()[1].mz_padded_channels(c)


def _ulp(dt):
    return 2.0 ** -11 if dt == torch.float16 else 2.0 ** -8


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _maxerr(a, b):
    return (a.double().cpu() - b.double().cpu()).abs().max().item()


def _no_nan(name, t):
    n = torch.isnan(t.float()).sum().item()
    assert n == 0, f"{name}: {n} element(s) never written (still NaN)"


# ---------------------------------------------------------------------------------------------------------------------
# bicubic
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("r,tol", [(2, 2e-6), (3, 1e-4), (4, 2e-6)])
@pytest.mark.parametrize("shape", [(1, 3, 1, 1), (1, 3, 5, 129), (2, 3, 7, 300), (1, 1, 2, 300), (3, 3, 9, 126)])
def test_bicubic(dev, r, tol, shape):
    native, lib = _lib()
    B, Cc, H, W = shape
    x = torch.rand(shape, generator=torch.Generator().manual_seed(sum(shape) + r))
    gx = Guarded(shape, torch.float32, dev, row=W, fill=x, src=True)
    gy = Guarded((B, Cc, H * r, W * r), torch.float32, dev, row=W * r).poison()
    sx = gx.snapshot()
    native.check(lib.mz_bicubic_f32(gx.ptr(), gy.ptr(), B * Cc, H, W, r, _stream(dev)))
    torch.cuda.synchronize()
    ref = F.interpolate(x.double(), scale_factor=r, mode="bicubic")
    _no_nan("y", gy.view)
    assert _maxerr(gy.view, ref) <= tol
    assert_guards(("y", gy))
    assert_unchanged(("x", gx, sx))


# ---------------------------------------------------------------------------------------------------------------------
# stem
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("C,zb_pitch,shape", [(16, 0, (2, 9, 11)), (48, 0, (1, 1, 1)), (48, 64, (2, 7, 129)),
                                              (54, 0, (1, 5, 252)), (54, 64, (1, 3, 126)), (96, 0, (2, 4, 256)),
                                              (16, 64, (1, 2, 128))])
def test_stem_pack(dev, C, zb_pitch, shape, dt):
    native, lib = _lib()
    g = torch.Generator().manual_seed(C + zb_pitch + sum(shape))
    B, H, W = shape
    Cp = _pad(C)
    Cz = zb_pitch or Cp
    x = torch.rand(B, 3, H, W, generator=g)
    w = torch.zeros(Cp, 3)
    b = torch.zeros(Cp)
    w[:C] = torch.randn(C, 3, generator=g) * 0.5
    b[:C] = torch.randn(C, generator=g) * 0.1
    gx = Guarded(x.shape, torch.float32, dev, row=W, fill=x, src=True)
    gw = Guarded(w.shape, torch.float32, dev, fill=w, src=True)
    gb = Guarded(b.shape, torch.float32, dev, fill=b, src=True)
    gzf = Guarded((B, H, W, Cp), torch.float32, dev, row=W * Cp).poison()
    gzb = Guarded((B, H, W, Cz), dt, dev, row=W * Cz).poison()
    snaps = [(n, t, t.snapshot()) for n, t in (("x", gx), ("w", gw), ("bias", gb))]
    native.check(lib.mz_stem_pack(gx.ptr(), gw.ptr(), gb.ptr(), gzf.ptr(), gzb.ptr(), B, H, W, Cp, zb_pitch,
                                  native.dtype_code(dt), _stream(dev)))
    torch.cuda.synchronize()
    ref = torch.einsum("bchw,nc->bhwn", x.double(), w.double()) + b.double()
    zf, zb = gzf.view.cpu(), gzb.view.cpu()
    _no_nan("zf", zf)
    _no_nan("zb", zb)
    assert _maxerr(zf[..., :C], ref[..., :C]) <= 1e-5
    assert bool((bits(zf[..., C:]) == 0).all())                        # padded channels: +0.0
    n = min(Cp, Cz)
    assert torch.equal(bits(zb[..., :n]), bits(zf[..., :n].to(dt)))    # the shadow is exactly round16(zf)
    assert bool((bits(zb[..., n:]) == 0).all())                        # a wider shadow pitch is zero-filled
    assert_guards(("zf", gzf), ("zb", gzb))
    assert_unchanged(*snaps)


# ---------------------------------------------------------------------------------------------------------------------
# FiLM table
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("L,B,hC", [(3, 2, 108), (1, 1, 96), (2, 3, 20)])
@pytest.mark.parametrize("broadcast", [False, True])
def test_control_film(dev, L, B, hC, broadcast):
    native, lib = _lib()
    g = torch.Generator().manual_seed(L * 100 + B + hC)
    Fc = 3
    hCp = _pad(hC)
    w, bb = torch.randn(L, 2 * hC, Fc, generator=g), torch.randn(L, 2 * hC, generator=g)
    c = torch.rand(1 if broadcast else B, Fc, generator=g)
    gc = Guarded(c.shape, torch.float32, dev, fill=c, src=True)
    gw = Guarded(w.shape, torch.float32, dev, fill=w, src=True)
    gb = Guarded(bb.shape, torch.float32, dev, fill=bb, src=True)
    gf = Guarded((L, B, 2, hCp), torch.float32, dev, row=2 * hCp).poison()
    snaps = [(n, t, t.snapshot()) for n, t in (("c", gc), ("w", gw), ("b", gb))]
    native.check(lib.mz_control_film(gc.ptr(), c.shape[0], gw.ptr(), gb.ptr(), gf.ptr(), L, B, Fc, hC, hCp, _stream(dev)))
    torch.cuda.synchronize()
    gl = torch.einsum("bf,lnf->lbn", c.double(), w.double()) + bb.double()[:, None, :]
    gl = gl.expand(-1, B, -1)
    film = gf.view.cpu()
    _no_nan("film", film)
    assert _maxerr(film[:, :, 0, :hC], 1 + gl[..., :hC]) <= 1e-5
    assert _maxerr(film[:, :, 1, :hC], gl[..., hC:]) <= 1e-5
    assert bool((film[:, :, 0, hC:] == 1).all()) and bool((bits(film[:, :, 1, hC:]) == 0).all())   # pad: scale 1, shift 0
    assert_guards(("film", gf))
    assert_unchanged(*snaps)


# ---------------------------------------------------------------------------------------------------------------------
# tcgen05 / SIMT convolution, modes 0 and 1
# ---------------------------------------------------------------------------------------------------------------------
CONV_CASES = [
    # cin, cout, (B, H, W), tune, channels before the slice, channels after it, extra input channels beyond cin_p[, modes]
    (48, 96, (2, 13, 150), {}, 0, 0, 0),
    (48, 96, (2, 13, 150), {}, 0, 32, 0),                         # out_pitch > cout_p
    (96, 48, (2, 13, 150), {}, 16, 16, 0),                        # a channel slice of a wider out / zf
    (96, 48, (2, 13, 150), {}, 0, 0, 16),                         # in_pitch > cin_p, NaN beyond cin_p
    (16, 32, (1, 1, 1), {}, 0, 16, 0),
    (54, 108, (1, 10, 70), {}, 0, 16, 0),
    (32, 32, (1, 5, 130), dict(rows=1), 0, 0, 0),
    (96, 192, (1, 21, 300), dict(pair=1), 0, 0, 16),
    (64, 64, (1, 5, 130), dict(pair=1), 64, 0, 0),
    (48, 96, (2, 13, 150), dict(resident=1), 0, 32, 0),
    (48, 96, (2, 13, 150), dict(resident=2), 32, 0, 0),
    (64, 128, (1, 9, 257), dict(resident=1, max_ctas=2), 0, 0, 0),
    (48, 96, (2, 41, 300), dict(fuse=1, max_ctas=3), 0, 0, 0, (0,)),  # (the fused-row kernel has no conv2 of this shape)
    (96, 48, (2, 41, 300), dict(fuse=1, max_ctas=3), 0, 16, 0),
    (32, 48, (1, 7, 130), dict(fuse=1, rows=4), 16, 16, 0),
    (96, 192, (2, 30, 260), dict(cluster=4), 0, 0, 0),
    (48, 96, (2, 13, 150), dict(cluster=4, max_ctas=6), 0, 0, 16),
    (48, 96, (2, 13, 150), dict(epi_warps=4), 32, 32, 0),
    (96, 48, (1, 5, 700), dict(epi_warps=4, rows=4), 0, 0, 0),
    (96, 192, (1, 9, 257), dict(kc=16, b_stages=2, halo_mode=1), 0, 0, 16),
    (48, 96, (2, 13, 150), dict(halo_mode=1), 16, 0, 0),
]


def _conv_operands(cin, cout, shape, seed, dt):
    g = torch.Generator().manual_seed(seed)
    B, H, W = shape
    cin_p, cout_p = _pad(cin), _pad(cout)
    inp = torch.zeros(B, H, W, cin_p, dtype=dt)
    inp[..., :cin] = torch.randn(B, H, W, cin, generator=g).to(dt)
    w = torch.randn(cout, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    film = torch.ones(B, 2, cout_p)
    film[:, 0, :cout] = 1 + 0.3 * torch.randn(B, cout, generator=g)
    film[:, 1] = 0
    film[:, 1, :cout] = 0.3 * torch.randn(B, cout, generator=g)
    zf0 = torch.zeros(B, H, W, cout_p)
    zf0[..., :cout] = torch.randn(B, H, W, cout, generator=g)
    acc = F.conv2d(_nchw(inp[..., :cin]).double(), w.to(dt).double(), padding=1).permute(0, 2, 3, 1)
    return inp, w, film, zf0, acc


def _conv_id(case):
    cin, cout, shape, tune, before, after, extra = case[:7]
    t = ",".join(f"{k}={v}" for k, v in tune.items()) or "default"
    return f"{cin}-{cout}-{'x'.join(map(str, shape))}-{t}-slice{before}+{after}-in{extra}"


@gpu
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("case", CONV_CASES, ids=[_conv_id(c) for c in CONV_CASES])
def test_conv3x3(dev, case, dt):
    from ultrazoom_b200 import ops

    native, lib = _lib()
    cin, cout, (B, H, W), tune, before, after, extra = case[:7]
    cin_p, cout_p = _pad(cin), _pad(cout)
    modes = case[7] if len(case) > 7 else (0, 1) if cout_p <= 128 else (0,)   # (mode 1 runs up to 128 channels a launch)
    inp, w, film, zf0, acc = _conv_operands(cin, cout, (B, H, W), cin + cout + H + W, dt)
    P = before + cout_p + after                                   # channel pitch of out (and of zf in mode 1)
    Pin = cin_p + extra
    gin = Guarded((B, H, W, Pin), dt, dev, row=W * Pin, src=True)
    gin.view[..., :cin_p].copy_(inp)
    bits(gin.view[..., cin_p:]).fill_(-1)                         # beyond cin_p: not read, so NaN
    gw = Guarded((9, cout_p, cin_p), dt, dev, fill=ops.pack_conv_weight(w, dev, dtype=dt), src=True)
    gfilm = Guarded(film.shape, torch.float32, dev, fill=film, src=True)
    t = native.tune(**tune)
    paths = [True] + ([False] if not tune else [])                # the SIMT twin has no tunables
    sl = slice(before, before + cout_p)
    for use_tc in paths:
        for mode in modes:
            gout = Guarded((B, H, W, P), dt, dev, row=W * P).poison()
            gzf = None
            if mode == 1:
                gzf = Guarded((B, H, W, P), torch.float32, dev, row=W * P).poison()
                gzf.view[..., sl].copy_(zf0)
            ins = [("in", gin), ("w", gw)] + ([("film", gfilm)] if mode == 0 else [])
            snaps = [(n, g, g.snapshot()) for n, g in ins]
            native.check(lib.mz_conv3x3(
                gin.ptr(), gw.ptr(), mode, gfilm.ptr() if mode == 0 else None, gout.ptr(before),
                gzf.ptr(before) if mode == 1 else None, B, H, W, cin_p, Pin if Pin != cin_p else 0, cout_p,
                P if P != cout_p else 0, P if (mode == 1 and P != cout_p) else 0, native.dtype_code(dt),
                1 if use_tc else 0, C.byref(t) if use_tc else None, _stream(dev)))
            torch.cuda.synchronize()
            what = f"mode {mode} {'tcgen05' if use_tc else 'SIMT'}"
            out = gout.view.cpu()
            assert is_poison(out[..., :before]) and is_poison(out[..., before + cout_p:]), f"{what}: a channel outside the slice was written"
            _no_nan(f"{what} out", out[..., sl])
            if mode == 0:
                ref = F.silu(acc * film[:, 0][:, None, None, :cout].double() + film[:, 1][:, None, None, :cout].double())
                tol = (2 * _ulp(dt) + 5e-4) * max(1.0, ref.abs().max().item())
                assert _maxerr(out[..., before:before + cout], ref) <= tol, what
                assert bool((out[..., before + cout:before + cout_p].float() == 0).all()), what
            else:
                zf = gzf.view.cpu()
                assert is_poison(zf[..., :before]) and is_poison(zf[..., before + cout_p:]), f"{what}: zf outside the slice was written"
                assert _maxerr(zf[..., before:before + cout], zf0[..., :cout].double() + acc) <= 1e-4, what
                assert bool((bits(zf[..., before + cout:before + cout_p]) == 0).all()), what
                assert torch.equal(bits(out[..., sl]), bits(zf[..., sl].to(dt))), what   # shadow = round16(zf)
                assert_guards(("zf", gzf))
            assert_guards(("out", gout))
            assert_unchanged(*snaps)


# ---------------------------------------------------------------------------------------------------------------------
# fused encoder block
# ---------------------------------------------------------------------------------------------------------------------
FUSED_CASES = [
    # (B, H, W), seg_rows, max_ctas  (the shapes of tests/test_gpu_fused_block.py)
    ((1, 1, 1), 0, 0), ((1, 1, 126), 0, 0), ((1, 2, 127), 0, 0), ((1, 3, 130), 0, 0), ((1, 5, 252), 0, 0),
    ((1, 4, 253), 0, 0), ((2, 9, 300), 0, 0), ((1, 23, 260), 8, 0), ((1, 23, 260), 3, 2), ((1, 40, 140), 1, 2),
    ((2, 17, 400), 5, 4), ((1, 64, 520), 0, 6), ((3, 7, 100), 2, 2), ((1, 33, 960), 0, 0),
]


@gpu
@pytest.mark.parametrize("with_film", [True, False])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape,seg_rows,max_ctas", FUSED_CASES)
def test_block_fused(dev, shape, seg_rows, max_ctas, dt, with_film):
    from ultrazoom_b200 import ops

    native, lib = _lib()
    B, H, W = shape
    g = torch.Generator().manual_seed(sum(shape) + seg_rows)
    zf0 = torch.randn(B, H, W, 48, generator=g)
    zb = zf0.to(dt)
    w1 = torch.randn(96, 48, 3, 3, generator=g) / (3.0 * 48 ** 0.5)
    w2 = torch.randn(48, 96, 3, 3, generator=g) / (3.0 * 96 ** 0.5)
    film = torch.empty(B, 2, 96)
    film[:, 0] = 1 + 0.3 * torch.randn(B, 96, generator=g)
    film[:, 1] = 0.3 * torch.randn(B, 96, generator=g)
    gzb = Guarded(zb.shape, dt, dev, row=W * 48, fill=zb, src=True)
    gout = Guarded(zb.shape, dt, dev, row=W * 48).poison()
    gzf = Guarded(zf0.shape, torch.float32, dev, row=W * 48, fill=zf0)
    gw1 = Guarded((9, 96, 48), dt, dev, fill=ops.pack_conv_weight(w1, dev, dtype=dt), src=True)
    gw2 = Guarded((9, 48, 96), dt, dev, fill=ops.pack_conv_weight(w2, dev, dtype=dt), src=True)
    gfilm = Guarded(film.shape, torch.float32, dev, fill=film, src=True)
    ins = [("zb_in", gzb), ("w1", gw1), ("w2", gw2)] + ([("film", gfilm)] if with_film else [])
    snaps = [(n, t, t.snapshot()) for n, t in ins]
    native.check(lib.mz_block_fused(gzb.ptr(), gout.ptr(), gzf.ptr(), gw1.ptr(), gw2.ptr(),
                                    gfilm.ptr() if with_film else None, B, H, W, native.dtype_code(dt), seg_rows, max_ctas,
                                    _stream(dev)))
    torch.cuda.synchronize()
    acc1 = F.conv2d(_nchw(zb).double(), w1.to(dt).double(), padding=1)
    if with_film:
        acc1 = acc1 * film[:, 0].double()[:, :, None, None] + film[:, 1].double()[:, :, None, None]
    hid = F.silu(acc1).to(dt).double()
    ref = zf0.double() + F.conv2d(hid, w2.to(dt).double(), padding=1).permute(0, 2, 3, 1)
    zf, out = gzf.view.cpu(), gout.view.cpu()
    _no_nan("zb_out", out)
    _no_nan("zf", zf)
    assert _maxerr(zf, ref) <= (3e-3 if dt == torch.float16 else 2e-2)
    assert torch.equal(bits(out), bits(zf.to(dt)))                    # the shadow is exactly round16(zf)
    assert_guards(("zb_out", gout), ("zf", gzf))
    assert_unchanged(*snaps)


# ---------------------------------------------------------------------------------------------------------------------
# head: conv3x3 + PixelShuffle + skip + clamp
# ---------------------------------------------------------------------------------------------------------------------
HEAD_CASES = [
    # cin, (B, H, W), extra input channels, tune (None: tcgen05 default and the SIMT twin)
    (48, (2, 7, 190), 0, None),
    (96, (1, 9, 129), 16, None),
    (54, (1, 1, 3), 0, None),
    (48, (1, 13, 300), 0, dict(fuse=1)),
    (48, (2, 5, 126), 16, dict(fuse=1)),
]


@gpu
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("r,tol", [(2, 1e-4), (3, 2e-4), (4, 1e-4)])
@pytest.mark.parametrize("cin,shape,extra,tune", HEAD_CASES)
def test_head_shuffle_add(dev, cin, shape, extra, tune, r, tol, dt):
    from ultrazoom_b200 import ops

    native, lib = _lib()
    g = torch.Generator().manual_seed(cin + sum(shape) + r)
    B, H, W = shape
    cin_p = _pad(cin)
    Pin = cin_p + extra
    zb = torch.zeros(B, H, W, cin_p, dtype=dt)
    zb[..., :cin] = torch.randn(B, H, W, cin, generator=g).to(dt)
    w = torch.randn(3 * r * r, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
    x = torch.rand(B, 3, H, W, generator=g)
    wp = ops.pack_conv_weight(w, dev, dtype=dt)
    gzb = Guarded((B, H, W, Pin), dt, dev, row=W * Pin, src=True)
    gzb.view[..., :cin_p].copy_(zb)
    bits(gzb.view[..., cin_p:]).fill_(-1)
    gw = Guarded(wp.shape, dt, dev, fill=wp, src=True)
    gx = Guarded(x.shape, torch.float32, dev, row=W, fill=x, src=True)
    u = F.pixel_shuffle(F.conv2d(_nchw(zb[..., :cin]).double(), w.to(dt).double(), padding=1), r)
    s = F.interpolate(x.double(), scale_factor=r, mode="bicubic")
    bic = ops.bicubic(x.to(dev), r)                               # what skip mode 1 finds in y
    t = native.tune(**(tune or {}))
    for use_tc in ([True, False] if tune is None else [True]):
        for skip_mode, clamp in ((2, True), (2, False), (1, False), (1, True), (0, False)):
            gy = Guarded((B, 3, H * r, W * r), torch.float32, dev, row=W * r)
            if skip_mode == 1:
                gy.view.copy_(bic)
            else:
                gy.poison()
            ins = [("zb", gzb), ("w", gw)] + ([("x", gx)] if skip_mode == 2 else [])
            snaps = [(n, t_, t_.snapshot()) for n, t_ in ins]
            native.check(lib.mz_head_shuffle_add(
                gzb.ptr(), gw.ptr(), gx.ptr() if skip_mode == 2 else None, gy.ptr(), B, H, W, cin_p,
                Pin if Pin != cin_p else 0, r, skip_mode, 1 if clamp else 0, native.dtype_code(dt), 1 if use_tc else 0,
                C.byref(t) if use_tc else None, _stream(dev)))
            torch.cuda.synchronize()
            ref = u + (s if skip_mode == 2 else bic.cpu().double() if skip_mode == 1 else 0)
            if clamp:
                ref = ref.clamp(0, 1)
            what = f"skip {skip_mode} clamp {clamp} {'tcgen05' if use_tc else 'SIMT'}"
            _no_nan(what, gy.view)
            assert _maxerr(gy.view, ref) <= tol, what
            assert_guards(("y", gy))
            assert_unchanged(*snaps)


# ---------------------------------------------------------------------------------------------------------------------
# U-Net operators on NHWC fp32 feature maps
# ---------------------------------------------------------------------------------------------------------------------
TF32_TOL = 3e-3      # x the output scale (tests/test_gpu_unet_ops.py)
MATHS = ["tf32", "fp32"]


def _feature_map(shape, C, P, g, dev, row_w):
    """(B,H,W,P) guarded fp32 map: C logical channels of data, NaN in the channels beyond C (not read)."""
    v = torch.randn(*shape, C, generator=g)
    gm = Guarded((*shape, P), torch.float32, dev, row=row_w * P, src=True).poison()
    gm.view[..., :C].copy_(v)
    return v, gm


def _check_out16(name, g16, out, C, dt):
    o16 = g16.view.cpu()
    assert torch.equal(bits(o16[..., :C]), bits(out[..., :C].to(dt))), f"{name}: shadow != round16(out)"
    assert is_poison(o16[..., C:]), f"{name}: shadow pad channels were written"
    assert_guards((name + "16", g16))


@gpu
@pytest.mark.parametrize("math_", MATHS)
@pytest.mark.parametrize("dt", [None, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape,C,P", [((2, 21, 150), 40, 48), ((1, 1, 1), 16, 24), ((3, 5, 257), 32, 40),
                                       ((1, 9, 126), 96, 104)])
def test_adaptive_mix(dev, shape, C, P, dt, math_):
    native, lib = _lib()
    g = torch.Generator().manual_seed(C + P + sum(shape))
    npix = math.prod(shape)
    x, gx = _feature_map(shape, C, P, g, dev, shape[2])
    z, gz = _feature_map(shape, C, P, g, dev, shape[2])
    w = torch.randn(C, 2 * C, generator=g) / (2 * C) ** 0.5
    gw = Guarded(w.shape, torch.float32, dev, fill=w, src=True)
    gout = Guarded((*shape, P), torch.float32, dev, row=shape[2] * P).poison()
    g16 = Guarded((*shape, P), dt, dev, row=shape[2] * P).poison() if dt is not None else None
    snaps = [(n, t, t.snapshot()) for n, t in (("x", gx), ("z", gz), ("w", gw))]
    alpha = 0.4
    native.check(lib.mz_adaptive_mix(gx.ptr(), gz.ptr(), gw.ptr(), alpha, gout.ptr(), g16.ptr() if g16 else None, npix, C, P,
                                     native.dtype_code(dt or torch.float16),
                                     native.MATH_TF32 if math_ == "tf32" else native.MATH_FP32, _stream(dev)))
    torch.cuda.synchronize()
    xd, zd = x.double(), z.double()
    beta = torch.sigmoid(torch.cat([xd, zd], -1) @ w.double().t())
    wgt = torch.sigmoid(torch.tensor(alpha, dtype=torch.float64)) * beta
    ref = (1 - wgt) * xd + wgt * zd
    out = gout.view.cpu()
    _no_nan("out", out[..., :C])
    assert _maxerr(out[..., :C], ref) <= (TF32_TOL * ref.abs().max().item() if math_ == "tf32" else 2e-5)
    assert is_poison(out[..., C:]), "pad channels of out were written"
    assert_guards(("out", gout))
    if g16 is not None:
        _check_out16("out", g16, out, C, dt)
    assert_unchanged(*snaps)


@gpu
@pytest.mark.parametrize("math_", MATHS)
@pytest.mark.parametrize("dt", [None, torch.float16])
@pytest.mark.parametrize("f,shape,Cin,Pin,Co,Po", [(2, (2, 21, 150), 40, 48, 72, 80), (3, (2, 21, 150), 40, 48, 72, 80),
                                                   (4, (1, 9, 257), 32, 32, 64, 72), (2, (1, 3, 2), 16, 24, 32, 40),
                                                   (3, (3, 7, 128), 48, 56, 24, 24)])
def test_pixel_crush(dev, f, shape, Cin, Pin, Co, Po, dt, math_):
    native, lib = _lib()
    g = torch.Generator().manual_seed(f + Cin + Co + sum(shape))
    B, H, W = shape
    Ho, Wo = H // f, W // f
    x, gx = _feature_map(shape, Cin, Pin, g, dev, W)
    wc = torch.randn(Co, Cin, f, f, generator=g) / (f * f * Cin) ** 0.5
    wt = wc.permute(0, 2, 3, 1).reshape(Co, f * f * Cin).contiguous()
    gw = Guarded(wt.shape, torch.float32, dev, fill=wt, src=True)
    gout = Guarded((B, Ho, Wo, Po), torch.float32, dev, row=Wo * Po).poison()
    g16 = Guarded((B, Ho, Wo, Po), dt, dev, row=Wo * Po).poison() if dt is not None else None
    snaps = [(n, t, t.snapshot()) for n, t in (("in", gx), ("w", gw))]
    native.check(lib.mz_pixel_crush(gx.ptr(), gw.ptr(), gout.ptr(), g16.ptr() if g16 else None, B, H, W, Cin, Co, f, Pin, Po,
                                    native.dtype_code(dt or torch.float16),
                                    native.MATH_TF32 if math_ == "tf32" else native.MATH_FP32, _stream(dev)))
    torch.cuda.synchronize()
    ref = F.conv2d(_nchw(x).double(), wc.double(), stride=f).permute(0, 2, 3, 1)
    out = gout.view.cpu()
    _no_nan("out", out[..., :Co])
    assert _maxerr(out[..., :Co], ref) <= (TF32_TOL * ref.abs().max().item() if math_ == "tf32" else 2e-5)
    assert is_poison(out[..., Co:]), "pad channels of out were written"
    assert_guards(("out", gout))
    if g16 is not None:
        _check_out16("out", g16, out, Co, dt)
    assert_unchanged(*snaps)


@gpu
@pytest.mark.parametrize("r", [2, 3, 4])
@pytest.mark.parametrize("dt", [None, torch.bfloat16])
@pytest.mark.parametrize("shape,C,extra_in,extra_out", [((2, 5, 33), 8, 0, 0), ((1, 3, 130), 12, 4, 4), ((1, 1, 1), 3, 1, 5),
                                                         ((2, 2, 64), 16, 8, 8)])
def test_pixel_shuffle_nhwc(dev, shape, C, extra_in, extra_out, r, dt):
    """Reads the first C r r channels of each input pixel and writes channels [0, C) of each output pixel; channels beyond
    them (pitch_in / pitch_out) are neither read nor written."""
    native, lib = _lib()
    g = torch.Generator().manual_seed(C + r + sum(shape))
    B, H, W = shape
    Pi, Po = C * r * r + extra_in, C + extra_out
    x, gx = _feature_map(shape, C * r * r, Pi, g, dev, W)
    gout = Guarded((B, H * r, W * r, Po), torch.float32, dev, row=W * r * Po).poison()
    g16 = Guarded((B, H * r, W * r, Po), dt, dev, row=W * r * Po).poison() if dt is not None else None
    snaps = [("in", gx, gx.snapshot())]
    native.check(lib.mz_pixel_shuffle_nhwc(gx.ptr(), gout.ptr(), g16.ptr() if g16 else None, B, H, W, C, r, Pi, Po,
                                           native.dtype_code(dt or torch.float16), _stream(dev)))
    torch.cuda.synchronize()
    ref = F.pixel_shuffle(_nchw(x).double(), r).permute(0, 2, 3, 1)
    out = gout.view.cpu()
    _no_nan("out", out[..., :C])
    assert torch.equal(out[..., :C].double(), ref)
    assert is_poison(out[..., C:]), "pad channels of out were written"
    assert_guards(("out", gout))
    if g16 is not None:
        _check_out16("out", g16, out, C, dt)
    assert_unchanged(*snaps)


@gpu
@pytest.mark.parametrize("shape,C,Pi,Po,target", [((2, 9, 70), 16, 16, 16, (7, 73)), ((1, 5, 130), 12, 16, 20, (8, 126)),
                                                  ((3, 4, 5), 3, 5, 7, (6, 3)), ((1, 1, 1), 4, 8, 4, (2, 2)),
                                                  ((2, 11, 129), 8, 8, 12, (11, 128))])
def test_crop_feature_maps(dev, shape, C, Pi, Po, target):
    """Writes channels [0, C) of every output pixel -- the input's centre crop, zeros where the target is larger -- and
    leaves channels beyond C (pitch_out) alone; the input's channels beyond C are not read."""
    native, lib = _lib()
    g = torch.Generator().manual_seed(C + Pi + Po + sum(shape))
    B, H, W = shape
    th, tw = target
    x, gx = _feature_map(shape, C, Pi, g, dev, W)
    gout = Guarded((B, th, tw, Po), torch.float32, dev, row=tw * Po).poison()
    snaps = [("in", gx, gx.snapshot())]
    native.check(lib.mz_crop_feature_maps(gx.ptr(), gout.ptr(), B, H, W, C, th, tw, Pi, Po, _stream(dev)))
    torch.cuda.synchronize()
    ref = torch.zeros(B, th, tw, C)
    oy, ox = (H - th) // 2 if H > th else -((th - H) // 2), (W - tw) // 2 if W > tw else -((tw - W) // 2)
    for y in range(th):
        for xx in range(tw):
            iy, ix = y + oy, xx + ox
            if 0 <= iy < H and 0 <= ix < W:
                ref[:, y, xx] = x[:, iy, ix]
    out = gout.view.cpu()
    _no_nan("out", out[..., :C])
    assert torch.equal(bits(out[..., :C]), bits(ref))             # zero padding is +0.0
    assert is_poison(out[..., C:]), "pad channels of out were written"
    assert_guards(("out", gout))
    assert_unchanged(*snaps)


@gpu
@pytest.mark.parametrize("shape,C,P,Fq", [((2, 9, 70), 16, 24, 3), ((1, 1, 1), 8, 8, 1), ((3, 5, 129), 20, 32, 5)])
def test_quality_assessor(dev, shape, C, P, Fq):
    native, lib = _lib()
    g = torch.Generator().manual_seed(C + P + Fq + sum(shape))
    B, H, W = shape
    x, gx = _feature_map(shape, C, P, g, dev, W)
    wq, bq = torch.randn(Fq, C, 3, 3, generator=g) / (9 * C) ** 0.5, torch.randn(Fq, generator=g)
    wt = wq.permute(0, 2, 3, 1).reshape(Fq, 9 * C).contiguous()
    gw = Guarded(wt.shape, torch.float32, dev, fill=wt, src=True)
    gb = Guarded(bq.shape, torch.float32, dev, fill=bq, src=True)
    gout = Guarded((B, Fq), torch.float32, dev).poison()
    snaps = [(n, t, t.snapshot()) for n, t in (("in", gx), ("w", gw), ("b", gb))]
    native.check(lib.mz_quality_assessor(gx.ptr(), gw.ptr(), gb.ptr(), gout.ptr(), B, H, W, C, Fq, P, _stream(dev)))
    torch.cuda.synchronize()
    ref = F.conv2d(_nchw(x).double(), wq.double(), bq.double(), padding=1).mean(dim=(2, 3))
    _no_nan("out", gout.view)
    assert _maxerr(gout.view, ref) <= 2e-5
    assert_guards(("out", gout))
    assert_unchanged(*snaps)


# ---------------------------------------------------------------------------------------------------------------------
# model level: the workspace never leaks into a result
# ---------------------------------------------------------------------------------------------------------------------
def _model(cfg, dev, seed, operand_dtype="float16"):
    from ultrazoom_b200 import MewZoom

    torch.manual_seed(seed)
    return MewZoom(**cfg, operand_dtype=operand_dtype).to(dev).eval()


def _ctrl(name, L):
    from ultrazoom_b200 import MODEL_CONFIGS

    cfg = dict(MODEL_CONFIGS[name])
    cfg["num_encoder_layers"] = L
    return cfg


MODEL_CASES = {
    "2x-fused-f16": (lambda: _ctrl("MewZoom-2X-Ctrl", 3), "float16", {}, (2, 3, 37, 131)),
    "2x-fused-bf16": (lambda: _ctrl("MewZoom-2X-Ctrl", 3), "bfloat16", {}, (1, 3, 21, 253)),
    "2x-two-kernels": (lambda: _ctrl("MewZoom-2X-Ctrl", 3), "float16", dict(block=2), (2, 3, 19, 127)),
    "2x-simt": (lambda: _ctrl("MewZoom-2X-Ctrl", 2), "float16", "simt", (1, 3, 13, 70)),
    "3x": (lambda: _ctrl("MewZoom-3X-Ctrl", 2), "float16", {}, (2, 3, 17, 129)),
    "3x-dense7": (lambda: _ctrl("MewZoom-3X-Ctrl", 2), "float16", "dense7", (1, 3, 25, 126)),
    "4x-pair": (lambda: _ctrl("MewZoom-4X-Ctrl", 2), "float16", {}, (1, 3, 33, 130)),
    "2x-c160-sliced": (lambda: dict(upscale_ratio=2, num_channels=160, hidden_ratio=2, num_encoder_layers=2,
                                    control_features=3), "float16", {}, (2, 3, 15, 129)),
}


@gpu
@pytest.mark.parametrize("name", list(MODEL_CASES))
def test_poisoned_workspace_changes_nothing(dev, name, monkeypatch):
    """upscale, forward and 8-bit upscale: the same result bit for bit whether the engine's workspace held the previous
    call's state, zeros or 0xFF bytes (NaN in every fp32 / 16-bit region) when the call began."""
    from ultrazoom_b200 import _native

    make_cfg, odt, how, shape = MODEL_CASES[name]
    if how == "dense7":
        monkeypatch.setenv("MZ_DENSE_LAYOUT", "7")                 # read when the native model is created
    m = _model(make_cfg(), dev, seed=sum(shape), operand_dtype=odt)
    if isinstance(how, dict) and how:
        m.set_conv_tune(0, dev, **how)
    if how == "simt":
        m._flags_extra = _native.FLAG_SIMT_CONV
    eng = m._engine(dev)
    if name.startswith("2x-fused"):
        assert eng.lib.mz_model_fused_block(eng.handle) == 1
    if name == "2x-two-kernels":
        assert eng.lib.mz_model_fused_block(eng.handle) == 0
    g = torch.Generator().manual_seed(7 + sum(shape))
    x = torch.rand(shape, generator=g).to(dev)
    c = torch.rand(shape[0], 3, generator=g).to(dev)
    x8 = (x * 255).to(torch.uint8)
    for what, fn, xx in (("upscale", m.upscale, x), ("forward", m.forward, x), ("upscale u8", m.upscale, x8)):
        y0 = fn(xx, c)
        if xx.dtype != torch.uint8:
            _no_nan(what, y0)
        for fill in (0x00, 0xFF):
            with torch.inference_mode():                           # (the workspace was allocated inside upscale)
                eng.ws.fill_(fill)
            y = fn(xx, c)
            assert torch.equal(y, y0), (name, what, hex(fill), (y.float() - y0.float()).abs().max().item())


@gpu
def test_poisoned_graph_workspace_changes_nothing(dev):
    """A captured graph replays on its private workspace: poisoning it between replays changes nothing."""
    m = _model(_ctrl("MewZoom-2X-Ctrl", 3), dev, seed=5)
    g = torch.Generator().manual_seed(6)
    x, c = torch.rand(2, 3, 29, 131, generator=g).to(dev), torch.rand(2, 3, generator=g).to(dev)
    want = m.upscale(x, c)
    graph = m.capture(x, c)
    for fill in (0xFF, 0x00, 0xFF):
        graph.ws.fill_(fill)
        assert torch.equal(graph.replay(), want), hex(fill)
    assert torch.equal(graph(x, c), want)


@gpu
@pytest.mark.parametrize("name,L,k", [("MewZoom-2X-Ctrl", 4, 2), ("MewZoom-3X-Ctrl", 3, 1)])
def test_poisoned_stage_buffers_change_nothing(dev, name, L, k):
    """sharding.upscale_tiled_refresh reusing its state: every tile's workspace filled with 0xFF before the run; the
    frame still equals the un-tiled result.  (Between the stages of one run the workspace legitimately carries state.)"""
    from ultrazoom_b200.sharding import close_refresh_state, upscale_tiled_refresh

    m = _model(_ctrl(name, L), dev, seed=L + k)
    r = m.upscale_ratio
    g = torch.Generator().manual_seed(8)
    x, c = torch.rand(1, 3, 50, 300, generator=g).to(dev), torch.rand(1, 3, generator=g).to(dev)
    full = m.upscale(x, c)
    frame = torch.full_like(full, -1.0)
    state = upscale_tiled_refresh(m, x, c, r, L, 2, 2, k, frame, align_w=128)
    try:
        assert torch.equal(frame, full)
        for fill in (0xFF, 0x00):
            for buf in state["buf"].values():
                buf.tensor.fill_(fill)
            frame.fill_(-1.0)
            upscale_tiled_refresh(m, x, c, r, L, 2, 2, k, frame, align_w=128, state=state)
            assert torch.equal(frame, full), (hex(fill), (frame - full).abs().max().item())
    finally:
        torch.cuda.synchronize()
        close_refresh_state(state)


@gpu
@pytest.mark.parametrize("name", ["MewZoom-2X-Ctrl", "MewZoom-3X-Ctrl", "MewZoom-4X-Ctrl"])
def test_guarded_frame_gets_exactly_the_image(dev, name):
    """upscale_into a frame that is exactly the output size, inside a guarded buffer, the window covering the whole
    image: the frame equals upscale and no byte around it changes -- float32 (NaN-prefilled) and uint8 (run twice,
    prefilled with 0x00 and 0xFF: identical)."""
    m = _model(_ctrl(name, 2), dev, seed=9)
    r = m.upscale_ratio
    g = torch.Generator().manual_seed(10)
    B, H, W = 2, 23, 131
    x, c = torch.rand(B, 3, H, W, generator=g).to(dev), torch.rand(B, 3, generator=g).to(dev)
    want = m.upscale(x, c)
    gx = Guarded(x.shape, torch.float32, dev, row=W, fill=x, src=True)
    sx = gx.snapshot()
    gf = Guarded((B, 3, H * r, W * r), torch.float32, dev, row=W * r).poison()
    m.upscale_into(gx.view, c, gf.view, (0, H, 0, W), (0, 0))
    torch.cuda.synchronize()
    assert torch.equal(gf.view, want), name
    assert_guards(("frame", gf))
    assert_unchanged(("x", gx, sx))
    x8 = (x * 255).to(torch.uint8)
    want8 = m.upscale(x8, c)
    got = []
    for fill in (0x00, 0xFF):
        gf8 = Guarded((B, 3, H * r, W * r), torch.uint8, dev, row=W * r)
        gf8.view.fill_(fill)
        m.upscale_into(x8, c, gf8.view, (0, H, 0, W), (0, 0))
        torch.cuda.synchronize()
        assert_guards(("frame u8", gf8))
        got.append(gf8.view.clone())
    assert torch.equal(got[0], got[1]) and torch.equal(got[0], want8), name
