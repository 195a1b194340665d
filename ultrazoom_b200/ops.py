"""Per-kernel Python entry points over the C ABI (torch tensors in, torch tensors out, current stream).

These are what the unit tests and micro-benchmarks call; ``MewZoom`` itself uses ``mz_upscale``.
All tensors must live on a B200; there is no fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
from torch import Tensor

from . import _native


def _stream(t: Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _need_cuda(*ts: Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("ultrazoom_b200.ops: CUDA tensors required (no CPU fallback)")


def padded_channels(c: int) -> int:
    return _native.load().mz_padded_channels(c)


def bicubic(x: Tensor, r: int) -> Tensor:
    """Upsample(scale_factor=r, mode="bicubic") -- reference model.py:71,156."""
    _need_cuda(x)
    assert x.dim() == 4, "Expected (B, C, H, W)."
    x = x.to(torch.float32).contiguous()
    B, Cc, H, W = x.shape
    y = torch.empty((B, Cc, H * r, W * r), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(_native.load().mz_bicubic_f32(x.data_ptr(), y.data_ptr(), B * Cc, H, W, r, _stream(x)))
    return y


def yuv420_to_rgb16(x: Tensor, yuv: Optional["Yuv420"] = None) -> Tensor:
    """4:2:0 frames (B, 3H/2, W) -- uint8 NV12 or uint16 P010 -- to 16-bit planar RGB (B, 3, H, W) (mz_yuv420_to_rgb16);
    ``yuv`` (default ``Yuv420()``) names the colour matrix and range."""
    from .model import Yuv420, _yuv_dims

    _need_cuda(x)
    B, H, W = _yuv_dims(x)
    flags = (yuv or Yuv420()).flags(x.dtype)
    x = x.contiguous()
    y = torch.empty((B, 3, H, W), dtype=torch.uint16, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(_native.load().mz_yuv420_to_rgb16(x.data_ptr(), y.data_ptr(), B, H, W, flags, _stream(x)))
    return y


def rgb16_to_yuv420(rgb: Tensor, dtype: torch.dtype = torch.uint8, yuv: Optional["Yuv420"] = None) -> Tensor:
    """16-bit planar RGB (B, 3, H, W) to 4:2:0 frames (B, 3H/2, W) of ``dtype``: uint8 NV12 or uint16 P010
    (mz_rgb16_to_yuv420)."""
    from .model import Yuv420

    _need_cuda(rgb)
    assert rgb.dim() == 4 and rgb.shape[1] == 3 and rgb.dtype == torch.uint16, "Expected a uint16 image (B, 3, H, W)."
    B, _, H, W = rgb.shape
    flags = (yuv or Yuv420()).flags(dtype)
    rgb = rgb.contiguous()
    y = torch.empty((B, H * 3 // 2, W), dtype=dtype, device=rgb.device)
    with torch.cuda.device(rgb.device):
        _native.check(_native.load().mz_rgb16_to_yuv420(rgb.data_ptr(), y.data_ptr(), B, H, W, flags, _stream(rgb)))
    return y


def pack_conv_weight(w: Tensor, device: torch.device, cout_p: Optional[int] = None,
                     cin_p: Optional[int] = None, dtype: torch.dtype = torch.float16) -> Tensor:
    """OIHW fp32 -> device fp16|bf16 [9][cout_p][cin_p]."""
    lib = _native.load()
    w = w.detach().to(device="cpu", dtype=torch.float32).contiguous()
    cout, cin = w.shape[0], w.shape[1]
    assert tuple(w.shape[2:]) == (3, 3), "Expected a 3x3 kernel."
    cout_p = cout_p or lib.mz_padded_channels(cout)
    cin_p = cin_p or lib.mz_padded_channels(cin)
    out = torch.empty((9, cout_p, cin_p), dtype=dtype, device=device)
    nbytes = C.c_size_t()
    with torch.cuda.device(device):
        _native.check(lib.mz_pack_conv_weight(w.data_ptr(), cout, cin, cout_p, cin_p, _native.dtype_code(dtype),
                                              out.data_ptr(), C.byref(nbytes)))
    assert nbytes.value == out.numel() * 2
    return out


def stem_pack(x: Tensor, weight: Tensor, bias: Tensor, cp: Optional[int] = None, dtype: torch.dtype = torch.float16,
              zb_pitch: int = 0):
    """FanOutProjection + NCHW->NHWC: returns (zf fp32 (B,H,W,Cp), zb fp16|bf16 (B,H,W,zb_pitch or Cp))."""
    _need_cuda(x)
    lib = _native.load()
    x = x.to(torch.float32).contiguous()
    B, _, H, W = x.shape
    Cc = weight.shape[0]
    cp = cp or lib.mz_padded_channels(Cc)
    w = torch.zeros((cp, 3), dtype=torch.float32, device=x.device)
    b = torch.zeros((cp,), dtype=torch.float32, device=x.device)
    w[:Cc] = weight.detach().reshape(Cc, 3).to(x.device, torch.float32)
    b[:Cc] = bias.detach().to(x.device, torch.float32)
    zf = torch.empty((B, H, W, cp), dtype=torch.float32, device=x.device)
    zb = torch.empty((B, H, W, zb_pitch or cp), dtype=dtype, device=x.device)
    with torch.cuda.device(x.device):
        _native.check(lib.mz_stem_pack(x.data_ptr(), w.data_ptr(), b.data_ptr(), zf.data_ptr(), zb.data_ptr(),
                                       B, H, W, cp, zb_pitch, _native.dtype_code(dtype), _stream(x)))
    return zf, zb


def control_film(c: Tensor, weight: Tensor, bias: Tensor, B: int, hcp: Optional[int] = None) -> Tensor:
    """FiLM table (L,B,2,hCp) from c (1|B, F), weight (L, 2hC, F), bias (L, 2hC)."""
    _need_cuda(c, weight, bias)
    lib = _native.load()
    L, two_hc, F = weight.shape
    hC = two_hc // 2
    hcp = hcp or lib.mz_padded_channels(hC)
    c = c.to(torch.float32).contiguous()
    film = torch.empty((L, B, 2, hcp), dtype=torch.float32, device=c.device)
    with torch.cuda.device(c.device):
        _native.check(lib.mz_control_film(c.data_ptr(), c.shape[0], weight.contiguous().data_ptr(),
                                          bias.contiguous().data_ptr(), film.data_ptr(), L, B, F, hC, hcp,
                                          _stream(c)))
    return film


def conv3x3(inp: Tensor, wpacked: Tensor, mode: int, film: Optional[Tensor] = None, zf: Optional[Tensor] = None,
            use_tc: bool = True, tune: Optional[_native.MzConvTune] = None, out_pitch: int = 0,
            out: Optional[Tensor] = None, channel_offset: int = 0) -> Tensor:
    """3x3 conv on NHWC fp16|bf16 with the fused block epilogues; returns the 16-bit NHWC output (dtype of `inp`).

    mode 0: SiLU(scale*acc+shift) with film (B,2,cout_p) or None; mode 1: zf += acc (in place), returns round16(zf).
    The input may be wider than the weights' cin_p (its first cin_p channels are used).  ``out`` (B,H,W,P) 16-bit and
    ``channel_offset``: this launch owns output channels [channel_offset, channel_offset + cout_p) of a wider ``out`` (and,
    in mode 1, of a wider ``zf``) -- how a convolution wider than one launch is sliced."""
    _need_cuda(inp, wpacked)
    assert inp.dtype in (torch.float16, torch.bfloat16) and wpacked.dtype == inp.dtype
    inp = inp.contiguous()
    B, H, W, in_pitch = inp.shape
    _, cout_p, cin_p = wpacked.shape
    assert in_pitch >= cin_p, "weight / activation channel mismatch"
    assert mode in (0, 1), "mode must be 0 (conv1 + FiLM + SiLU) or 1 (conv2 + residual)"
    zf_pitch = 0
    if out is None:
        assert channel_offset == 0
        alloc = torch.zeros if out_pitch > cout_p else torch.empty   # pad channels are never written by the kernel
        out = alloc((B, H, W, out_pitch or cout_p), dtype=inp.dtype, device=inp.device)
        if mode == 1:
            assert zf is not None and zf.is_contiguous() and tuple(zf.shape) == (B, H, W, cout_p)
    else:
        assert out.is_contiguous() and out.dtype == inp.dtype and tuple(out.shape[:3]) == (B, H, W)
        out_pitch = out.shape[3]
        assert 0 <= channel_offset and channel_offset + cout_p <= out_pitch and channel_offset % 8 == 0
        if mode == 1:
            assert zf is not None and zf.is_contiguous() and tuple(zf.shape[:3]) == (B, H, W)
            zf_pitch = zf.shape[3]
            assert channel_offset + cout_p <= zf_pitch
    with torch.cuda.device(inp.device):
        _native.check(_native.load().mz_conv3x3(
            inp.data_ptr(), wpacked.data_ptr(), mode, film.data_ptr() if film is not None else None,
            out.data_ptr() + 2 * channel_offset, zf.data_ptr() + 4 * channel_offset if zf is not None else None, B, H, W, cin_p,
            in_pitch if in_pitch != cin_p else 0, cout_p, out_pitch if out_pitch != cout_p else 0,
            zf_pitch if zf_pitch != cout_p else 0, _native.dtype_code(inp.dtype), 1 if use_tc else 0,
            C.byref(tune) if tune is not None else None, _stream(inp)))
    return out


def block_fused(zb: Tensor, w1_packed: Tensor, w2_packed: Tensor, film: Optional[Tensor], zf: Tensor, seg_rows: int = 0,
                max_ctas: int = 0) -> Tensor:
    """One encoder block as one kernel (mz_block_fused): zf += conv2(SiLU(scale * conv1(zb) + shift)) in place, returns
    the new 16-bit stream round16(zf).  zb (B,H,W,48) 16-bit, w1_packed (9,96,48), w2_packed (9,48,96), film (B,2,96)."""
    _need_cuda(zb, w1_packed, w2_packed, zf)
    assert zb.dtype in (torch.float16, torch.bfloat16) and w1_packed.dtype == zb.dtype and w2_packed.dtype == zb.dtype
    zb = zb.contiguous()
    B, H, W, Cc = zb.shape
    assert Cc == 48 and tuple(w1_packed.shape) == (9, 96, 48) and tuple(w2_packed.shape) == (9, 48, 96), "48 / 96 channels only"
    assert zf.is_contiguous() and tuple(zf.shape) == (B, H, W, 48) and zf.dtype == torch.float32
    out = torch.empty_like(zb)
    with torch.cuda.device(zb.device):
        _native.check(_native.load().mz_block_fused(
            zb.data_ptr(), out.data_ptr(), zf.data_ptr(), w1_packed.data_ptr(), w2_packed.data_ptr(),
            film.data_ptr() if film is not None else None, B, H, W, _native.dtype_code(zb.dtype), seg_rows, max_ctas,
            _stream(zb)))
    return out


def head_shuffle_add(zb: Tensor, wpacked: Tensor, r: int, x: Optional[Tensor] = None, y: Optional[Tensor] = None,
                     skip_mode: int = 2, clamp01: bool = False, use_tc: bool = True,
                     tune: Optional[_native.MzConvTune] = None) -> Tensor:
    """SubpixelConv2d + skip add (+ clamp): returns y (B,3,rH,rW) fp32 NCHW."""
    _need_cuda(zb, wpacked)
    assert zb.dtype in (torch.float16, torch.bfloat16) and wpacked.dtype == zb.dtype
    zb = zb.contiguous()
    B, H, W, in_pitch = zb.shape
    cin_p = wpacked.shape[2]
    assert in_pitch >= cin_p, "weight / activation channel mismatch"
    if y is None:
        assert skip_mode != 1, "skip_mode 1 needs y preloaded with the bicubic image"
        y = torch.empty((B, 3, H * r, W * r), dtype=torch.float32, device=zb.device)
    if x is not None:
        x = x.to(torch.float32).contiguous()
    with torch.cuda.device(zb.device):
        _native.check(_native.load().mz_head_shuffle_add(
            zb.data_ptr(), wpacked.data_ptr(), x.data_ptr() if x is not None else None, y.data_ptr(), B, H, W, cin_p,
            in_pitch if in_pitch != cin_p else 0, r, skip_mode, 1 if clamp01 else 0, _native.dtype_code(zb.dtype), 1 if use_tc else 0, C.byref(tune) if tune is not None else None,
            _stream(zb)))
    return y


def probe_umma(kc: int, row_shift: int, base_offset_mode: int) -> float:
    err = C.c_float()
    _native.check(_native.load().mz_probe_umma(kc, row_shift, base_offset_mode, C.byref(err)))
    return err.value


def probe_mma_rate(n: int, kc: int, iters: int = 2000, ctas: int = 1, distinct_a: int = 1,
                   distinct_d: int = 1, a_row_shift: int = 0) -> float:
    cyc = C.c_float()
    _native.check(_native.load().mz_probe_mma_rate(n, kc, iters, ctas, distinct_a, distinct_d, a_row_shift,
                                                   C.byref(cyc)))
    return cyc.value
