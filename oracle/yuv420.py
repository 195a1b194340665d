"""float64 reference of the 4:2:0 frame conversions (NV12 / P010 <-> 16-bit planar RGB) that ``MZ_FLAG_YUV420`` wraps
around a 16-bit upscale.  TEST INFRASTRUCTURE ONLY.

A batch of frames is ``(B, 3H/2, W)``: per frame the H x W luma plane, then H/2 rows of W/2 interleaved Cb,Cr pairs.
NV12 is uint8 (8-bit codes); P010 is uint16 with the 10-bit code in the top bits (``word = code << 6``).  Chroma sample
(i, j) sits at luma row 2i + 1/2, column 2j (the H.264 / HEVC default).  See ``mz_yuv420_to_rgb16`` in
include/mewzoom_b200.h for the contract this restates.
"""
from __future__ import annotations

import numpy as np

MATRICES = {"bt709": (0.2126, 0.0722), "bt601": (0.299, 0.114), "bt2020": (0.2627, 0.0593)}


def code_range(bits: int, full_range: bool):
    """``(yoff, yscale, coff, cscale, maxcode)``: Y = yoff + yscale Y', C = coff + cscale C'."""
    maxcode = (1 << bits) - 1
    coff = 1 << (bits - 1)
    if full_range:
        return 0.0, float(maxcode), float(coff), float(maxcode), maxcode
    u = 1 << (bits - 8)
    return 16.0 * u, 219.0 * u, float(coff), 224.0 * u, maxcode


def _bits(dtype) -> int:
    return 8 if np.dtype(dtype) == np.uint8 else 10


def rgb_to_ycbcr(rgb: np.ndarray, matrix: str):
    """(..., 3) RGB in [0, 1] -> (Y', Cb', Cr') as float64 arrays (Cb', Cr' in [-1/2, 1/2])."""
    kr, kb = MATRICES[matrix]
    kg = 1.0 - kr - kb
    rgb = np.asarray(rgb, dtype=np.float64)
    r, g, b = rgb[..., 0], rgb[..., 1], rgb[..., 2]
    y = kr * r + kg * g + kb * b
    return y, (b - y) / (2.0 * (1.0 - kb)), (r - y) / (2.0 * (1.0 - kr))


def ycbcr_to_rgb(y, cb, cr, matrix: str) -> np.ndarray:
    """(Y', Cb', Cr') -> (..., 3) RGB, not clamped."""
    kr, kb = MATRICES[matrix]
    kg = 1.0 - kr - kb
    r = y + 2.0 * (1.0 - kr) * cr
    b = y + 2.0 * (1.0 - kb) * cb
    g = (y - kr * r - kb * b) / kg
    return np.stack([r, g, b], axis=-1)


def quantise(v, off: float, scale: float, maxcode: int) -> np.ndarray:
    """floor(off + scale v + 0.5), clamped to [0, maxcode]."""
    return np.clip(np.floor(off + scale * np.asarray(v, dtype=np.float64) + 0.5), 0, maxcode).astype(np.int64)


def encode_pixel(rgb, bits: int = 8, matrix: str = "bt709", full_range: bool = False):
    """One RGB colour -> its (Y, Cb, Cr) codes: what a flat frame of that colour encodes to."""
    yoff, ys, coff, cs, mx = code_range(bits, full_range)
    y, cb, cr = rgb_to_ycbcr(np.asarray(rgb, dtype=np.float64), matrix)
    return int(quantise(y, yoff, ys, mx)), int(quantise(cb, coff, cs, mx)), int(quantise(cr, coff, cs, mx))


def split_frames(frames: np.ndarray):
    """(B, 3H/2, W) -> integer codes: luma (B, H, W), cb and cr (B, H/2, W/2)."""
    frames = np.asarray(frames)
    B, rows, W = frames.shape
    H = rows // 3 * 2
    codes = frames.astype(np.int64)
    if frames.dtype == np.uint16:
        codes = codes >> 6
    luma = codes[:, :H]
    chroma = codes[:, H:].reshape(B, H // 2, W // 2, 2)
    return luma, chroma[..., 0], chroma[..., 1]


def join_frames(luma: np.ndarray, cb: np.ndarray, cr: np.ndarray, dtype) -> np.ndarray:
    """Inverse of ``split_frames`` (codes -> NV12 / P010 elements)."""
    B, H, W = luma.shape
    chroma = np.stack([cb, cr], axis=-1).reshape(B, H // 2, W)
    codes = np.concatenate([luma, chroma], axis=1)
    if np.dtype(dtype) == np.uint16:
        codes = codes << 6
    return codes.astype(dtype)


def decode(frames: np.ndarray, matrix: str = "bt709", full_range: bool = False, quantised: bool = True) -> np.ndarray:
    """NV12 / P010 frames -> (B, 3, H, W): uint16 codes floor(65535 clamp(v) + 0.5), or (``quantised=False``) the float64
    RGB before clamping."""
    bits = _bits(np.asarray(frames).dtype)
    yoff, ys, coff, cs, _ = code_range(bits, full_range)
    luma, cb, cr = split_frames(frames)

    def up(c):
        c = c.astype(np.float64)
        above = np.concatenate([c[:, :1], c[:, :-1]], axis=1)        # C[i-1], clamped
        below = np.concatenate([c[:, 1:], c[:, -1:]], axis=1)        # C[i+1], clamped
        v = np.empty((c.shape[0], 2 * c.shape[1], c.shape[2]))
        v[:, 0::2] = 0.75 * c + 0.25 * above
        v[:, 1::2] = 0.75 * c + 0.25 * below
        right = np.concatenate([v[:, :, 1:], v[:, :, -1:]], axis=2)  # C[j+1], clamped
        h = np.empty((v.shape[0], v.shape[1], 2 * v.shape[2]))
        h[:, :, 0::2] = v
        h[:, :, 1::2] = 0.5 * (v + right)
        return h

    y = (luma - yoff) / ys
    rgb = ycbcr_to_rgb(y, (up(cb) - coff) / cs, (up(cr) - coff) / cs, matrix)
    rgb = np.moveaxis(rgb, -1, 1)
    if not quantised:
        return rgb
    return np.floor(65535.0 * np.clip(rgb, 0.0, 1.0) + 0.5).astype(np.uint16)


def encode(rgb16: np.ndarray, dtype=np.uint8, matrix: str = "bt709", full_range: bool = False) -> np.ndarray:
    """(B, 3, H, W) uint16 RGB -> NV12 (``dtype`` uint8) or P010 (uint16) frames (B, 3H/2, W)."""
    bits = _bits(dtype)
    yoff, ys, coff, cs, mx = code_range(bits, full_range)
    v = np.moveaxis(np.asarray(rgb16).astype(np.float64) / 65535.0, 1, -1)
    y, cb, cr = rgb_to_ycbcr(v, matrix)

    def down(c):
        m = 0.5 * (c[:, 0::2] + c[:, 1::2])                          # rows 2i, 2i+1
        left = np.concatenate([m[:, :, :1], m[:, :, 1:-1:2]], axis=2)  # column 2j-1, column -1 clamped to 0
        return 0.25 * left + 0.5 * m[:, :, 0::2] + 0.25 * m[:, :, 1::2]

    return join_frames(quantise(y, yoff, ys, mx), quantise(down(cb), coff, cs, mx), quantise(down(cr), coff, cs, mx),
                       dtype)
