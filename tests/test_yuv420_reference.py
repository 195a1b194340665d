"""CPU: the float64 reference of the 4:2:0 conversions (oracle/yuv420.py) that the GPU tests hold the kernels to.

Colour bars pin the matrices, ranges and bit depths; flat in-gamut frames survive decode then encode exactly; the filters
are checked on frames whose result is known in closed form (a chroma step, one coloured column)."""
import itertools

import numpy as np
import pytest

from oracle import yuv420 as ref

MATRICES = ("bt709", "bt601", "bt2020")
BARS = {"white": (1, 1, 1), "yellow": (1, 1, 0), "cyan": (0, 1, 1), "green": (0, 1, 0), "magenta": (1, 0, 1),
        "red": (1, 0, 0), "blue": (0, 0, 1), "black": (0, 0, 0)}


def test_published_anchors():
    """100 % red, 8-bit limited range: BT.709 (63, 102, 240), BT.601 (81, 90, 240), BT.2020 (74, 97, 240); 10-bit BT.709
    (250, 409, 960)."""
    assert ref.encode_pixel((1, 0, 0), 8, "bt709") == (63, 102, 240)
    assert ref.encode_pixel((1, 0, 0), 8, "bt601") == (81, 90, 240)
    assert ref.encode_pixel((1, 0, 0), 8, "bt2020") == (74, 97, 240)
    assert ref.encode_pixel((1, 0, 0), 10, "bt709") == (250, 409, 960)


@pytest.mark.parametrize("matrix,full,bits", list(itertools.product(MATRICES, (False, True), (8, 10))))
def test_colour_bars(matrix, full, bits):
    """Every bar of every matrix, range and depth: white and black at the ends of the luma range with neutral chroma, the
    luma of each bar the matrix's weighted sum, each primary at the top of its own chroma axis, complementary bars
    mirrored about the chroma midpoint, and a flat frame of each bar encodes to the same codes as the single pixel."""
    kr, kb = ref.MATRICES[matrix]
    kg = 1 - kr - kb
    yoff, ys, coff, cs, mx = ref.code_range(bits, full)
    u = 1 << (bits - 8)
    lo, hi = (0, mx) if full else (16 * u, 235 * u)
    mid = 128 * u
    got = {name: ref.encode_pixel(rgb, bits, matrix, full) for name, rgb in BARS.items()}
    assert got["white"] == (hi, mid, mid) and got["black"] == (lo, mid, mid)
    for name, (r, g, b) in BARS.items():
        assert got[name][0] == int(np.floor(yoff + ys * (kr * r + kg * g + kb * b) + 0.5)), name
    cmax = mx if full else 240 * u                                  # (full range: 2^bits - 1/2 is clamped)
    assert got["red"][2] == cmax and got["blue"][1] == cmax
    tie = 1 if full else 0                                          # (full range: C' = -1/2 lands on a rounding tie)
    assert abs(got["cyan"][2] - (2 * mid - cmax)) <= tie and abs(got["yellow"][1] - (2 * mid - cmax)) <= tie
    for a, b in (("red", "cyan"), ("green", "magenta"), ("blue", "yellow")):
        ya, cba, cra = got[a]
        yb, cbb, crb = got[b]
        assert abs((cba - mid) + (cbb - mid)) <= 1 and abs((cra - mid) + (crb - mid)) <= 1, (a, b)
    dtype = np.uint8 if bits == 8 else np.uint16
    for name, rgb in BARS.items():
        rgb16 = np.tile(np.round(np.array(rgb, dtype=np.float64) * 65535).astype(np.uint16).reshape(1, 3, 1, 1), (1, 1, 4, 6))
        f = ref.encode(rgb16, dtype, matrix, full)
        luma, cb, cr = ref.split_frames(f)
        assert (luma == got[name][0]).all() and (cb == got[name][1]).all() and (cr == got[name][2]).all(), name


@pytest.mark.parametrize("matrix,full,bits", list(itertools.product(MATRICES, (False, True), (8, 10))))
def test_flat_in_gamut_colours_survive_decode_then_encode(matrix, full, bits):
    """A flat frame of any (Y, Cb, Cr) whose RGB lies inside [0, 1] comes back with the same codes: the 16-bit
    intermediate is fine enough that the second quantisation lands on the first."""
    rng = np.random.default_rng(bits + 3 * len(matrix) + full)
    dtype = np.uint8 if bits == 8 else np.uint16
    yoff, ys, coff, cs, mx = ref.code_range(bits, full)
    kept = 0
    for _ in range(600):
        y, cb, cr = (int(v) for v in rng.integers(0, mx + 1, 3))
        rgb = ref.ycbcr_to_rgb(np.float64((y - yoff) / ys), np.float64((cb - coff) / cs), np.float64((cr - coff) / cs), matrix)
        if not ((rgb >= 0).all() and (rgb <= 1).all()):
            continue
        kept += 1
        luma = np.full((1, 4, 6), y)
        f = ref.join_frames(luma, np.full((1, 2, 3), cb), np.full((1, 2, 3), cr), dtype)
        back = ref.encode(ref.decode(f, matrix, full), dtype, matrix, full)
        assert np.array_equal(back, f), (y, cb, cr)
    assert kept > 50


def test_p010_low_bits_and_layout():
    """P010 words carry the code in their top 10 bits: the low 6 bits are ignored by decode and zero after encode; frames
    are (B, 3H/2, W) with the luma plane first."""
    rng = np.random.default_rng(5)
    f = ref.join_frames(rng.integers(64, 941, (2, 4, 8)), rng.integers(64, 961, (2, 2, 4)), rng.integers(64, 961, (2, 2, 4)),
                        np.uint16)
    assert f.shape == (2, 6, 8) and not (f & 63).any()
    noisy = f | rng.integers(0, 64, f.shape).astype(np.uint16)
    assert np.array_equal(ref.decode(noisy), ref.decode(f))
    out = ref.encode(ref.decode(f), np.uint16)
    assert out.dtype == np.uint16 and not (out & 63).any()


def test_chroma_filters():
    """Decode: a vertical chroma step between chroma rows 0 and 1 gives luma rows 0..3 weights 0, 1/4, 3/4, 1 of the
    step; a horizontal step gives columns 0..3 weights 0, 1/2, 1, 1.  Encode of a single blue luma column: an even column
    2j gives chroma column j 1/2 of its chroma, an odd column 2j+1 gives columns j and j+1 1/4 each, and column 0 gives
    chroma column 0 3/4 (its left tap is clamped onto it)."""
    H, W = 4, 4
    luma = np.full((1, H, W), 126)
    base = np.full((1, 2, 2), 128)
    step = base.copy()
    step[:, 1] = 128 + 80                                          # Cr of chroma row 1
    rgb = ref.decode(ref.join_frames(luma, base, step, np.uint8), quantised=False)
    r = rgb[0, 0, :, 0]
    w = (r - r[0]) / (r[-1] - r[0])
    assert np.allclose(w, [0, 0.25, 0.75, 1])
    step = base.copy()
    step[:, :, 1] = 128 + 80
    rgb = ref.decode(ref.join_frames(luma, base, step, np.uint8), quantised=False)
    r = rgb[0, 0, 0, :]
    assert np.allclose((r - r[0]) / (r[-1] - r[0]), [0, 0.5, 1, 1])
    kr, kb = ref.MATRICES["bt709"]
    full = 255 / 2                                                # Cb' of pure blue (1/2), in full-range codes

    def cb_row(col):
        img = np.zeros((1, 3, 2, 8), dtype=np.uint16)
        img[:, 2, :, col] = 65535                                 # blue in one luma column
        return list(ref.split_frames(ref.encode(img, np.uint8, full_range=True))[1][0, 0])

    q = lambda w: int(np.floor(128 + w * full + 0.5))             # noqa: E731
    assert cb_row(2) == [128, q(0.5), 128, 128]
    assert cb_row(3) == [128, q(0.25), q(0.25), 128]
    assert cb_row(0) == [q(0.75), 128, 128, 128]                  # (column -1 is column 0)
