"""Every pixel of the benchmark's frames, block by block, against a reference that rounds where the kernels round.

The reference (``Emulation``) is the MewZoom network in ``torch.nn.functional``, fp32 with TF32 off, fed the model's
own parameters, rounding to the 16-bit operand type at exactly the points the kernels do and nowhere else:
    stem   zf = conv1x1(x) + b (fp32), zb = round16(zf)
    block  hid = round16(SiLU(conv3x3(zb, round16(w1)) * (1 + gamma_l) + beta_l)),  gamma_l | beta_l = control_l(c)
           zf += conv3x3(hid, round16(w2)),  zb = round16(zf)
    head   clamp(pixel_shuffle(conv3x3(zb, round16(wh)), r) + bicubic(x), 0, 1), bicubic with the exact phase table
The real model is stepped one encoder block at a time (``upscale_stage``), and every block is compared with the
reference started from the kernel's own fp32 stream of the block before, so each block's bound is single-block noise:
fp32 summation order, and ``tanh.approx`` in the SiLU flipping the 16-bit rounding of some hidden elements.  For every
block, over every pixel of every image: max|zf - ref|, its 99.99th percentile, and the largest per-channel mean of
zf - ref (a bias: what rounding toward zero instead of to nearest leaves behind, and the flips do not); the 16-bit
stream equals round16(zf) bit for bit and the padded channels are zero.  The output frame is compared with the
reference's head applied to the kernel's final 16-bit stream, and the whole call (``upscale``) equals the staged one
bit for bit, so what is checked is what the benchmark times.

Measured on one NVIDIA B200 (1000 W power limit), worst over the blocks of a case (the max grows with depth: 4e-5 -
2.3e-4 from the first to the last blocks with fp16 operands), the oracle's random-init weights:
                                               max       p99.99    |channel mean|
    cfg2   2X-Ctrl 16 x 540x960       bf16     1.21e-3   5.18e-4   8.2e-7
                                      fp16     2.38e-4   9.1e-5    9.7e-7
    cfg3   3X-Ctrl 720x1280           fp16     2.16e-4   1.09e-4   2.3e-6
    cfg4a  4X-Ctrl 540x960            fp16     2.31e-4   1.30e-4   5.8e-6
    cfg4b  4X-Ctrl 1080x1920          fp16     2.31e-4   1.12e-4   4.5e-6
                                      bf16     1.10e-3   6.79e-4   4.0e-6
    cfg4c  2X-Ctrl 1080x1920          fp16     1.50e-4   6.4e-5    8.0e-7
    2X-Ctrl 22 x 540x960 (> 2^31 B)   bf16     1.04e-3   5.26e-4   9.6e-7
    3X-Ctrl 11 x 720x1280, 56 ch      fp16     3.23e-4   1.49e-4   2.7e-6
    3X-Ctrl 10 x 720x1280, 64 ch      fp16     2.64e-4   1.43e-4   3.0e-6
    controls' runs: 4X-Ctrl 540x960 fp16 2.36e-4 / 1.30e-4 / 6.0e-6, bf16 1.47e-3 / 7.22e-4 / 5.5e-6;
                    2X-Ctrl 2 x 540x960 fp16 1.65e-4 / 8.2e-5 / 8.4e-7, bf16 1.04e-3 / 5.03e-4 / 6.9e-7
    stem 2.4e-7 everywhere; output frame max 7.7e-6, p99.99 3.9e-6 (cfg4a)
Bounds (BLOCK_BOUNDS, STEM_BOUND, HEAD_BOUNDS) are 1.8 - 2.0x the worst of these per model and operand type.
What each control is rejected by, at its weakest block: (a) by the channel mean, 9.8x the bound on 4X-Ctrl fp16 (its max
is only 1.7x the real one there: the 16-bit flips of tanh.approx are nearly as large as a truncation, but they average
out and a truncation does not) and 57 - 450x elsewhere; (b), (c), (d) by the max, 100 - 200000x; (e) by the max, 5.4x
the head bound.  So the bounds weakened 10x let (a) pass at one block of 4X-Ctrl fp16, and (e).

Past 2^31 bytes: batches whose fp32 stream alone exceeds 2^31 bytes (2X-Ctrl 22 x 540x960 at 48 channels; 3X-Ctrl
720x1280 at 56 channels, 11 images, and at 64 with MZ_DENSE_LAYOUT=0, 10 images).  The last two images are compared at
every block, every image's frame with the reference head, and every image -- float and 8-bit -- with the same image
run alone (batch independence is bit-exact, so any difference is an addressing fault).  Their images are 8-bit
values, so that the float call is the 8-bit call's own reference.

Negative controls: deliberately wrong references, each rejected by the bounds at every block where it applies:
(a) hidden tensor rounded toward zero, (b) layer l with the FiLM rows of layer l+1, (c) conv1 reading the 16-bit
stream of one block earlier, (d) conv1's 3x3 filter transposed, (e) the bicubic skip at r = 3 from F.interpolate.

MZ_EMULATED_REPORT=<path> writes the measured values of a run to that JSON file.
"""
import json
import math
import os

import pytest
import torch
from torch.nn import functional as F

from oracle import bicubic_upsample_ref, make_oracle, max_abs_err

DT = {"float16": torch.float16, "bfloat16": torch.bfloat16}

# per-block bounds (max, p99.99, |per-channel mean|) per model and operand type; stem and head bounds for all
BLOCK_BOUNDS = {
    ("MewZoom-2X-Ctrl", "float16"): (4.5e-4, 1.8e-4, 1.9e-6),
    ("MewZoom-2X-Ctrl", "bfloat16"): (2.4e-3, 1.05e-3, 1.9e-6),
    ("MewZoom-3X-Ctrl", "float16"): (6.4e-4, 2.9e-4, 5.8e-6),
    ("MewZoom-4X-Ctrl", "float16"): (4.7e-4, 2.6e-4, 1.2e-5),
    ("MewZoom-4X-Ctrl", "bfloat16"): (2.9e-3, 1.4e-3, 1.0e-5),
}
STEM_BOUND = 4.7e-7
HEAD_BOUNDS = (1.5e-5, 7.8e-6)    # (max, p99.99) on the clamped output frame
MIN_RESIDUAL_STD = 0.2            # degeneracy guard: the residual branch (head convolution) is alive (measured >= 0.46)


# --------------------------------------------------------------------------------------------------------------------
# the emulating reference
# --------------------------------------------------------------------------------------------------------------------

def round16(v: torch.Tensor, dt: torch.dtype, mode: str = "nearest") -> torch.Tensor:
    """fp32 ``v`` rounded to ``dt``: to nearest even, as the kernels' conversions do, or toward zero (a wrong variant)."""
    out = v.to(dt)
    if mode == "nearest" or dt == torch.float32:
        return out
    assert mode == "toward_zero", mode
    bits = out.view(torch.int16)               # sign-magnitude: one less is one step toward zero
    return torch.where(out.float().abs() > v.abs(), bits - 1, bits).view(dt)


def _assert_fp32_exact(t: torch.Tensor) -> None:
    assert t.dtype == torch.float32
    assert not torch.backends.cudnn.allow_tf32 and not torch.backends.cuda.matmul.allow_tf32, "TF32 must be off"


class Emulation:
    """The network of ``model`` (a MewZoom or an OracleMewZoom: the same parameter names), evaluated with
    ``torch.nn.functional`` on ``device`` and rounded to ``dt`` where the kernels round (``dt = torch.float32`` rounds
    nowhere: the fp32 network).  The keyword arguments make it wrong on purpose, for the negative controls."""

    def __init__(self, model, dt: torch.dtype, device, hidden_rounding: str = "nearest", film_of_next_layer: bool = False,
                 conv1_transposed: bool = False, skip: str = "table"):
        def fp32(t):
            return t.detach().to(device=device, dtype=torch.float32)

        def operand(t):
            return fp32(t).to(dt).float()

        self.dt, self.r, self.C, self.L = dt, model.upscale_ratio, model.num_channels, model.num_encoder_layers
        self.hidden_rounding, self.film_of_next_layer, self.skip = hidden_rounding, film_of_next_layer, skip
        self.stem_w, self.stem_b = fp32(model.stem.conv.weight), fp32(model.stem.conv.bias)
        self.w1 = [operand(b.convnet.conv1.weight) for b in model.encoder]
        if conv1_transposed:
            self.w1 = [w.transpose(-1, -2) for w in self.w1]
        self.w2 = [operand(b.convnet.conv2.weight) for b in model.encoder]
        self.wh = operand(model.head.conv.weight)
        self.control = ([(fp32(b.control.linear.weight), fp32(b.control.linear.bias)) for b in model.encoder]
                        if model.control_features else None)

    def stem(self, x: torch.Tensor) -> torch.Tensor:
        _assert_fp32_exact(x)
        return F.conv2d(x, self.stem_w, self.stem_b)

    def block(self, l: int, zf: torch.Tensor, zb: torch.Tensor, c) -> torch.Tensor:
        """The fp32 stream after encoder block ``l``, from the stream ``zf`` (B,C,H,W) and the 16-bit operand ``zb``."""
        _assert_fp32_exact(zf)
        acc = F.conv2d(zb.float(), self.w1[l], padding=1)
        if self.control is not None:
            w, b = self.control[min(l + 1, self.L - 1) if self.film_of_next_layer else l]
            g = F.linear(c, w, b)
            hc = acc.shape[1]
            acc = acc * (1.0 + g[:, :hc])[:, :, None, None] + g[:, hc:][:, :, None, None]
        hid = round16(F.silu(acc), self.dt, self.hidden_rounding).float()
        return zf + F.conv2d(hid, self.w2[l], padding=1)

    def head(self, zb: torch.Tensor, x: torch.Tensor, clamp: bool = True):
        """``(output frame, residual)`` from the final 16-bit stream ``zb`` (B,C,H,W) and the image ``x``."""
        _assert_fp32_exact(x)
        u = F.pixel_shuffle(F.conv2d(zb.float(), self.wh, padding=1), self.r)
        if self.skip == "interpolate":
            s = F.interpolate(x, scale_factor=self.r, mode="bicubic")
        else:
            s = bicubic_upsample_ref(x, self.r)
        y = u + s
        return (y.clamp(0, 1) if clamp else y), u

    def forward(self, x: torch.Tensor, c=None) -> torch.Tensor:
        """The whole un-clamped pass, rounding where the kernels round."""
        if c is not None:
            c = c.reshape(-1, c.shape[-1]).expand(x.shape[0], -1).float()
        zf = self.stem(x)
        for l in range(self.L):
            zf = self.block(l, zf, round16(zf, self.dt), c)
        return self.head(round16(zf, self.dt), x, clamp=False)[0]


@pytest.fixture
def fp32_exact():
    """The reference's convolutions and control linears in true fp32 (no TF32); the old settings come back after."""
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


# --------------------------------------------------------------------------------------------------------------------
# the reference is the oracle's network (CPU, default suite)
# --------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name,tol16", [("MewZoom-2X-Ctrl", 4e-3), ("MewZoom-3X-Ctrl", 6e-3)])
def test_emulation_is_the_oracle_network(fp32_exact, name, tol16):
    """Rounding nowhere, the reference is ``OracleMewZoom.forward`` within fp32 noise (and the bicubic table's 1e-5
    at r = 3); rounding to fp16 it is within the stated fp16 tolerance of it; rounding toward zero rounds toward zero."""
    o = make_oracle(name, seed=0)
    g = torch.Generator().manual_seed(77)
    x, c = torch.rand(2, 3, 20, 28, generator=g), torch.rand(2, 3, generator=g)
    with torch.inference_mode():
        ref = o.forward(x, c)
        exact = Emulation(o, torch.float32, "cpu").forward(x, c)
        e16 = Emulation(o, torch.float16, "cpu").forward(x, c)
    assert max_abs_err(exact, ref) <= 1e-4, max_abs_err(exact, ref)
    assert 0.0 < max_abs_err(e16, ref) <= tol16, max_abs_err(e16, ref)
    v = torch.randn(100000, generator=g) * 10.0
    for dt in (torch.float16, torch.bfloat16):
        t = round16(v, dt, "toward_zero")
        up = (t.view(torch.int16) + 1).view(dt)                          # the next value away from zero
        assert torch.all(t.float().abs() <= v.abs()) and torch.all(up.float().abs() > v.abs())
        assert torch.all(t.float() * v >= 0) and not torch.equal(t, round16(v, dt))
    masked = (v.view(torch.int32) & ~0xFFFF).view(torch.float32)            # bf16 toward zero = the high half-word
    assert torch.equal(round16(v, torch.bfloat16, "toward_zero"), masked.to(torch.bfloat16))


# --------------------------------------------------------------------------------------------------------------------
# stepping the model one block at a time
# --------------------------------------------------------------------------------------------------------------------

WORKLOADS = {  # bench.py's workloads at their benchmark sizes: (model, batch, H, W)
    "cfg2": ("MewZoom-2X-Ctrl", 16, 540, 960),
    "cfg3": ("MewZoom-3X-Ctrl", 1, 720, 1280),
    "cfg4a": ("MewZoom-4X-Ctrl", 1, 540, 960),
    "cfg4b": ("MewZoom-4X-Ctrl", 1, 1080, 1920),
    "cfg4c": ("MewZoom-2X-Ctrl", 1, 1080, 1920),
}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def _model(name: str, operands: str, dev):
    from ultrazoom_b200 import MODEL_CONFIGS, MewZoom

    o = make_oracle(name, seed=0)
    m = MewZoom(**MODEL_CONFIGS[name], operand_dtype=operands)
    m.load_state_dict(o.state_dict())
    return m.to(dev).eval()


def _images(B: int, H: int, W: int, seed: int, dev):
    g = torch.Generator().manual_seed(seed)
    x, c = torch.rand(B, 3, H, W, generator=g), torch.rand(B, 3, generator=g)
    return x.to(dev), c.to(dev)


def _nchw(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 3, 1, 2)


def _stats(d: torch.Tensor, labels: str, first_image: int) -> dict:
    """max |d|, its 99.99th percentile, the largest per-channel mean of d, and where the max is (``labels`` names d's
    dimensions; the first is the image, counted from ``first_image``)."""
    err = d.abs().reshape(-1)
    i = int(torch.argmax(err))
    k = max(1, math.ceil(err.numel() * 1e-4))
    ch = labels.index("c")
    dims = [j for j in range(d.dim()) if j != ch]
    at = [int(v) for v in torch.unravel_index(torch.tensor(i), d.shape)]
    at[0] += first_image
    return {"max": float(err[i]), "p9999": float(torch.topk(err, k, sorted=False).values.min()),
            "bias": float(d.mean(dim=dims).abs().max()), "at": dict(zip(labels, at))}


def _check_shadow(zf: torch.Tensor, z16: torch.Tensor, C: int, dt: torch.dtype, where: str) -> None:
    """The 16-bit stream is round16 of the fp32 stream bit for bit over the real channels; padded channels are zero."""
    want = zf[..., :C].to(dt).view(torch.int16)
    got = z16[..., :C].view(torch.int16)
    if not torch.equal(got, want):
        b, y, x, ch = (int(v) for v in torch.nonzero(got != want)[0])
        raise AssertionError(f"{where}: 16-bit stream != round16(fp32 stream) first at image {b}, (y, x, channel) = "
                             f"({y}, {x}, {ch}): {z16[b, y, x, ch].item()} vs {zf[b, y, x, ch].item()}")
    assert not torch.any(zf[..., C:] != 0) and not torch.any(z16[..., C:] != 0), f"{where}: padded channels are not zero"


def step_through(m, x, c, emu: Emulation, images: slice, variants=None, stale_zb: bool = False):
    """Run ``m`` one encoder block at a time (``upscale_stage``) and compare each block's fp32 stream on ``images`` with
    ``emu`` (and with each wrong reference of ``variants``) started from the kernel's own stream of the block before.

    Returns the output frame and the statistics of the stem, of every block (and of every variant at every block where
    it applies: ``variants[name]`` is an Emulation, ``stale_zb`` adds (c)), of the frame, and the degeneracy guard's
    residual std."""
    B, _, H, W = x.shape
    shape, r, C, L, dt = tuple(x.shape), m.upscale_ratio, m.num_channels, m.num_encoder_layers, emu.dt
    variants = dict(variants or {})
    ws = m.stage_workspace(shape, x.device)
    frame = torch.full((B, 3, H * r, W * r), float("nan"), device=x.device)

    def stage(l0, l1):
        m.upscale_stage(x, c, frame, (0, H, 0, W), (0, 0), l0, l1, ws)

    ci = c[images]
    stage(0, 0)                                            # the FiLM table and the stem
    zf, z16 = m.stage_views(ws, shape, 0)
    _check_shadow(zf, z16, C, dt, "stem")
    out = {"stream_bytes": zf.numel() * 4, "channels_in_memory": zf.shape[-1],
           "stem": _stats(zf[images, ..., :C] - emu.stem(x[images]).permute(0, 2, 3, 1), "byxc", images.start),
           "blocks": [], "variants": {n: {} for n in list(variants) + (["stale_zb"] if stale_zb else [])}}
    prev, older = zf[images, ..., :C].clone(), None
    for l in range(L):
        stage(l, l + 1)
        zf, z16 = m.stage_views(ws, shape, l + 1)
        _check_shadow(zf, z16, C, dt, f"block {l}")
        got = zf[images, ..., :C]
        ref = emu.block(l, _nchw(prev), _nchw(prev.to(dt)), ci).permute(0, 2, 3, 1)
        out["blocks"].append(_stats(got - ref, "byxc", images.start))
        for name, v in variants.items():
            if name == "film_of_next_layer" and l == L - 1:
                continue
            vref = v.block(l, _nchw(prev), _nchw(prev.to(dt)), ci).permute(0, 2, 3, 1)
            out["variants"][name][l] = _stats(got - vref, "byxc", images.start)
        if stale_zb and older is not None:
            vref = emu.block(l, _nchw(prev), _nchw(older.to(dt)), ci).permute(0, 2, 3, 1)
            out["variants"]["stale_zb"][l] = _stats(got - vref, "byxc", images.start)
        older, prev = prev, got.clone()
    torch.cuda.synchronize()
    y_ref, u = emu.head(_nchw(z16[..., :C]), x)
    out["head"] = _stats(frame - y_ref, "bcyx", 0)
    out["residual_std"] = float(u.std())
    return frame, out


def _report(key: str, value) -> None:
    path = os.environ.get("MZ_EMULATED_REPORT")
    if not path:
        return
    try:
        with open(path) as f:
            acc = json.load(f)
    except (OSError, ValueError):
        acc = {}
    acc[key] = value
    with open(path, "w") as f:
        json.dump(acc, f, indent=1)


def _where(st: dict) -> str:
    return ", ".join(f"{k} {v}" for k, v in st["at"].items())


def _check_blocks(out: dict, name: str, operands: str, label: str) -> None:
    bmax, bp, bbias = BLOCK_BOUNDS[(name, operands)]
    s = out["stem"]
    assert s["max"] <= STEM_BOUND, f"{label}: stem: max|zf - ref| {s['max']:.3g} > {STEM_BOUND:.3g} at {_where(s)}"
    for l, st in enumerate(out["blocks"]):
        assert st["max"] <= bmax and st["p9999"] <= bp and st["bias"] <= bbias, (
            f"{label}: block {l}: max|zf - ref| {st['max']:.3g} (bound {bmax:.3g}) at {_where(st)}, p99.99 "
            f"{st['p9999']:.3g} (bound {bp:.3g}), |channel mean| {st['bias']:.3g} (bound {bbias:.3g})")
    h = out["head"]
    assert h["max"] <= HEAD_BOUNDS[0] and h["p9999"] <= HEAD_BOUNDS[1], (
        f"{label}: output frame: max|y - ref| {h['max']:.3g} at {_where(h)}, p99.99 {h['p9999']:.3g}; bounds {HEAD_BOUNDS}")
    assert out["residual_std"] > MIN_RESIDUAL_STD, f"{label}: degenerate: residual std {out['residual_std']:.3g}"


def _rejected(st: dict, name: str, operands: str) -> bool:
    bmax, bp, bbias = BLOCK_BOUNDS[(name, operands)]
    return st["max"] > bmax or st["p9999"] > bp or st["bias"] > bbias


# --------------------------------------------------------------------------------------------------------------------
# the benchmark's workloads, every pixel of every image at every block
# --------------------------------------------------------------------------------------------------------------------

CASES = [("cfg2", "bfloat16"), ("cfg2", "float16"), ("cfg3", "float16"), ("cfg4a", "float16"), ("cfg4b", "float16"),
         ("cfg4b", "bfloat16"), ("cfg4c", "float16")]


@pytest.mark.gpu
@pytest.mark.parametrize("workload,operands", CASES)
def test_every_block_of_the_benchmark_frames(fp32_exact, dev, workload, operands):
    name, B, H, W = WORKLOADS[workload]
    m = _model(name, operands, dev)
    x, c = _images(B, H, W, 4321, dev)
    frame, out = step_through(m, x, c, Emulation(m, DT[operands], dev), slice(0, B))
    _report(f"{workload}/{operands}", out)
    _check_blocks(out, name, operands, f"{workload}/{operands}")
    assert torch.equal(m.upscale(x, c), frame), "the whole call differs from the staged one"
    if operands == "float16":
        assert not m.saturated()


# --------------------------------------------------------------------------------------------------------------------
# past 2^31 bytes of fp32 stream
# --------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name,H,W,operands,dense,channels", [
    ("MewZoom-2X-Ctrl", 540, 960, "bfloat16", None, 48),
    ("MewZoom-3X-Ctrl", 720, 1280, "float16", None, 56),
    ("MewZoom-3X-Ctrl", 720, 1280, "float16", "0", 64),
])
def test_batches_past_2_31_bytes(fp32_exact, dev, monkeypatch, name, H, W, operands, dense, channels):
    if dense is None:
        monkeypatch.delenv("MZ_DENSE_LAYOUT", raising=False)
    else:
        monkeypatch.setenv("MZ_DENSE_LAYOUT", dense)
    m = _model(name, operands, dev)
    ws1 = m.stage_workspace((1, 3, H, W), dev)
    Cp = m.stage_views(ws1, (1, 3, H, W), 0)[0].shape[-1]
    del ws1
    assert Cp == channels, (name, dense, Cp)
    per_image = H * W * Cp * 4
    B = 2 ** 31 // per_image + 1                   # the smallest batch whose fp32 stream alone exceeds 2^31 bytes
    assert B * per_image > 2 ** 31 >= (B - 1) * per_image
    g = torch.Generator().manual_seed(99)
    x8 = torch.randint(0, 256, (B, 3, H, W), generator=g, dtype=torch.uint8).to(dev)
    c = torch.rand(B, 3, generator=g).to(dev)
    # the exact quotient the stem reads from 8-bit images (torch divides by a CUDA scalar as a reciprocal multiply,
    # 1 ulp off for some codes)
    x = (x8.double() / 255.0).float()
    frame, out = step_through(m, x, c, Emulation(m, DT[operands], dev), slice(B - 2, B))
    assert out["stream_bytes"] == B * per_image and out["stream_bytes"] > 2 ** 31
    label = f"{name}/{operands}/B{B}/Cp{Cp}"
    _report(label, out)
    _check_blocks(out, name, operands, label)
    y = m.upscale(x, c)
    assert torch.equal(y, frame), "the whole call differs from the staged one"
    del frame
    for i in range(B):
        assert torch.equal(m.upscale(x[i:i + 1], c[i:i + 1]), y[i:i + 1]), f"{label}: image {i} differs from itself alone"
    y8 = m.upscale(x8, c)
    for i in range(B):
        assert torch.equal(m.upscale(x8[i:i + 1], c[i:i + 1]), y8[i:i + 1]), f"{label}: 8-bit image {i} differs alone"
    d = (y8.int() - torch.floor(y * 255.0 + 0.5).int()).abs()
    assert int(d.max()) <= 1 and float((d == 0).float().mean()) >= 0.999, (label, int(d.max()), float((d == 0).float().mean()))
    if operands == "float16":
        assert not m.saturated()


# --------------------------------------------------------------------------------------------------------------------
# negative controls: wrong references must be rejected
# --------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("operands", ["float16", "bfloat16"])
@pytest.mark.parametrize("name,B,H,W", [("MewZoom-4X-Ctrl", 1, 540, 960), ("MewZoom-2X-Ctrl", 2, 540, 960)])
def test_wrong_references_are_rejected(fp32_exact, dev, name, B, H, W, operands):
    """(a) - (d): accepted with the right reference, each wrong one rejected at every block where it applies."""
    m = _model(name, operands, dev)
    x, c = _images(B, H, W, 555, dev)
    dt = DT[operands]
    variants = {"toward_zero": Emulation(m, dt, dev, hidden_rounding="toward_zero"),
                "film_of_next_layer": Emulation(m, dt, dev, film_of_next_layer=True),
                "conv1_transposed": Emulation(m, dt, dev, conv1_transposed=True)}
    _, out = step_through(m, x, c, Emulation(m, dt, dev), slice(0, B), variants, stale_zb=True)
    label = f"controls/{name}/{operands}"
    _report(label, out)
    _check_blocks(out, name, operands, label)
    L = m.num_encoder_layers
    applies = {"toward_zero": range(L), "film_of_next_layer": range(L - 1), "conv1_transposed": range(L),
               "stale_zb": range(1, L)}
    for vname, blocks in applies.items():
        assert sorted(out["variants"][vname]) == list(blocks), vname
        passed = [l for l, st in out["variants"][vname].items() if not _rejected(st, name, operands)]
        assert not passed, f"{label}: the wrong reference '{vname}' passes the bounds at blocks {passed}"


@pytest.mark.gpu
def test_interpolated_skip_at_r3_is_rejected(fp32_exact, dev):
    """(e): at r = 3 F.interpolate evaluates the bicubic phase per pixel in fp32 and is off by up to 1e-4 on a
    960-pixel row; the head bound accepts the exact phase table the kernel uses and rejects F.interpolate."""
    m = _model("MewZoom-3X-Ctrl", "float16", dev)
    H, W = 540, 960
    x, c = _images(1, H, W, 556, dev)
    L = m.num_encoder_layers
    ws = m.stage_workspace(tuple(x.shape), dev)
    frame = torch.full((1, 3, 3 * H, 3 * W), float("nan"), device=dev)
    m.upscale_stage(x, c, frame, (0, H, 0, W), (0, 0), 0, L, ws)
    zb = _nchw(m.stage_views(ws, tuple(x.shape), L)[1][..., :m.num_channels])
    right = _stats(frame - Emulation(m, torch.float16, dev).head(zb, x)[0], "bcyx", 0)
    wrong = _stats(frame - Emulation(m, torch.float16, dev, skip="interpolate").head(zb, x)[0], "bcyx", 0)
    _report("controls/interpolate_r3", {"table": right, "interpolate": wrong})
    assert right["max"] <= HEAD_BOUNDS[0] and right["p9999"] <= HEAD_BOUNDS[1], right
    assert wrong["max"] > HEAD_BOUNDS[0] or wrong["p9999"] > HEAD_BOUNDS[1], wrong
