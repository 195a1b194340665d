"""GPU: the fp16 range guard -- fp16 operands end at 65504, and a value beyond that is never returned clipped.

  A. Every kernel that rounds fp32 values into a 16-bit operand rounds at the edge of the range as the references do,
     bit for bit: fp16 as ``ref16(v) = v.clamp(-65504, 65504).to(torch.float16)`` (``cvt.rn.satfinite``: +-65504, not
     inf; NaN stays NaN; subnormals round to nearest even), bf16 as ``v.to(torch.bfloat16)``.  NaN is compared by
     NaN-ness, not payload.
  B. At model level every site that rounds a value beyond 65504 raises the flag (``model.saturated()``) -- the stem, the
     residual stream's shadow and the hidden tensor, on fused blocks, two-kernel tcgen05 blocks (both residual
     epilogues), the SIMT twin and convolutions sliced over output channels -- and in-range values do not.
  C. Every entry point honours the flag: with "float16" it raises instead of returning (in the call itself where the
     call synchronises anyway, else on the next call); with "auto" the calls that can be repeated return the bf16
     result, the others raise.

Magnitudes in (65504, 65520) round to 65504 without clipping; whether they raise the flag is left unspecified.
"""
import pytest
import torch
from torch.nn import functional as F

from oracle import make_oracle, max_abs_err
from tests.test_gpu_robustness import _scaled_block

pytestmark = pytest.mark.gpu

F16_MAX = 65504.0
INF, NAN = float("inf"), float("nan")
# the edge of the fp16 range and its subnormals, both signs
EDGE = [0.0, -0.0, 2.0**-24, 2.0**-25, 3 * 2.0**-25, 2.0**-14, 65504.0, 65519.99, 65520.0, 1e5, 3e38, INF]
VALUES = EDGE + [-v for v in EDGE[2:]] + [NAN]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda", 0)


def ref16(v, dt=torch.float16):
    return v.clamp(-F16_MAX, F16_MAX).to(dt) if dt == torch.float16 else v.to(dt)


def same16(got, want, what=""):
    """16-bit tensors equal bit for bit; NaN compared by NaN-ness."""
    got, want = got.cpu(), want.cpu()
    assert got.dtype == want.dtype and got.shape == want.shape, what
    gn, wn = torch.isnan(got.float()), torch.isnan(want.float())
    assert torch.equal(gn, wn), (what, gn.sum().item(), wn.sum().item())
    g, w = got.view(torch.int16)[~gn], want.view(torch.int16)[~wn]
    bad = (g != w).nonzero()
    assert bad.numel() == 0, (what, got.float()[~gn][bad[:4, 0]].tolist(), want.float()[~wn][bad[:4, 0]].tolist())


def same32(got, want, what=""):
    """fp32 values equal (-0 == +0), NaN where NaN."""
    torch.testing.assert_close(got.cpu(), want.cpu(), rtol=0, atol=0, equal_nan=True, msg=what)


def _spread(n, shape):
    """VALUES over a tensor of `shape`: every value at many positions and channels."""
    v = torch.tensor(VALUES, dtype=torch.float32)
    return v[(torch.arange(n) * 7 + torch.arange(n) // len(VALUES)) % len(VALUES)].reshape(shape)


# ---------------------------------------------------------------------------------------------------------------------
# A. rounding at the edge of the range, per kernel
# ---------------------------------------------------------------------------------------------------------------------
DTYPES = [torch.float16, torch.bfloat16]


@pytest.mark.parametrize("dt", DTYPES)
def test_stem_rounds_at_the_edge(dev, dt):
    """Stem weights 0 and the values in the bias: zf holds them as they are (fma(0, x, b) = b), the shadow is ref16(zf)."""
    from ultrazoom_b200 import ops

    Cc = len(VALUES)
    bias = torch.tensor(VALUES)
    x = torch.rand(2, 3, 5, 37, generator=torch.Generator().manual_seed(1)).to(dev)
    zf, zb = ops.stem_pack(x, torch.zeros(Cc, 3, 1, 1), bias, dtype=dt)
    same32(zf[..., :Cc], bias.expand(2, 5, 37, Cc), "zf")
    same16(zb, ref16(zf, dt), "zb")
    assert float(zf[..., Cc:].abs().max()) == 0.0 if zf.shape[-1] > Cc else True


# conv2 tunes: each residual epilogue of the tcgen05 kernel (conv_tc.cu fill_geometry).  One-row patches leave one residual
# row per warp (res_rows == 1): the sliced epilogue.  Two-row patches on four epilogue warps with a streamed filter bank fit
# the deep staging (staging 2, res_rows == 2): the all-rows epilogue.
RESIDUAL_TUNES = {"default": {}, "sliced": dict(rows=1), "all-rows": dict(rows=2, epi_warps=4, resident=2)}


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("how", list(RESIDUAL_TUNES) + ["simt"])
def test_conv_residual_shadow_rounds_at_the_edge(dev, how, dt):
    """conv3x3 mode 1 on a zero input (non-negative weights: the accumulator is +0): zf = zf0 + 0 -- unchanged but for
    -0, which becomes +0 -- and the shadow is ref16(zf0 + 0)."""
    from ultrazoom_b200 import _native, ops

    B, H, W, cin, cout = 1, 6, 140, 96, 48
    w = torch.rand(cout, cin, 3, 3, generator=torch.Generator().manual_seed(2)) / 100
    wp = ops.pack_conv_weight(w, dev, dtype=dt)
    zf0 = _spread(B * H * W * cout, (B, H, W, cout))
    zf = zf0.to(dev)
    tc = how != "simt"
    zb = ops.conv3x3(torch.zeros(B, H, W, cin, dtype=dt, device=dev), wp, 1, None, zf, use_tc=tc,
                     tune=_native.tune(**RESIDUAL_TUNES[how]) if tc else None)
    same32(zf, zf0 + 0.0, "zf")
    same16(zb, ref16(zf0 + 0.0, dt), "zb")


@pytest.mark.parametrize("dt", DTYPES)
@pytest.mark.parametrize("use_tc", [True, False])
def test_conv_hidden_rounds_at_the_edge(dev, use_tc, dt):
    """conv3x3 mode 0 on a zero input with FiLM scale 0 and shift s stores SiLU(s) = h + h tanh.approx(h), h = s / 2.
    For |s| >= 1000 tanh.approx returns exactly +-1: the stored value is ref16(s) for s > 0 (+inf included) and +0 for
    s < 0 (h - h); NaN stays NaN."""
    from ultrazoom_b200 import ops

    B, H, W, cin, cout = 1, 3, 130, 48, 96
    big = [1000.0, 4096.0, 65504.0, 65519.99, 65520.0, 1e5, 3e38]
    s = torch.tensor((big + [-v for v in big] + [INF, NAN]) * 6)[:cout]
    film = torch.zeros(B, 2, cout)
    film[:, 1] = s
    wp = ops.pack_conv_weight(torch.randn(cout, cin, 3, 3, generator=torch.Generator().manual_seed(3)) / 20, dev, dtype=dt)
    got = ops.conv3x3(torch.zeros(B, H, W, cin, dtype=dt, device=dev), wp, 0, film.to(dev), use_tc=use_tc)
    want = torch.where(s < 0, torch.zeros_like(s), s)
    same16(got, ref16(want, dt).expand(B, H, W, cout), "hidden")


def _fused_operands(dt, dev):
    from ultrazoom_b200 import ops

    g = torch.Generator().manual_seed(4)
    w1 = torch.randn(96, 48, 3, 3, generator=g) / 20
    w2 = torch.rand(48, 96, 3, 3, generator=g) * 1e-5          # non-negative: a zero hidden tensor accumulates +0
    return w1, w2, ops.pack_conv_weight(w1, dev, dtype=dt), ops.pack_conv_weight(w2, dev, dtype=dt)


@pytest.mark.parametrize("dt", DTYPES)
def test_fused_block_residual_shadow_rounds_at_the_edge(dev, dt):
    """ops.block_fused on a zero stream with zero FiLM (hidden = SiLU(0) = 0): zf = zf0 + 0, zb_out = ref16(zf0 + 0)."""
    from ultrazoom_b200 import ops

    B, H, W = 2, 9, 140
    _, _, w1p, w2p = _fused_operands(dt, dev)
    zf0 = _spread(B * H * W * 48, (B, H, W, 48))
    zf = zf0.to(dev)
    out = ops.block_fused(torch.zeros(B, H, W, 48, dtype=dt, device=dev), w1p, w2p, torch.zeros(B, 2, 96, device=dev), zf)
    same32(zf, zf0 + 0.0, "zf")
    same16(out, ref16(zf0 + 0.0, dt), "zb_out")


def test_fused_block_saturated_hidden_equals_two_kernels_and_reference(dev):
    """FiLM shift 7e4 (scale 0): every hidden value is SiLU(7e4) = 7e4, stored as 65504 by both paths.  The fused block
    equals the two-kernel path and a float64 reference built on hid = ref16(7e4) = 65504 -- a path that kept 7e4, or
    stored inf, would be 7 % off or not finite."""
    from ultrazoom_b200 import ops

    dt = torch.float16
    B, H, W = 1, 11, 133
    g = torch.Generator().manual_seed(5)
    _, w2, w1p, w2p = _fused_operands(dt, dev)
    zb = torch.randn(B, H, W, 48, generator=g).to(dt)
    zf0 = torch.randn(B, H, W, 48, generator=g)
    film = torch.zeros(B, 2, 96)
    film[:, 1] = 7e4
    hid = ops.conv3x3(zb.to(dev), w1p, 0, film.to(dev))
    same16(hid, torch.full((B, H, W, 96), F16_MAX, dtype=dt), "two-kernel hidden")
    zf_two = zf0.to(dev)
    ops.conv3x3(hid, w2p, 1, None, zf_two)
    zf_one = zf0.to(dev)
    out = ops.block_fused(zb.to(dev), w1p, w2p, film.to(dev), zf_one)
    want = zf0.double() + F.conv2d(torch.full((B, 96, H, W), F16_MAX, dtype=torch.float64), w2.to(dt).double(),
                                   padding=1).permute(0, 2, 3, 1)
    tol = 3e-5 * want.abs().max().item()
    assert torch.isfinite(zf_one).all()
    assert (zf_one.cpu().double() - want).abs().max().item() <= tol
    assert (zf_one - zf_two).abs().max().item() <= tol
    same16(out, ref16(zf_one), "zb_out")


# ---------------------------------------------------------------------------------------------------------------------
# B. the flag, site by site, at model level
# ---------------------------------------------------------------------------------------------------------------------
def _cfg(name, **over):
    from ultrazoom_b200 import MODEL_CONFIGS

    cfg = dict(MODEL_CONFIGS[name]) if name in MODEL_CONFIGS else {}
    cfg.update(num_encoder_layers=3, **over)
    return cfg


# name -> (config, per-model setting, a channel of the residual stream: in conv2's last output slice)
MODELS = {
    "2x-fused": (_cfg("MewZoom-2X-Ctrl"), None, 41),
    "2x-two-kernels": (_cfg("MewZoom-2X-Ctrl"), "two-kernels", 41),
    "3x": (_cfg("MewZoom-3X-Ctrl"), None, 50),
    "4x": (_cfg("MewZoom-4X-Ctrl"), None, 90),
    "2x-simt": (_cfg("MewZoom-2X-Ctrl"), "simt", 41),
    "2x-c160-sliced": (_cfg("", upscale_ratio=2, num_channels=160, hidden_ratio=2, control_features=3), None, 153),
}


def _model(name, dev, operand_dtype="float16"):
    from ultrazoom_b200 import MewZoom, _native

    cfg, how, _ = MODELS[name]
    torch.manual_seed(7)
    m = MewZoom(**cfg, operand_dtype=operand_dtype).to(dev).eval()
    if how == "two-kernels":
        m.set_conv_tune(0, dev, block=2)
    if how == "simt":
        m._flags_extra = _native.FLAG_SIMT_CONV
    return m


def _inputs(dev, shape=(1, 3, 12, 70), seed=8):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g).to(dev), torch.rand(shape[0], 3, generator=g).to(dev)


def _hidden_scaled(m, name, k):
    """The hidden tensor of block 1 grows by k, its output does not (conv1 x k, conv2 / k).  On the sliced model only
    conv1's second slice (hidden channels 160..319) and the conv2 input columns it feeds are scaled."""
    if name != "2x-c160-sliced":
        return _scaled_block(m, k)
    sd = {n: t.clone() for n, t in m.state_dict().items()}
    sd["encoder.1.convnet.conv1.weight"][160:] *= k
    sd["encoder.1.convnet.conv2.weight"][:, 160:] /= k
    return sd


@pytest.mark.parametrize("name", list(MODELS))
def test_every_site_raises_the_flag(dev, name):
    """Sites isolated with ``upscale_stage``: stage [0, 0) runs FiLM and the stem only; a value written into the fp32
    stream between stages [0, 1) and [1, 2) reaches only block 1's residual shadow; a scaled block only its hidden
    tensor.  Each saturating case has an in-range control that leaves the flag down."""
    m = _model(name, dev)
    ch = MODELS[name][2]
    x, c = _inputs(dev)
    shape = tuple(x.shape)
    r = m.upscale_ratio
    frame = torch.zeros(shape[0], 3, shape[2] * r, shape[3] * r, device=dev)
    ws = m.stage_workspace(shape, dev)

    def stage(lo, hi):
        m.upscale_stage(x, c, frame, (0, 0, 0, 0), (0, 0), lo, hi, ws)

    assert not m.saturated()
    # stem: bias beyond the range -> flag; exactly 65504 with zero weights -> none
    w0, b0 = m.stem.conv.weight.detach().clone(), m.stem.conv.bias.detach().clone()
    with torch.no_grad():
        m.stem.conv.bias[ch] = 7e4
    stage(0, 0)
    assert m.saturated(reset=True), "stem"
    with torch.no_grad():
        m.stem.conv.weight.zero_()
        m.stem.conv.bias[ch] = F16_MAX
    stage(0, 0)
    assert not m.saturated(), "stem at 65504"
    with torch.no_grad():
        m.stem.conv.weight.copy_(w0)
        m.stem.conv.bias.copy_(b0)
    # residual shadow of block 1 (on the sliced model: a channel of conv2's second slice)
    for v, up in ((6e4, False), (7e4, True)):
        stage(0, 1)
        zf, _ = m.stage_views(ws, shape, 1)
        zf[0, 5, 33, ch] = v
        stage(1, 2)
        assert m.saturated(reset=True) == up, ("residual", v)
    if name == "2x-two-kernels":       # both residual epilogues of the tcgen05 kernel
        for tune in RESIDUAL_TUNES.values():
            m.set_conv_tune(1, dev, **tune)
            stage(0, 1)
            m.stage_views(ws, shape, 1)[0][0, 5, 33, ch] = 7e4
            stage(1, 2)
            assert m.saturated(reset=True), ("residual", tune)
        m.set_conv_tune(1, dev)
    # hidden tensor of block 1 (on the sliced model: conv1's second slice only)
    m.upscale(x, c)
    assert not m.saturated(), "hidden, unscaled"
    m.load_state_dict(_hidden_scaled(m, name, 1e6))
    m.upscale(x, c)
    assert m.saturated(reset=True), "hidden"


def test_packers_accept_65504_and_reject_65536(dev):
    """A conv weight of exactly 65504 is accepted by the host packer (parameters on the CPU) and the device packer
    (parameters on the GPU) and gives a finite image; 65536 is rejected by both.  A bf16 model given 1e5 in the weights
    and in the stem bias never raises the flag."""
    from ultrazoom_b200 import MewZoom

    cfg = _cfg("MewZoom-2X-Ctrl")
    x, c = _inputs(dev)
    o = make_oracle(cfg, seed=9)
    for v, ok in ((F16_MAX, True), (65536.0, False)):
        sd = {n: t.clone() for n, t in o.state_dict().items()}
        sd["encoder.2.convnet.conv2.weight"][3, 5, 1, 1] = v
        host = MewZoom(**cfg)
        host.load_state_dict(sd)
        devm = MewZoom(**cfg)
        devm.load_state_dict(sd)
        devm = devm.to(dev).eval()
        if ok:
            host._engine(dev)
            y = devm.upscale(x, c)
            assert torch.isfinite(y).all()
            devm.saturated(reset=True)
        else:
            with pytest.raises(AssertionError, match="fp16 operand range"):
                host._engine(dev)
            with pytest.raises(AssertionError, match="fp16 operand range"):
                devm.upscale(x, c)
    sd = {n: t.clone() for n, t in o.state_dict().items()}
    sd["encoder.2.convnet.conv2.weight"][3, 5, 1, 1] = 1e5
    sd["stem.conv.bias"][7] = 1e5
    mb = MewZoom(**cfg, operand_dtype="bfloat16")
    mb.load_state_dict(sd)
    mb = mb.to(dev).eval()
    assert torch.isfinite(mb.upscale(x, c)).all()
    torch.cuda.synchronize()
    assert not mb._engine(dev).saturated()


# ---------------------------------------------------------------------------------------------------------------------
# C. every entry point honours the flag
# ---------------------------------------------------------------------------------------------------------------------
CFG = dict(upscale_ratio=2, num_channels=48, hidden_ratio=2, num_encoder_layers=4, control_features=3)
TOL_2X = 4e-3          # the 2X max-abs tolerance of tests/test_gpu_parity.py


@pytest.fixture(scope="module")
def ckpt():
    """A checkpoint whose hidden tensor overflows fp16 (test_gpu_robustness), an input and the fp32 oracle's image."""
    o = make_oracle(CFG, seed=5)
    sd = _scaled_block(o, 3.0e5)
    o.load_state_dict(sd)
    g = torch.Generator().manual_seed(6)
    x, c = torch.rand(1, 3, 24, 136, generator=g), torch.rand(1, 3, generator=g)
    with torch.inference_mode():
        ref = o.upscale(x, c)
    return sd, x, c, ref


def _m(sd, dev, operand_dtype="float16"):
    from ultrazoom_b200 import MewZoom

    m = MewZoom(**CFG, operand_dtype=operand_dtype)
    m.load_state_dict(sd)
    return m.to(dev).eval()


def _tile(x):
    from ultrazoom_b200.sharding import halo_radius, plan_tiles

    return plan_tiles(x.shape[2], x.shape[3], 1, 2, halo_radius(CFG["num_encoder_layers"]))[1]


def test_a_clip_would_be_visible(dev, ckpt):
    """The fp16 result of this checkpoint is clipped: further from the oracle than the 2X tolerance (so an entry point
    that returned it would return a wrong image), while bf16 is within it."""
    sd, x, c, ref = ckpt
    m = _m(sd, dev)
    y = m.upscale(x.to(dev), c.to(dev)).cpu()
    assert m.saturated(reset=True)
    assert max_abs_err(y, ref) > TOL_2X
    assert max_abs_err(_m(sd, dev, "bfloat16").upscale(x.to(dev), c.to(dev)).cpu(), ref) <= 2e-2


def test_float16_every_entry_point_raises(dev, ckpt):
    """operand_dtype="float16": calls that synchronise anyway (upscale_host, host_wait, capture) raise themselves; the
    others return at once and the next call on the model raises.  ``replay()`` is the unchecked path."""
    from ultrazoom_b200.sharding import run_tile_into, upscale_tiled_refresh

    sd, x, c, _ = ckpt
    xd, cd = x.to(dev), c.to(dev)
    m = _m(sd, dev)
    raises = pytest.raises(RuntimeError, match="fp16 range")
    frame = torch.zeros(1, 3, 48, 272, device=dev)
    t = _tile(x)
    L = CFG["num_encoder_layers"]

    def asynchronous(call):
        call()
        torch.cuda.synchronize()
        with raises:
            call()
        assert m.saturated(reset=True)

    asynchronous(lambda: m.upscale(xd, cd))
    asynchronous(lambda: m.forward(xd, cd))
    asynchronous(lambda: m.upscale_into(xd, cd, frame, (0, 24, 0, 136), (0, 0)))
    asynchronous(lambda: run_tile_into(m, xd, cd, t, 2, frame))
    ws = m.stage_workspace(xd.shape, dev)
    asynchronous(lambda: m.upscale_stage(xd, cd, frame, (0, 24, 0, 136), (0, 0), 0, L, ws))
    with raises:                       # (a stage of the same call may already see an earlier group's flag)
        for _ in range(2):
            upscale_tiled_refresh(m, xd, cd, 2, L, 1, 2, 2, frame)
            torch.cuda.synchronize()
    assert m.saturated(reset=True)
    with raises:
        m.upscale_host(x, c)
    assert m.saturated(reset=True)
    m.upscale_host(x, c, lane=0)
    with raises:
        m.host_wait(0)
    assert m.saturated(reset=True)
    with raises:
        m.capture(xd, cd)
    assert m.saturated(reset=True)


@pytest.mark.parametrize("operand_dtype", ["float16", "auto"])
def test_graph_call_after_a_saturated_replay_raises(dev, operand_dtype):
    """A graph captured on in-range values, replayed with a control vector that drives the hidden tensors beyond the
    range: the flag goes up, and the next ``__call__`` raises (in "auto" too: a graph cannot be re-run with another
    operand type; the model moves on to bf16)."""
    from ultrazoom_b200 import MewZoom

    torch.manual_seed(10)
    m = MewZoom(**CFG, operand_dtype=operand_dtype).to(dev).eval()
    x, c = _inputs(dev)
    g = m.capture(x, c)
    want = g(x, c).clone()
    assert torch.equal(g(x, c), want) and not m.saturated()
    g.replay()
    g.c.fill_(1e7)                     # FiLM scales ~1e6
    g.replay()
    assert m.saturated()
    with pytest.raises(RuntimeError, match="fp16 range"):
        g(x, c)
    if operand_dtype == "auto":
        assert m._auto_dtype == "bfloat16" and not m.saturated()
    else:
        assert m.saturated(reset=True)
    assert torch.equal(g(x, c), want)


def test_auto_repeats_what_it_can_and_raises_otherwise(dev, ckpt):
    """operand_dtype="auto" on the saturating checkpoint: upscale, forward, upscale_host and upscale_into return the
    result of a bfloat16 model, bit for bit; stages and lanes raise on their next call; a graph captured on this
    checkpoint records and holds the bf16 engine."""
    sd, x, c, _ = ckpt
    xd, cd = x.to(dev), c.to(dev)
    mb = _m(sd, dev, "bfloat16")
    raises = pytest.raises(RuntimeError, match="fp16 range")
    L = CFG["num_encoder_layers"]

    def fresh():
        a = _m(sd, dev, "auto")
        assert a._auto_dtype == "float16"
        return a

    a = fresh()
    assert torch.equal(a.upscale(xd, cd), mb.upscale(xd, cd)) and a._auto_dtype == "bfloat16"
    a = fresh()
    assert torch.equal(a.forward(xd, cd), mb.forward(xd, cd)) and a._auto_dtype == "bfloat16"
    a = fresh()
    assert torch.equal(a.upscale_host(x, c), mb.upscale_host(x, c)) and a._auto_dtype == "bfloat16"
    a = fresh()
    fa, fb = torch.full((1, 3, 60, 300), -1.0, device=dev), torch.full((1, 3, 60, 300), -1.0, device=dev)
    a.upscale_into(xd, cd, fa, (2, 20, 4, 130), (6, 10))
    mb.upscale_into(xd, cd, fb, (2, 20, 4, 130), (6, 10))
    assert torch.equal(fa, fb) and a._auto_dtype == "bfloat16"
    # stages
    a = fresh()
    frame = torch.zeros(1, 3, 48, 272, device=dev)
    ws = a.stage_workspace(xd.shape, dev)
    a.upscale_stage(xd, cd, frame, (0, 0, 0, 0), (0, 0), 0, L, ws)
    torch.cuda.synchronize()
    with raises:
        a.upscale_stage(xd, cd, frame, (0, 0, 0, 0), (0, 0), 0, L, ws)
    assert a._auto_dtype == "bfloat16"
    a.upscale_stage(xd, cd, frame, (0, 0, 0, 0), (0, 0), 0, L, ws)     # the repeated call runs with bf16
    assert torch.equal(frame, mb.upscale(xd, cd))
    # lanes
    a = fresh()
    out = a.upscale_host(x, c, lane=1)
    with raises:
        a.host_wait(1)
    assert a._auto_dtype == "bfloat16"
    a.upscale_host(x, c, out=out, lane=1)
    a.host_wait(1)
    assert torch.equal(out, mb.upscale_host(x, c))
    # a graph captured in "auto" holds the engine its warm-up switched to
    a = fresh()
    g = a.capture(xd, cd)
    assert g.engine.operand_dtype == "bfloat16" and a._auto_dtype == "bfloat16"
    assert torch.equal(g(xd, cd), mb.upscale(xd, cd))


@pytest.mark.parametrize("operand_dtype", ["float16", "auto"])
def test_both_lanes_in_flight_are_reported(dev, ckpt, operand_dtype):
    """The double-buffered loop: frames on both lanes before the first ``host_wait``, both clipped.  Each wait raises.
    In "auto" the first wait switches the model to bf16; the second still waits on the fp16 engine that runs its frame
    and reports it (the flag is one word per engine: a lane's frame in flight when it is found up is reported too)."""
    sd, _, _, _ = ckpt
    g = torch.Generator().manual_seed(11)
    x, c = torch.rand(8, 3, 192, 256, generator=g).pin_memory(), torch.rand(1, 3, generator=g)
    m = _m(sd, dev, operand_dtype)
    m._engine(dev)                                   # (packs the weights: the lanes below only enqueue)
    outs = [torch.empty(8, 3, 384, 512, pin_memory=True) for _ in (0, 1)]   # (pinned: the copies do not block)
    for ln in (0, 1):
        m.upscale_host(x, c, out=outs[ln], lane=ln)
    for ln in (0, 1):
        with pytest.raises(RuntimeError, match="fp16 range"):
            m.host_wait(ln)
    if operand_dtype == "auto":
        assert m._auto_dtype == "bfloat16"
        for ln in (0, 1):
            m.upscale_host(x, c, out=outs[ln], lane=ln)
        m.host_wait()
        want = _m(sd, dev, "bfloat16").upscale_host(x, c)
        assert torch.equal(outs[0], want) and torch.equal(outs[1], want)


@pytest.mark.parametrize("then", ["upscale", "forward", "upscale_into", "upscale_host"])
def test_auto_does_not_absorb_an_earlier_asynchronous_clip(dev, ckpt, then):
    """"auto": a stage that clipped, followed at once (no synchronisation) by a call that "auto" can re-run.  That call
    raises -- the stage's frame was clipped and already handed out -- rather than taking the stage's flag for its own and
    re-running only itself with bf16.  Repeated, it runs with bf16."""
    sd, x, c, _ = ckpt
    xd, cd = x.to(dev), c.to(dev)
    a = _m(sd, dev, "auto")
    frame = torch.zeros(1, 3, 48, 272, device=dev)
    calls = {"upscale": lambda: a.upscale(xd, cd), "forward": lambda: a.forward(xd, cd),
             "upscale_into": lambda: a.upscale_into(xd, cd, frame, (0, 24, 0, 136), (0, 0)),
             "upscale_host": lambda: a.upscale_host(x, c)}
    a.upscale_stage(xd, cd, frame, (0, 0, 0, 0), (0, 0), 0, CFG["num_encoder_layers"], a.stage_workspace(xd.shape, dev))
    with pytest.raises(RuntimeError, match="fp16 range"):
        calls[then]()
    assert a._auto_dtype == "bfloat16"
    calls[then]()
    assert torch.equal(a.upscale(xd, cd), _m(sd, dev, "bfloat16").upscale(xd, cd))


def test_auto_does_not_absorb_a_clipped_replay(dev):
    """"auto": a graph replay that clipped (the graph holds the fp16 engine), followed at once by ``upscale``: it raises."""
    from ultrazoom_b200 import MewZoom

    torch.manual_seed(10)
    m = MewZoom(**CFG, operand_dtype="auto").to(dev).eval()
    x, c = _inputs(dev)
    g = m.capture(x, c)
    g.c.fill_(1e7)                     # FiLM scales ~1e6
    g.replay()
    with pytest.raises(RuntimeError, match="fp16 range"):
        m.upscale(x, c)
    assert m._auto_dtype == "bfloat16"
