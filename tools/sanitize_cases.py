"""Small-shape run of every kernel variant behind the C ABI, for `compute-sanitizer --tool memcheck|racecheck|synccheck`
(tools/sanitize.sh; SURVEY.md section 5 "race detection"): bicubic r = 2/3/4, stem, FiLM table, device weight packer, the
tcgen05 convolution in every epilogue MODE (0 conv1+FiLM+SiLU, 1 conv2+residual, 2 head) and VAR (0 plain,
1 CTA pair / cta_group::2, 2 vertical taps fused along N), resident and streamed filter banks, 4 and 8 epilogue warps,
the SIMT twin, the fused encoder block (one segment; several segments and rounds per CTA pair), the U-Net operators
(tcgen05 tf32 mix / crush and their fp32 twins, NHWC pixel shuffle, crop / pad, quality head), and whole small models
through mz_upscale (dependent launches included).  Every result is also checked against its twin (the SIMT kernel, the
two-kernel block, the fp32 GEMM, torch) so that a sanitizer-induced timing change that exposes a protocol bug shows up
as a mismatch."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ultrazoom_b200 import MODEL_CONFIGS, MewZoom, _native, ops  # noqa: E402


def main():
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(0)
    n = 0
    for r in (2, 3, 4):
        ops.bicubic(torch.rand(1, 3, 9, 37, generator=g).to(dev), r)
        n += 1
    cases = [  # cin, cout, (B,H,W), tune
        (48, 96, (1, 5, 150), {}), (48, 96, (1, 5, 150), dict(fuse=2)), (48, 96, (1, 5, 150), dict(resident=2)),
        (96, 48, (1, 6, 140), {}), (96, 48, (1, 6, 140), dict(fuse=2)), (96, 192, (1, 4, 260), {}),
        (96, 192, (1, 4, 260), dict(pair=1)), (96, 192, (1, 4, 260), dict(pair=2, resident=2)),
        (192, 96, (1, 4, 260), {}), (192, 96, (1, 4, 260), dict(pair=2)), (64, 128, (1, 3, 130), dict(epi_warps=4)),
        (128, 64, (2, 3, 130), dict(epi_warps=4)), (32, 48, (1, 7, 130), dict(fuse=1, rows=4)),
    ]
    for cin, cout, (B, H, W), tune in cases:
        cin_p, cout_p = ops.padded_channels(cin), ops.padded_channels(cout)
        inp = torch.zeros(B, H, W, cin_p, dtype=torch.float16)
        inp[..., :cin] = torch.randn(B, H, W, cin, generator=g).half()
        w = torch.randn(cout, cin, 3, 3, generator=g) / (3.0 * cin ** 0.5)
        wp = ops.pack_conv_weight(w, dev)
        film = torch.ones(B, 2, cout_p)
        film[:, 1] = 0.1
        t = _native.tune(**tune)
        a = ops.conv3x3(inp.to(dev), wp, 0, film.to(dev), use_tc=True, tune=t)
        b = ops.conv3x3(inp.to(dev), wp, 0, film.to(dev), use_tc=False)
        assert (a.float() - b.float()).abs().max().item() <= 2e-2, ("mode 0", cin, cout, tune)
        if cout_p <= 128:
            zf0 = torch.randn(B, H, W, cout_p, generator=g)
            zfa, zfb = zf0.to(dev).contiguous(), zf0.to(dev).contiguous()
            ops.conv3x3(inp.to(dev), wp, 1, None, zfa, use_tc=True, tune=t)
            ops.conv3x3(inp.to(dev), wp, 1, None, zfb, use_tc=False)
            assert (zfa - zfb).abs().max().item() <= 1e-3, ("mode 1", cin, cout, tune)
        n += 1
    # the fused encoder block against the same block as two kernels (one segment; several segments and rounds)
    for (B, H, W), seg_rows, max_ctas in (((1, 5, 130), 0, 0), ((2, 9, 260), 2, 2)):
        zf0 = torch.randn(B, H, W, 48, generator=g)
        zb = zf0.half().to(dev)
        w1p = ops.pack_conv_weight(torch.randn(96, 48, 3, 3, generator=g) / 20.0, dev)
        w2p = ops.pack_conv_weight(torch.randn(48, 96, 3, 3, generator=g) / 30.0, dev)
        film = torch.ones(B, 2, 96)
        film[:, 1] = 0.1
        fd = film.to(dev)
        zf_one, zf_two = zf0.to(dev).contiguous(), zf0.to(dev).contiguous()
        ops.block_fused(zb, w1p, w2p, fd, zf_one, seg_rows=seg_rows, max_ctas=max_ctas)
        ops.conv3x3(ops.conv3x3(zb, w1p, 0, fd, use_tc=True), w2p, 1, None, zf_two, use_tc=True)
        assert (zf_one - zf_two).abs().max().item() <= 3e-3, ("block_fused", B, H, W, seg_rows, max_ctas)
        n += 1
    # U-Net operators: the tcgen05 tf32 mix / crush against their fp32 twins (with the 16-bit shadow and padded
    # pitches), the NHWC pixel shuffle, crop / pad and the quality head against torch on the same device
    from oracle import unet_oracle as U
    from ultrazoom_b200 import unet as N

    x, z = torch.randn(2, 9, 130, 48, generator=g).to(dev), torch.randn(2, 9, 130, 48, generator=g).to(dev)
    wm = torch.randn(48, 96, 1, 1, generator=g) / 10.0
    a, a16 = N.adaptive_residual_mix(x, z, wm, torch.tensor(0.3), "tf32", shadow=torch.float16)
    b, b16 = N.adaptive_residual_mix(x, z, wm, torch.tensor(0.3), "fp32", shadow=torch.float16)
    assert (a - b).abs().max().item() <= 3e-2 and torch.equal(a16, a.half()) and torch.equal(b16, b.half()), "mix"
    n += 1
    for f in (2, 3, 4):
        wc = torch.randn(40, 48, f, f, generator=g) / (4.0 * f)
        a, a16 = N.pixel_crush(x, wc, f, "tf32", shadow=torch.float16)
        b, b16 = N.pixel_crush(x, wc, f, "fp32", shadow=torch.float16)
        assert (a - b).abs().max().item() <= 3e-2 and torch.equal(a16, a.half()) and torch.equal(b16, b.half()), ("crush", f)
        n += 1
    stream = torch.cuda.current_stream(dev).cuda_stream
    lib = _native.load()
    xp, zp = torch.randn(1, 7, 131, 48, generator=g).to(dev), torch.randn(1, 7, 131, 48, generator=g).to(dev)
    wt_mix = (torch.randn(40, 80, generator=g) / 10.0).to(dev)
    wt_crush = (torch.randn(32, 4 * 40, generator=g) / 10.0).to(dev)
    outs = []
    for math in (_native.MATH_TF32, _native.MATH_FP32):     # 40 channels at a pitch of 48 through the C ABI
        mix = torch.zeros(1, 7, 131, 48, device=dev)
        _native.check(lib.mz_adaptive_mix(xp.data_ptr(), zp.data_ptr(), wt_mix.data_ptr(), 0.2, mix.data_ptr(), None, 7 * 131,
                                          40, 48, _native.DTYPE_F16, math, stream))
        crush = torch.zeros(1, 3, 65, 40, device=dev)
        _native.check(lib.mz_pixel_crush(xp.data_ptr(), wt_crush.data_ptr(), crush.data_ptr(), None, 1, 7, 131, 40, 32, 2, 48,
                                         40, _native.DTYPE_F16, math, stream))
        outs.append((mix, crush))
    assert (outs[0][0] - outs[1][0]).abs().max().item() <= 3e-2 and (outs[0][1] - outs[1][1]).abs().max().item() <= 3e-2, "pitch"
    n += 2
    for r in (2, 3, 4):
        s = N.pixel_shuffle_nhwc(x[..., :3 * r * r].contiguous(), r)
        assert torch.equal(N.to_nchw(s), torch.nn.functional.pixel_shuffle(N.to_nchw(x[..., :3 * r * r].contiguous()), r)), ("shuffle", r)
        n += 1
    for size in ((7, 140), (12, 100)):
        assert torch.equal(N.to_nchw(N.crop_feature_maps(x, size)), U.crop_feature_maps(N.to_nchw(x), size)), ("crop", size)
        n += 1
    wq, bq = torch.randn(3, 48, 3, 3, generator=g) / 20.0, torch.randn(3, generator=g)
    q = N.quality_assessor(x, wq, bq)
    assert (q - U.quality_assessor(N.to_nchw(x), wq.to(dev), bq.to(dev))).abs().max().item() <= 1e-4, "quality"
    n += 1
    for name, shape in (("MewZoom-2X-Ctrl", (2, 3, 9, 140)), ("MewZoom-3X-Ctrl", (1, 3, 7, 131)), ("MewZoom-4X-Ctrl", (1, 3, 6, 260))):
        cfg = dict(MODEL_CONFIGS[name])
        cfg["num_encoder_layers"] = 2
        torch.manual_seed(1)
        for rs in ("float32",):
            m = MewZoom(**cfg, residual_stream=rs).to(dev).eval()
            x, c = torch.rand(shape, generator=g).to(dev), torch.rand(shape[0], 3, generator=g).to(dev)
            y = m.upscale(x, c)
            m._flags_extra = _native.FLAG_SIMT_CONV
            ys = m.upscale(x, c)
            assert (y - ys).abs().max().item() <= 2e-3, (name, rs)
            y8 = m.upscale((x * 255).to(torch.uint8), c)
            assert y8.dtype == torch.uint8
            n += 1
    torch.cuda.synchronize()
    print(f"sanitize_cases: {n} cases ok")


if __name__ == "__main__":
    main()
