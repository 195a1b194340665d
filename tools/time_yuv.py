"""4:2:0 frames (MZ_FLAG_YUV420): conversion kernel times, step time against planar RGB, and frames per second end to end.

    python tools/time_yuv.py --out DIR [--rounds 5] [--iters 10] [--frames 20]

Writes JSON lines to DIR/time_yuv.jsonl (and prints them):
  * "gpu": card name, power limit and max SM clock (nvidia-smi, read-only query);
  * "copy": device-to-device copy bandwidth of a 1 GiB buffer in this run (read + write bytes over CUDA-event time), the
    peak the kernels are set against;
  * "kernel": decode (mz_yuv420_to_rgb16) at the LR size and encode (mz_rgb16_to_yuv420) at the HR size of cfg2
    (16 x 960x540 -> 1080p) and cfg4a (960x540 -> 4K), NV12 and P010: CUDA events around `launches` launches that rotate
    through enough input / output pairs to cover 3x the 126 MB L2, so every launch reads and writes HBM.  Algorithmic
    bytes: decode 1.5 es + 6 B per LR pixel, encode 6 + 1.5 es B per HR pixel (es = 1 NV12, 2 P010);
  * "step": device time per upscale call, NV12 against planar uint8 RGB and P010 against planar uint16 RGB, variants
    alternating round by round (min / median / max over the rounds);
  * "stream": frames per second through upscale_host with pinned NV12 frames in and out (synchronous, and alternating the
    two lanes), against what a video caller does without MZ_FLAG_YUV420: copy the NV12 frame to the GPU, convert it to
    rgb24 with torch ops, the interleaved uint8 upscale, convert back with torch ops and copy the NV12 frame back.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ultrazoom_b200 import MODEL_CONFIGS, MewZoom, Yuv420, _native  # noqa: E402

CONFIGS = {"cfg2": ("MewZoom-2X-Ctrl", 16, 540, 960), "cfg4a": ("MewZoom-4X-Ctrl", 1, 540, 960)}
L2_BYTES = 126 << 20


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"kind": "gpu", "nvidia_smi": q.stdout.strip().splitlines()[:1], "torch_name": torch.cuda.get_device_name(0)}


def _events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn(0)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def copy_peak(dev, emit):
    a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    ms = min(_events_ms(lambda i: b.copy_(a), 20) for _ in range(3))
    gbs = 2 * a.numel() / ms / 1e6
    emit({"kind": "copy", "bytes": 2 * a.numel(), "ms": ms, "GB_per_s": gbs})
    return gbs


def time_kernels(dev, peak, launches, emit):
    lib = _native.load()
    stream = torch.cuda.current_stream(dev).cuda_stream
    for cfg, (name, B, H, W) in CONFIGS.items():
        r = MODEL_CONFIGS[name]["upscale_ratio"]
        for dt in (torch.uint8, torch.uint16):
            es = 1 if dt == torch.uint8 else 2
            flags = Yuv420().flags(dt)
            for what, h, w in (("decode", H, W), ("encode", H * r, W * r)):
                npx = B * h * w
                frame, rgb = npx * 3 // 2 * es, npx * 6
                pairs = min(128, math.ceil(3 * L2_BYTES / (frame + rgb)))
                yuv = [torch.zeros(frame, dtype=torch.uint8, device=dev) for _ in range(pairs)]
                img = [torch.zeros(npx * 3, dtype=torch.int16, device=dev) for _ in range(pairs)]
                if what == "decode":
                    fn = lambda i: lib.mz_yuv420_to_rgb16(yuv[i % pairs].data_ptr(), img[i % pairs].data_ptr(),  # noqa: E731
                                                          B, h, w, flags, stream)
                else:
                    fn = lambda i: lib.mz_rgb16_to_yuv420(img[i % pairs].data_ptr(), yuv[i % pairs].data_ptr(),  # noqa: E731
                                                          B, h, w, flags, stream)
                ms = [_events_ms(fn, launches) for _ in range(3)]
                us = statistics.median(ms) * 1e3
                nbytes = frame + rgb
                gbs = nbytes / us / 1e3
                emit({"kind": "kernel", "cfg": cfg, "format": "NV12" if es == 1 else "P010", "kernel": what,
                      "shape": [B, h, w], "us_median": us, "us_min": min(ms) * 1e3, "algorithmic_bytes": nbytes,
                      "GB_per_s": gbs, "fraction_of_copy": gbs / peak, "buffer_pairs": pairs,
                      "rotated_bytes": pairs * nbytes, "launches": launches})
                del yuv, img
                torch.cuda.empty_cache()


def model_for(cfg, dev):
    name, B, H, W = CONFIGS[cfg]
    torch.manual_seed(0)
    m = MewZoom(**MODEL_CONFIGS[name]).to(dev).eval()
    g = torch.Generator().manual_seed(1)
    rgb = torch.rand(B, 3, H, W, generator=g)
    c = torch.rand(B, 3, generator=g).to(dev)
    return m, rgb, c


def _frames(B, H, W, dt, seed):
    g = torch.Generator().manual_seed(seed)
    mx = 256 if dt == torch.uint8 else 1024
    f = torch.randint(16, mx - 16, (B, H * 3 // 2, W), generator=g, dtype=torch.int32)
    return (f if dt == torch.uint8 else f << 6).to(dt)


def time_steps(cfg, dev, rounds, iters, emit):
    m, rgb, c = model_for(cfg, dev)
    B, _, H, W = rgb.shape
    f = Yuv420()
    variants = {
        "NV12": (_frames(B, H, W, torch.uint8, 2).to(dev), f),
        "rgb u8 planar": ((rgb * 255).to(torch.uint8).to(dev), None),
        "P010": (_frames(B, H, W, torch.uint16, 3).to(dev), f),
        "rgb u16 planar": ((rgb * 65535).round().to(torch.uint16).to(dev), None),
    }
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, (x, yuv) in variants.items():
            times[k].append(_events_ms(lambda i: m.upscale(x, c, yuv=yuv), iters))
    for k, t in times.items():
        emit({"kind": "step", "cfg": cfg, "variant": k, "ms_min": min(t), "ms_median": statistics.median(t),
              "ms_max": max(t), "rounds": rounds, "iters": iters})


def _torch_nv12_to_rgb(f, H, W):
    """BT.709 limited-range NV12 (B, 3H/2, W) on the GPU -> rgb24 (B, 3, H, W) uint8 in channels-last strides."""
    B = f.shape[0]
    y = (f[:, :H].float() - 16) / 219
    uv = f[:, H:].reshape(B, H // 2, W // 2, 2).permute(0, 3, 1, 2).float()
    uv = (F.interpolate(uv, scale_factor=2, mode="bilinear", align_corners=False) - 128) / 224
    cb, cr = uv[:, 0], uv[:, 1]
    kr, kb = 0.2126, 0.0722
    r = y + 2 * (1 - kr) * cr
    b = y + 2 * (1 - kb) * cb
    g = (y - kr * r - kb * b) / (1 - kr - kb)
    rgb = torch.stack([r, g, b], dim=-1).clamp_(0, 1).mul_(255).round_().to(torch.uint8)
    return rgb.permute(0, 3, 1, 2)


def _torch_rgb_to_nv12(rgb):
    """rgb24 (B, 3, H, W) uint8 on the GPU -> BT.709 limited-range NV12 (B, 3H/2, W)."""
    B, _, H, W = rgb.shape
    v = rgb.float() / 255
    kr, kb = 0.2126, 0.0722
    y = kr * v[:, 0] + (1 - kr - kb) * v[:, 1] + kb * v[:, 2]
    cb = F.avg_pool2d(((v[:, 2] - y) / (2 * (1 - kb))).unsqueeze(1), 2)
    cr = F.avg_pool2d(((v[:, 0] - y) / (2 * (1 - kr))).unsqueeze(1), 2)
    luma = (16 + 219 * y).round_().clamp_(0, 255)
    uv = (128 + 224 * torch.cat([cb, cr], dim=1)).round_().clamp_(0, 255).permute(0, 2, 3, 1).reshape(B, H // 2, W)
    return torch.cat([luma, uv], dim=1).to(torch.uint8)


def time_stream(cfg, dev, frames, emit):
    m, _, c = model_for(cfg, dev)
    name, B, H, W = CONFIGS[cfg]
    r = m.upscale_ratio
    f = Yuv420()
    xs = [_frames(B, H, W, torch.uint8, 5 + i).pin_memory() for i in range(2)]
    outs = [torch.empty(B, H * r * 3 // 2, W * r, dtype=torch.uint8).pin_memory() for _ in range(2)]
    ch = c.cpu()

    def sync_route(i):
        m.upscale_host(xs[i % 2], ch, out=outs[i % 2], yuv=f)

    def lanes_route(i):
        if i >= 2:
            m.host_wait(i % 2)
        m.upscale_host(xs[i % 2], ch, out=outs[i % 2], lane=i % 2, yuv=f)

    def status_quo(i):
        x = xs[i % 2].to(dev, non_blocking=True)
        y = m.upscale(_torch_nv12_to_rgb(x, H, W), c, memory_format=torch.channels_last)
        outs[i % 2].copy_(_torch_rgb_to_nv12(y), non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()

    routes = [("upscale_host NV12, synchronous", sync_route), ("upscale_host NV12, two lanes", lanes_route),
              ("NV12 -> torch ops -> rgb24 upscale -> torch ops -> NV12", status_quo)]
    res = {}
    for _ in range(3):                                                # alternate the routes
        for rname, fn in routes:
            fn(0)
            m.host_wait()
            t0 = time.perf_counter()
            for i in range(frames):
                fn(i)
            m.host_wait()
            res.setdefault(rname, []).append(frames * B / (time.perf_counter() - t0))
    for rname, _ in routes:
        t = res[rname]
        emit({"kind": "stream", "cfg": cfg, "route": rname, "batch": [B, H, W], "frames_per_s_median": statistics.median(t),
              "frames_per_s_max": max(t), "calls": frames})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--frames", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_yuv.py measures on the GPU; there is no CPU fallback"
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    with open(os.path.join(args.out, "time_yuv.jsonl"), "w") as fh:
        def emit(rec):
            line = json.dumps(rec)
            print(line, flush=True)
            fh.write(line + "\n")
            fh.flush()

        emit(gpu_info())
        peak = copy_peak(dev, emit)
        time_kernels(dev, peak, args.launches, emit)
        for cfg in CONFIGS:
            time_steps(cfg, dev, args.rounds, args.iters, emit)
            torch.cuda.empty_cache()
        for cfg in CONFIGS:
            time_stream(cfg, dev, args.frames, emit)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
