"""RGBA images (MZ_FLAG_RGBA): step time against RGB, and frames per second end to end against the manual route.

    python tools/time_rgba.py --out DIR [--rounds 5] [--iters 10] [--frames 20]

Writes JSON lines to DIR/time_rgba.jsonl (and prints them):
  * "gpu": card name, power limit and max SM clock (nvidia-smi, read-only query), taken in this run;
  * "step": device time per upscale call (CUDA events over `iters` calls), interleaved uint8 RGBA in and out against
    interleaved uint8 RGB, at cfg2 (16 x 960x540 -> 1080p, 2X-Ctrl) and cfg4a (960x540 -> 4K, 4X-Ctrl); the variants
    alternate round by round (min / median / max over the rounds);
  * "stream": frames per second through upscale_host with pinned interleaved uint8 RGBA frames in and out (synchronous,
    and alternating the two lanes), against what a caller does without the flag: copy the RGBA frame to the GPU, the
    RGB call on x[:, :3], ops.bicubic of the alpha, quantise and interleave with torch ops, copy the result back.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ultrazoom_b200 import MODEL_CONFIGS, MewZoom, ops  # noqa: E402

CONFIGS = {"cfg2": ("MewZoom-2X-Ctrl", 16, 540, 960), "cfg4a": ("MewZoom-4X-Ctrl", 1, 540, 960)}
CL = torch.channels_last


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


def model_for(cfg, dev):
    name, B, H, W = CONFIGS[cfg]
    torch.manual_seed(0)
    m = MewZoom(**MODEL_CONFIGS[name]).to(dev).eval()
    g = torch.Generator().manual_seed(1)
    rgba = (torch.rand(B, H, W, 4, generator=g) * 255).to(torch.uint8)      # (B,H,W,4) HWC frames
    c = torch.rand(B, 3, generator=g).to(dev)
    return m, rgba, c


def time_steps(cfg, dev, rounds, iters, emit):
    m, rgba, c = model_for(cfg, dev)
    x4 = rgba.to(dev).permute(0, 3, 1, 2)                                 # interleaved (channels-last strides)
    x3 = rgba[..., :3].contiguous().to(dev).permute(0, 3, 1, 2)
    variants = {"rgba u8 interleaved": x4, "rgb u8 interleaved": x3}
    times = {k: [] for k in variants}
    for _ in range(rounds):
        for k, x in variants.items():
            times[k].append(_events_ms(lambda i: m.upscale(x, c, memory_format=CL), iters))
    for k, t in times.items():
        emit({"kind": "step", "cfg": cfg, "variant": k, "ms_min": min(t), "ms_median": statistics.median(t),
              "ms_max": max(t), "rounds": rounds, "iters": iters})


def time_stream(cfg, dev, frames, emit):
    m, rgba, c = model_for(cfg, dev)
    _, B, H, W = CONFIGS[cfg]
    r = m.upscale_ratio
    xs = [rgba.roll(i, dims=2).pin_memory().permute(0, 3, 1, 2) for i in range(2)]
    outs = [torch.empty(B, H * r, W * r, 4, dtype=torch.uint8).pin_memory().permute(0, 3, 1, 2) for _ in range(2)]
    ch = c.cpu()

    def sync_route(i):
        m.upscale_host(xs[i % 2], ch, out=outs[i % 2])

    def lanes_route(i):
        if i >= 2:
            m.host_wait(i % 2)
        m.upscale_host(xs[i % 2], ch, out=outs[i % 2], lane=i % 2)

    def manual(i):
        x = xs[i % 2].to(dev, non_blocking=True)
        colour = m.upscale(x[:, :3], c, memory_format=CL)
        alpha = ops.bicubic(x[:, 3:].float() / 255, r).clamp_(0, 1).mul_(255).add_(0.5).floor_().to(torch.uint8)
        y = torch.cat([colour, alpha], dim=1).contiguous(memory_format=CL)
        outs[i % 2].copy_(y, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()

    routes = [("upscale_host RGBA, synchronous", sync_route), ("upscale_host RGBA, two lanes", lanes_route),
              ("RGBA -> GPU, RGB upscale + ops.bicubic alpha + torch interleave -> host", manual)]
    res = {}
    for _ in range(3):                                                # alternate the routes
        for rname, fn in routes:
            fn(0)
            m.host_wait()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(frames):
                fn(i)
            m.host_wait()
            torch.cuda.synchronize()
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
    ap.add_argument("--frames", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_rgba.py measures on the GPU; there is no CPU fallback"
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    with open(os.path.join(args.out, "time_rgba.jsonl"), "w") as fh:
        def emit(rec):
            line = json.dumps(rec)
            print(line, flush=True)
            fh.write(line + "\n")
            fh.flush()

        emit(gpu_info())
        for cfg in CONFIGS:
            time_steps(cfg, dev, args.rounds, args.iters, emit)
            torch.cuda.empty_cache()
        for cfg in CONFIGS:
            time_stream(cfg, dev, args.frames, emit)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
