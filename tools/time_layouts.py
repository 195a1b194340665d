"""Image element types and layouts: device step time, head kernel time and frame-stream wall time.

    python tools/time_layouts.py --out DIR [--rounds 5] [--iters 10]

Writes JSON lines to DIR/time_layouts.jsonl (and prints them):
  * "gpu": card name and power limit (nvidia-smi, read-only query), so the numbers below carry what they were measured on;
  * "bytes": image bytes per HR pixel of each element type (computed, not measured): 12 fp32, 6 uint16, 3 uint8;
  * "step": device time per upscale call (CUDA events around `iters` calls after a warm-up) at cfg2 (MewZoom-2X-Ctrl,
    batch 16, 960x540 -> 1920x1080) and cfg4a (MewZoom-4X-Ctrl, 960x540 -> 3840x2160), for the four input / output layout
    combinations, fp32, uint8 and uint16.  The variants alternate round by round; min, median and max over the rounds are
    given.  The images and the workspace (0.1 - 2 GB) exceed the 126 MB L2;
  * "head": the head kernel's mean time per call in each variant, from a separate torch.profiler run (with the stem's);
  * "stream": wall time per frame of 960x540 frames through upscale_host at 4X: interleaved pinned frames in and out as
    uint8, uint16 and fp32, and the planar route a caller with interleaved uint8 frames had before interleaved images:
    CPU transpose HWC -> CHW, planar call, CPU transpose of the HR frame CHW -> HWC.
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
from ultrazoom_b200 import MODEL_CONFIGS, MewZoom  # noqa: E402

CL, NCHW = torch.channels_last, torch.contiguous_format
CONFIGS = {"cfg2": ("MewZoom-2X-Ctrl", 16, 540, 960), "cfg4a": ("MewZoom-4X-Ctrl", 1, 540, 960)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"kind": "gpu", "nvidia_smi": q.stdout.strip().splitlines()[:1], "torch_name": torch.cuda.get_device_name(0)}


def _channels_last(t):
    """(uint16 tensors are re-laid out through an int16 view: torch's CUDA support of uint16 is partial)"""
    if t.dtype == torch.uint16:
        return t.view(torch.int16).contiguous(memory_format=CL).view(torch.uint16)
    return t.contiguous(memory_format=CL)


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.uint16 else t


def variants(x):
    x8 = (x * 255).to(torch.uint8)
    x16 = (x.cpu() * 65535).round().to(torch.uint16).to(x.device)
    out = {}
    for dt, xx in (("fp32", x), ("u8", x8), ("u16", x16)):
        for xin_name, xin in (("nchw", xx), ("nhwc", _channels_last(xx))):
            for fmt_name, fmt in (("nchw", NCHW), ("nhwc", CL)):
                out[f"{dt} {xin_name}->{fmt_name}"] = (xin, fmt)
    return out


def model_for(cfg_name, dev):
    name, B, H, W = CONFIGS[cfg_name]
    torch.manual_seed(0)
    m = MewZoom(**MODEL_CONFIGS[name]).to(dev).eval()
    g = torch.Generator().manual_seed(1)
    x = torch.rand(B, 3, H, W, generator=g).to(dev)
    c = torch.rand(B, 3, generator=g).to(dev)
    return m, x, c


def time_steps(cfg_name, dev, rounds, iters, emit):
    m, x, c = model_for(cfg_name, dev)
    vs = variants(x)
    ref = {}
    for k, (xin, fmt) in vs.items():                                  # warm-up; every variant equals planar bit for bit
        y = m.upscale(xin, c, memory_format=fmt)
        base = k.split()[0] + " nchw->nchw"
        if base in ref:
            assert torch.equal(_bits(y), _bits(ref[base])), k
        else:
            ref[base] = y
    del ref
    times = {k: [] for k in vs}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for k, (xin, fmt) in vs.items():
            m.upscale(xin, c, memory_format=fmt)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                m.upscale(xin, c, memory_format=fmt)
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / iters)
    for k, t in times.items():
        emit({"kind": "step", "cfg": cfg_name, "variant": k, "ms_min": min(t), "ms_median": statistics.median(t),
              "ms_max": max(t), "rounds": rounds, "iters": iters})
    return m, x, c, vs


def time_head(cfg_name, m, c, vs, emit, iters=5):
    from torch.profiler import ProfilerActivity, profile

    for k, (xin, fmt) in vs.items():
        m.upscale(xin, c, memory_format=fmt)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(iters):
                m.upscale(xin, c, memory_format=fmt)
            torch.cuda.synchronize()
        head = stem = 0.0
        for e in prof.key_averages():
            if "conv_tc_kernel<2," in e.key:
                head += e.device_time_total
            elif "stem_kernel" in e.key:
                stem += e.device_time_total
        emit({"kind": "head", "cfg": cfg_name, "variant": k, "head_us": head / iters, "stem_us": stem / iters})


def time_stream(dev, frames, emit):
    torch.manual_seed(0)
    m = MewZoom(**MODEL_CONFIGS["MewZoom-4X-Ctrl"]).to(dev).eval()
    r = m.upscale_ratio
    H, W = 540, 960
    g = torch.Generator().manual_seed(2)
    base = [torch.rand(1, H, W, 3, generator=g) for _ in range(2)]
    hwc = {"uint8": [(b * 255).to(torch.uint8).pin_memory() for b in base],
           "uint16": [(b * 65535).round().to(torch.uint16).pin_memory() for b in base],
           "float32": [b.pin_memory() for b in base]}
    c = torch.rand(1, 3, generator=g)
    out_hwc = {k: torch.empty(1, H * r, W * r, 3, dtype=v[0].dtype).pin_memory() for k, v in hwc.items()}
    out_planar = torch.empty(1, 3, H * r, W * r, dtype=torch.uint8).pin_memory()
    x_planar = torch.empty(1, 3, H, W, dtype=torch.uint8).pin_memory()

    def interleaved(dt):
        def route(i):
            m.upscale_host(hwc[dt][i % 2].permute(0, 3, 1, 2), c, out=out_hwc[dt].permute(0, 3, 1, 2))
            return out_hwc[dt]
        return route

    def planar_route(i):
        x_planar.copy_(hwc["uint8"][i % 2].permute(0, 3, 1, 2))       # CPU transpose HWC -> CHW
        m.upscale_host(x_planar, c, out=out_planar)
        return out_planar.permute(0, 2, 3, 1).contiguous()            # CPU transpose CHW -> HWC of the HR frame

    assert torch.equal(interleaved("uint8")(0), planar_route(0))
    routes = [("uint8 interleaved", "uint8", interleaved("uint8")), ("uint8 planar+transposes", "uint8", planar_route),
              ("uint16 interleaved", "uint16", interleaved("uint16")), ("float32 interleaved", "float32", interleaved("float32"))]
    res = {}
    for _ in range(3):                                                # alternate the routes
        for name, _, fn in routes:
            fn(0)
            t0 = time.perf_counter()
            for i in range(frames):
                fn(i)
            res.setdefault(name, []).append((time.perf_counter() - t0) / frames * 1e3)
    for name, dt, _ in routes:
        t = res[name]
        emit({"kind": "stream", "route": name, "frame": f"1x960x540 {dt} -> 4X", "ms_per_frame_min": min(t),
              "ms_per_frame_median": statistics.median(t), "frames": frames, "cpu_threads": torch.get_num_threads()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--frames", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_layouts.py measures on the GPU; there is no CPU fallback"
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    path = os.path.join(args.out, "time_layouts.jsonl")
    with open(path, "w") as f:
        def emit(rec):
            line = json.dumps(rec)
            print(line, flush=True)
            f.write(line + "\n")
            f.flush()

        emit(gpu_info())
        emit({"kind": "bytes", "per_hr_pixel": {dt: 3 * torch.empty((), dtype=d).element_size()
                                                for dt, d in (("fp32", torch.float32), ("u16", torch.uint16),
                                                              ("u8", torch.uint8))}})
        for cfg_name in CONFIGS:
            m, x, c, vs = time_steps(cfg_name, dev, args.rounds, args.iters, emit)
            time_head(cfg_name, m, c, vs, emit)
            del m, x, c, vs
            torch.cuda.empty_cache()
        time_stream(dev, args.frames, emit)


if __name__ == "__main__":
    main()
