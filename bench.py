#!/usr/bin/env python
"""bench.py -- output Mpx/s of MewZoom.upscale on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg3|cfg4a|cfg4b|cfg4c|cfg5] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path (FiLM table, stem, 2L fused 3x3 convolutions, head) over one batch of
synthetic frames.  Default workload = BASELINE.json configs[1]: MewZoom-2X-Ctrl (48 ch / 20 layers), batch 16 of
960x540 -> 1920x1080.  With N > 1 (torchrun, one rank per GPU) every rank processes its own batch (weak scaling,
no data-path collective); time = max over ranks, value = all ranks' output pixels / time.
`--workload cfg5` (BASELINE configs[4]) is the STRONG-scaling case: ONE 1920x1080 -> 7680x4320 MewZoom-4X-Ctrl frame cut
into N halo-padded tiles, one per rank, each rank's head kernel storing its core straight into the frame on rank 0's GPU
(CUDA IPC mapping, NVLink); value = 33.2 Mpx / max-over-ranks time.  The default (cfg2) line carries it -- and the
4X-Ctrl / 3X-Ctrl frames -- under "also", so that the driver's 1 -> 8 GPU runs record the spatial split as well.

Prints ONE JSON line (rank 0).  `--impl reference` times the reference's CPU implementation of the path: the
reference is pure PyTorch, its 0.2.x model class is absent from the snapshot, so this is the oracle restatement
(oracle/mewzoom_oracle.py, built on the same torch ops) on all host cores -- kind "port".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (model, B, H, W, description)
    "cfg2": ("MewZoom-2X-Ctrl", 16, 540, 960, "MewZoom-2X-Ctrl 48ch/20L, batch 16, 960x540->1920x1080 (BASELINE configs[1])"),
    "cfg3": ("MewZoom-3X-Ctrl", 1, 720, 1280, "MewZoom-3X-Ctrl 54ch/30L, 1 frame 1280x720->3840x2160 (BASELINE configs[2] frame)"),
    "cfg4a": ("MewZoom-4X-Ctrl", 1, 540, 960, "MewZoom-4X-Ctrl 96ch/40L, 1 frame 960x540->3840x2160 (BASELINE configs[3], 4K output)"),
    "cfg4b": ("MewZoom-4X-Ctrl", 1, 1080, 1920, "MewZoom-4X-Ctrl 96ch/40L, 1 frame 1920x1080->7680x4320 (BASELINE configs[3], 1080p input)"),
    "cfg4c": ("MewZoom-2X-Ctrl", 1, 1080, 1920, "MewZoom-2X-Ctrl 48ch/20L, 1 frame 1920x1080->3840x2160 (literal 1080p->4K)"),
    "cfg5": ("MewZoom-4X-Ctrl", 1, 1080, 1920, "MewZoom-4X-Ctrl 96ch/40L, ONE 1920x1080->7680x4320 frame halo-tiled across the GPUs (BASELINE configs[4])"),
    "tiny": ("MewZoom-2X-Ctrl", 1, 64, 128, "MewZoom-2X-Ctrl 48ch/20L, 1 frame 128x64 (debug)"),
}


def operands_for(workload: str, args) -> str:
    """Tensor-core operand type of a workload.  `--operands auto` (default): bf16 -- the type BASELINE configs[1] and the
    north_star name -- for the 20-layer 2X model, where it meets BASELINE's envelope at full size (max-abs 0.015, PSNR
    55 dB vs <= 2e-2 / >= 45 dB: tests/test_gpu_fullsize.py) and runs 5 % faster than fp16 under the power cap (same
    tcgen05 rate and bytes, lower multiplier power: DESIGN.md section 7); fp16 for the 30- / 40-layer models, where bf16
    does not meet the envelope (0.018 / 0.026).  The same rule in both arms, so their `config` objects agree."""
    if args.operands != "auto":
        return args.operands
    return "bfloat16" if WORKLOADS[workload][0].startswith("MewZoom-2X") else "float16"


def config_of(workload: str, world: int, args, operands=None) -> dict:
    """The `config` object of the JSON line -- the same keys and values in both arms (`--impl reference` times the
    CPU path on THIS configuration), so that the driver can tell the two lines describe one workload."""
    model_name, B, H, W, desc = WORKLOADS[workload]
    tiled = workload == "cfg5"
    return {"workload": desc, "batch_per_gpu": B, "lr_h": H, "lr_w": W,
            "parallelism": (f"one halo-padded tile per GPU x{world} (halo 2L+1 = 81 LR px), cores stored into rank 0's "
                            "frame over NVLink, no collective") if tiled else
                           f"replica per GPU x{world}, batch-sharded, no collective",
            "l2": "activations per step (>= 1 GB) exceed the 126 MB L2; no explicit flush",
            "weights": "random init (seed 0)", "image_io": args.io,
            "residual_stream": "fp32",
            "accumulate": "fp32", "mma_operands": operands or operands_for(workload, args),
            "tune": {k: int(v) for k, v in (kv.split("=") for kv in args.tune.split(",") if kv)}}


def algorithmic_flops_per_lr_px(cfg) -> float:
    """2*MACs, unpadded, elementwise excluded (SURVEY.md 8(d)): 2*[3C + L*36C^2 + 27*C*r^2] for h = 2."""
    C, L, r, h = cfg["num_channels"], cfg["num_encoder_layers"], cfg["upscale_ratio"], cfg["hidden_ratio"]
    return 2.0 * (3 * C + L * 18 * h * C * C + 27 * C * r * r)


def conv_flops_per_launch(cfg, npix: int) -> float:
    """One encoder convolution launch: 2 * 9 * C * hC MACs-as-flops per LR pixel (conv1 and conv2 are equal)."""
    C, h = cfg["num_channels"], cfg["hidden_ratio"]
    return 2.0 * 9 * C * (h * C) * npix


class ClockSampler:
    """nvidia-smi clocks / throttle reasons every 100 ms.  The process is started BEFORE the warm-up steps (nvidia-smi
    needs a few hundred ms to deliver its first line -- longer than a short timed region) and the samples whose own
    timestamps fall inside the timed region (mark_begin() .. stop()) are the ones reported."""

    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []
        self.thread = None
        self.t_begin = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def mark_begin(self):
        self.t_begin = time.time()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.time()
        time.sleep(0.15)   # (a line stamped inside the region may still be on its way)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        import datetime
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = []
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(parts[1]), float(parts[2]), float(parts[3]),
                             [n for n, v in zip(names, parts[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        inside = [r for r in rows if self.t_begin is not None and self.t_begin <= r[0] <= t_end]
        window = "timed region"
        if not inside:   # (clock skew between nvidia-smi's stamps and this process, or a very short region)
            inside, window = rows[-3:], "last samples before the end of the timed region"
        sm = sorted(r[1] for r in inside)
        reasons = sorted({n for r in inside for n in r[4]})
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[2] for r in inside), "power_w_max": max(r[3] for r in inside),
                "samples": len(inside), "samples_since_warmup": len(rows), "window": window, "reasons": reasons}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_burst": p["bf16_tflops"], "bf16_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "hbm": p["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def cpu_port_sample(model_name: str, H: int, W: int, threads: int):
    """Time the oracle (CPU restatement of the reference path) on ONE frame of the workload's shape."""
    import torch

    from oracle import MODEL_CONFIGS, make_oracle

    torch.set_num_threads(threads)
    cfg = MODEL_CONFIGS[model_name]
    o = make_oracle(model_name, seed=0)
    r = cfg["upscale_ratio"]
    g = torch.Generator().manual_seed(1234)
    c = torch.tensor([[0.5, 0.2, 0.3]]) if cfg["control_features"] else None
    o.upscale(torch.rand(1, 3, 32, 32, generator=g), c)  # thread-pool / oneDNN warm-up
    x = torch.rand(1, 3, H, W, generator=g)
    t0 = time.perf_counter()
    o.upscale(x, c)
    dt = time.perf_counter() - t0
    return (H * r * W * r) / dt / 1e6, dt


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on the host cores, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model_name, B, H, W, desc = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    # bounded sample: one frame per step, capped in size so K + W steps stay within minutes
    sh, sw = H, W
    while sh * sw > 540 * 960:
        sh, sw = sh // 2, sw // 2
    vals, times = [], []
    for i in range(args.warmup + args.steps):
        mpx, dt = cpu_port_sample(model_name, sh, sw, threads)
        if i >= args.warmup:
            vals.append(mpx)
            times.append(dt)
    value = sum(vals) / len(vals)
    sample = f"1 frame {sw}x{sh} of the workload per step, fp32, torch {threads} threads"
    line = {
        "impl": "reference", "metric": "output_mpx_per_s", "value": value, "unit": "Mpx/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "strong" if args.workload == "cfg5" else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, args.gpus, args),
        "cpu_baseline": {"value": value, "unit": "Mpx/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


DUMP_MAX_ELEMENTS = 4 << 20   # float32 values + float64 indices of a sampled output: 48 MB, under 64 MB


def dump_output(out_dir: str, name: str, y) -> None:
    """--dump-outputs: write `y`, what the timed path returned in its last step, as out_dir/<name>.npy in float32 (an
    8-bit image as its values 0..255).  An output of more than DUMP_MAX_ELEMENTS elements is sampled: the flattened
    output is cut into DUMP_MAX_ELEMENTS equal blocks and one element of each is taken at an offset drawn from a fixed
    seed, its flat indices in out_dir/<name>_index.npy (float64, exact).  The same arguments give the same inputs,
    indices and files, so two builds compare element for element."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, name + ".npy")
    y = y.detach()
    if y.numel() <= DUMP_MAX_ELEMENTS:
        np.save(path, y.float().cpu().numpy())
        print(f"bench: wrote {path}, the whole output {tuple(y.shape)}", file=sys.stderr)
        return
    edges = torch.arange(DUMP_MAX_ELEMENTS + 1, dtype=torch.int64) * y.numel() // DUMP_MAX_ELEMENTS
    u = torch.rand(DUMP_MAX_ELEMENTS, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    idx = edges[:-1] + (u * (edges[1:] - edges[:-1])).long()
    np.save(path, y.reshape(-1)[idx.to(y.device)].float().cpu().numpy())
    np.save(os.path.join(out_dir, name + "_index.npy"), idx.double().numpy())
    print(f"bench: wrote {path}, {DUMP_MAX_ELEMENTS} sampled elements of the output {tuple(y.shape)}", file=sys.stderr)


_REAL_STDOUT = None


def _quiet_stdout():
    """Everything but the one JSON line goes to stderr: libraries (NCCL's version banner with NCCL_DEBUG set, torch
    warnings) write to file descriptor 1 behind Python's back."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--operands", default="auto", choices=["auto", "float16", "bfloat16"],
                    help="tensor-core operand type; auto = bf16 for the 20-layer 2X model, fp16 for the deeper ones (operands_for)")
    ap.add_argument("--residual-stream", default="auto", choices=["auto", "float32"])
    ap.add_argument("--tune", default="", help="comma list k=v of mz_conv_tune fields, e.g. cluster=4,rows=1")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--io", default="float32", choices=["float32", "uint8"],
                    help="image element type at the API (uint8: x = x8/255 in, floor(255 y + 0.5) out); the headline is float32")
    ap.add_argument("--e2e-sync", action="store_true", help="time the synchronous host call instead of the two-lane stream")
    ap.add_argument("--halo-refresh", type=int, default=-1,
                    help="cfg5: refresh the tiles' halo every K encoder blocks (halo 2K+1 instead of 2L+1 pixels, strips "
                         "exchanged between neighbour GPUs); 0 = full halo, no exchange; -1 = the default (see measure_tiled)")
    ap.add_argument("--unet-ops", action="store_true", help="add the U-Net operator microbenchmarks to the line (default with cfg2 at N = 1)")
    ap.add_argument("--no-also", action="store_true",
                    help="skip the secondary records (4X-Ctrl frame, 3X-Ctrl frame, halo-tiled 8K frame)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the output of the workload's last step (rank 0) to DIR/upscale.npy "
                         "(float32; a fixed sample of a larger output, its indices in DIR/upscale_index.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: at least three warm-up steps
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from ultrazoom_b200 import MODEL_CONFIGS, MewZoom, _native

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert torch.cuda.is_available(), "bench.py needs a B200 (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from ultrazoom_b200.sharding import bind_process_to_gpu
    # One process per GPU: node-local pinned buffers for the end-to-end leg.  Not at N = 1: the CPU baseline of that line
    # uses every host core, and threads started under a narrowed affinity would keep it.
    cpus = bind_process_to_gpu(local_rank) if world > 1 and not os.environ.get("MZ_NO_BIND") else None

    import ctypes as C

    tune_kw = {k: int(v) for k, v in (kv.split("=") for kv in args.tune.split(",") if kv)}

    def apply_tune(model):
        """--tune k=v,...: plain keys apply to every convolution; c1.k / c2.k / head.k to conv1 / conv2 / the head only."""
        if not tune_kw:
            return
        per = {-1: {}, 0: {}, 1: {}, 2: {}}
        for k, v in tune_kw.items():
            which, _, name = k.rpartition(".")
            per[{"": -1, "c1": 0, "c2": 1, "head": 2}[which]][name] = v
        for which in (0, 1, 2):
            kw = {**per[-1], **per[which]}
            if kw:
                model.set_conv_tune(which, dev, **kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(workload: str, steps: int, warmup: int, want_e2e: bool, sample_clocks: bool, operands=None, dump=False):
        """W untimed + exactly K timed steps (CUDA events on the launching stream, barrier + synchronize on both
        sides, max over ranks) of one workload; optionally the end-to-end leg with host buffers.  `dump`: write the
        last timed step's output to --dump-outputs."""
        if workload == "cfg5":
            return measure_tiled(steps, warmup, want_e2e, sample_clocks, dump)
        model_name, B, H, W, desc = WORKLOADS[workload]
        cfg = MODEL_CONFIGS[model_name]
        r = cfg["upscale_ratio"]
        torch.manual_seed(0)
        operands = operands or operands_for(workload, args)
        model = MewZoom(**cfg, operand_dtype=operands, residual_stream=args.residual_stream).to(dev).eval()
        apply_tune(model)
        eng = model._engine(dev)
        g = torch.Generator().manual_seed(1234 + rank)
        x_host = torch.rand(B, 3, H, W, generator=g)
        if args.io == "uint8":
            x_host = (x_host * 255.0).round().to(torch.uint8)
        x_host = x_host.pin_memory()
        io_dt = x_host.dtype
        c_host = torch.tensor([[0.5, 0.2, 0.3]]).pin_memory() if cfg["control_features"] else None
        x = x_host.to(dev)
        c = c_host.to(dev) if c_host is not None else None
        out_px = B * H * r * W * r
        sampler = ClockSampler(local_rank)
        if rank == 0 and sample_clocks:
            sampler.start()
        for _ in range(warmup):
            model.upscale(x, c)
        barrier()
        _native.check(eng.lib.mz_model_enable_timing(eng.handle, 1))
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.mark_begin()
        ev0.record()
        for _ in range(steps - 1):
            model.upscale(x, c)
        y = model.upscale(x, c)                             # the last step's output, for --dump-outputs
        ev1.record()
        barrier()
        ms_total = ev0.elapsed_time(ev1)
        clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
        if dump and rank == 0:
            dump_output(args.dump_outputs, "upscale", y)
        del y
        conv_ms = C.c_float()
        _native.check(eng.lib.mz_model_conv_stack_ms(eng.handle, C.byref(conv_ms)))
        _native.check(eng.lib.mz_model_enable_timing(eng.handle, 0))
        assert not model.saturated(dev), "fp16 operand saturation during the timed region"
        fused = bool(eng.lib.mz_model_fused_block(eng.handle))
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item()) / steps
        res = {"workload": workload, "operands": operands, "model_name": model_name, "cfg": cfg, "B": B, "H": H, "W": W, "desc": desc, "ms_step": ms_step,
               "conv_ms": conv_ms.value, "clocks": clocks, "value": world * out_px / (ms_step * 1e-3) / 1e6,
               "e2e": None, "scaling": "weak", "steps": steps, "fused": fused}
        # ---- end to end through the public API with HOST buffers (H2D + kernels + D2H inside the timed region) ----
        def run_e2e(xh):
            # Every step copies its inputs from pinned host memory and its result back to pinned host memory.  The
            # workload is a STREAM of steps (frames or batches): steps alternate between the two lanes of the async
            # form (submit step i, then wait for step i-2 on the same lane), each lane with its own pinned input /
            # output buffers, so the copies of step i+1 / i-1 run under the kernels of step i.
            # (--e2e-sync times the synchronous call instead, which pipelines chunks of one batch internally.)
            outs = [torch.empty((B, 3, H * r, W * r), dtype=xh.dtype).pin_memory() for _ in range(2)]
            xs = [xh, xh.clone().pin_memory()]
            stream_mode = not args.e2e_sync

            def e2e_steps(n):
                if not stream_mode:
                    for _ in range(n):
                        model.upscale_host(xh, c_host, out=outs[0], device=local_rank)
                    return
                for i in range(n):
                    ln = i & 1
                    if i >= 2:
                        model.host_wait(ln, device=local_rank)      # frame i-2 (same lane) has left its buffers
                    model.upscale_host(xs[ln], c_host, out=outs[ln], device=local_rank, lane=ln)
                model.host_wait(-1, device=local_rank)

            e2e_steps(2)
            barrier()
            t0 = time.perf_counter()
            e2e_steps(steps)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            out_host = outs[0]
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
            return {"value": world * out_px * steps / dt / 1e6, "unit": "Mpx/s",
                    "h2d_bytes_per_step": xh.numel() * xh.element_size() + (c_host.numel() * 4 if c_host is not None else 0),
                    "d2h_bytes_per_step": out_host.numel() * out_host.element_size(), "ms_per_step": 1e3 * dt / steps,
                    "image_io": "uint8" if xh.dtype == torch.uint8 else "float32",
                    "host_binding": (f"rank bound to the {len(cpus)} CPUs next to its GPU (NVML ideal-CPU set)" if cpus
                                     else "none"),
                    "api": ("MewZoom.upscale_host(lane=i%2) + host_wait -> mz_upscale_host_async (stream of steps, two "
                            "lanes, pinned host buffers)") if stream_mode else
                           "MewZoom.upscale_host -> mz_upscale_host (pinned host buffers, batch pipelined in chunks)"}

        if want_e2e:
            res["e2e"] = run_e2e(x_host)
            if x_host.dtype != torch.uint8:
                # The same stream with 8-bit images in and out (the reference's own callers read and write 8-bit images:
                # test_compare.py:53-57,89): a quarter of the host traffic.  Not the headline -- eight ranks moving fp32
                # images through one host are bound by the host, and this record shows by how much.
                res["e2e_uint8"] = run_e2e((x_host * 255.0).round().to(torch.uint8).pin_memory())
        del model, eng, x, c
        torch.cuda.empty_cache()
        return res

    def measure_tiled(steps: int, warmup: int, want_e2e: bool, sample_clocks: bool, dump=False):
        """cfg5 (BASELINE configs[4]), strong scaling: ONE 1080p -> 8K MewZoom-4X-Ctrl frame, `world` halo-padded tiles
        (sharding.best_grid / plan_tiles, columns sized for the kernel's 128-pixel tiles), one per rank.  Every rank
        runs the whole network on its tile and its head kernel stores the tile's core straight into the frame that
        lives on rank 0's GPU (CUDA IPC mapping opened with the rank's own GPU current: the stores ARE the NVLink
        transfer).  No collective on the data path; NCCL carries the timing barrier and the max-reduce only.
        value = 33.2 output Mpx / max-over-ranks device time.  Rank 0 checks the assembled frame against the
        un-tiled result (bit-exact) outside the timed region."""
        from ultrazoom_b200.sharding import (best_grid, frames_for_rank, halo_radius, plan_tiles, run_tile_into, share_frame,
                                             upscale_tiled_refresh)

        model_name, B, H, W, desc = WORKLOADS["cfg5"]
        cfg = MODEL_CONFIGS[model_name]
        r, L = cfg["upscale_ratio"], cfg["num_encoder_layers"]
        torch.manual_seed(0)
        operands = operands_for("cfg5", args)
        model = MewZoom(**cfg, operand_dtype=operands, residual_stream=args.residual_stream).to(dev).eval()
        apply_tune(model)
        eng = model._engine(dev)
        g = torch.Generator().manual_seed(1234)             # every rank holds the same LR frame
        x_host = torch.rand(B, 3, H, W, generator=g)
        if args.io == "uint8":
            x_host = (x_host * 255.0).round().to(torch.uint8)
        x_host = x_host.pin_memory()
        c_host = torch.tensor([[0.5, 0.2, 0.3]]).pin_memory()
        x, c = x_host.to(dev), c_host.to(dev)
        # Halo refresh every K blocks (K = 10: halo 21 instead of 81 LR pixels, 3 exchanges of halo strips between
        # neighbour GPUs per frame, executed work 1.11 x instead of 1.44 x on the 2 x 4 grid) when there is more than one
        # tile; --halo-refresh 0 measures the pure-recompute form.
        refresh = args.halo_refresh if args.halo_refresh >= 0 else (10 if world > 1 else 0)
        R = 2 * refresh + 1 if refresh else halo_radius(L)
        rows, cols = best_grid(H, W, world, R, align_w=128)
        plan = plan_tiles(H, W, rows, cols, R, align_w=128)
        mine = [plan[i] for i in frames_for_rank(len(plan), rank, world)]
        shared = share_frame((B, 3, H * r, W * r), x_host.dtype, 0, rank, dev)
        frame = shared.tensor
        out_px = B * H * r * W * r
        refresh_state = {}

        def step(cc=None):
            if refresh:
                refresh_state["s"] = upscale_tiled_refresh(model, x, c if cc is None else cc, r, L, rows, cols, refresh, frame,
                                                           rank, world, align_w=128, state=refresh_state.get("s"))
                return
            for t in mine:
                run_tile_into(model, x, c, t, r, frame)

        sampler = ClockSampler(local_rank)
        if rank == 0 and sample_clocks:
            sampler.start()
        for _ in range(warmup):
            step()
        barrier()
        _native.check(eng.lib.mz_model_enable_timing(eng.handle, 1))
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.mark_begin()
        ev0.record()
        for _ in range(steps):
            step()
        ev1.record()
        barrier()
        ms_total = ev0.elapsed_time(ev1)
        clocks = sampler.stop() if (rank == 0 and sample_clocks) else None
        conv_ms = C.c_float()
        _native.check(eng.lib.mz_model_conv_stack_ms(eng.handle, C.byref(conv_ms)))
        _native.check(eng.lib.mz_model_enable_timing(eng.handle, 0))
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item()) / steps
        executed = sum((t_.hy1 - t_.hy0) * (t_.hx1 - t_.hx0) for t_ in plan) / (H * W)
        err = None
        if rank == 0:                                       # every rank's stores landed before the barrier returned
            if dump:
                dump_output(args.dump_outputs, "upscale", frame)
            full = model.upscale(x, c)
            err = float((full.float() - frame.float()).abs().max())
            del full
        res = {"workload": "cfg5", "operands": operands, "model_name": model_name, "cfg": cfg, "B": B, "H": H, "W": W, "desc": desc,
               "ms_step": ms_step, "conv_ms": conv_ms.value, "clocks": clocks, "value": out_px / (ms_step * 1e-3) / 1e6,
               "e2e": None, "scaling": "strong", "steps": steps, "fused": bool(eng.lib.mz_model_fused_block(eng.handle)), "npix_executed": int(sum((t_.hy1 - t_.hy0) * (t_.hx1 - t_.hx0) for t_ in mine)),
               "tiling": {"grid": f"{rows}x{cols}", "halo_lr_px": R, "halo_refresh_every_blocks": refresh or None,
                          "exchange": ("halo rectangles of zf + zb pulled out of the neighbour tiles' workspaces by one-sided 2-D gets over NVLink (CUDA IPC mappings); two one-element stream-ordered all-reduces per refresh order them" if refresh and world > 1
                                       else None),
                          "executed_over_algorithmic_work": executed,
                          "max_abs_diff_vs_untiled": err,
                          "stitch": "head kernel stores the core into rank 0's frame (CUDA IPC peer mapping, NVLink)"}}
        if want_e2e:
            # end to end: every rank copies ITS haloed tile from pinned host memory, runs it into rank 0's frame, and
            # rank 0 copies the assembled frame to pinned host memory; wall clock with a barrier on both sides.
            tiles_host = [x_host[:, :, t_.hy0:t_.hy1, t_.hx0:t_.hx1].contiguous().pin_memory() for t_ in mine]
            out_host = torch.empty((B, 3, H * r, W * r), dtype=x_host.dtype).pin_memory() if rank == 0 else None

            def e2e_step():
                if refresh:                                 # the tile crops of the cached plan are refilled from the host
                    for t_, th in zip(mine, tiles_host):
                        refresh_state["s"]["xt"][t_.index].copy_(th, non_blocking=True)
                    step(c_host.to(dev, non_blocking=True))
                for t_, th in zip([] if refresh else mine, tiles_host):
                    xt = th.to(dev, non_blocking=True)
                    cc = c_host.to(dev, non_blocking=True)
                    model.upscale_into(xt, cc, frame, (t_.y0 - t_.hy0, t_.y1 - t_.hy0, t_.x0 - t_.hx0, t_.x1 - t_.hx0),
                                       (t_.y0 * r, t_.x0 * r))
                barrier()                                   # all cores are in the frame
                if rank == 0:
                    out_host.copy_(frame, non_blocking=True)
                    torch.cuda.synchronize()

            e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                e2e_step()
            barrier()
            dt = time.perf_counter() - t0
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
            res["e2e"] = {"value": out_px * steps / dt / 1e6, "unit": "Mpx/s",
                          "h2d_bytes_per_step": int(sum(th.numel() * th.element_size() for th in tiles_host)) + 12,
                          "d2h_bytes_per_step": out_px * 3 * x_host.element_size(), "ms_per_step": 1e3 * dt / steps,
                          "api": "MewZoom.upscale_into per tile (pinned host tile -> device), assembled frame -> pinned host on rank 0"}
        barrier()
        frame = None
        if refresh_state.get("s"):
            from ultrazoom_b200.sharding import close_refresh_state

            close_refresh_state(refresh_state["s"])
            barrier()
        shared.close()
        del model, eng, x, c
        torch.cuda.empty_cache()
        return res

    def roofline_of(res, peaks):
        """Roofline of the dominant kernel (one encoder convolution launch; conv1 and conv2 alternate, so per-launch
        figures are their mean), per SURVEY.md 8(d).  Algorithmic work per launch, unpadded:
          flops = 2 * 9 * C * hC per LR pixel (conv1 == conv2)
          bytes = 6C per LR pixel (16-bit in + out of a convolution: SURVEY 8(d) "conv-stack minimum traffic")
        and, beside it, the bytes THIS design moves per launch (fp32 residual stream + 16-bit shadow):
          mean of conv1 (read zb 2C, write hidden 2hC) and conv2 (read hidden 2hC + zf 4C, write zf 4C + zb 2C).
        The bound is whichever of flops / peak_tensor and algorithmic bytes / peak_hbm is the longer time; the
        tensor fraction is given against both the sustained and the burst 16-bit dense peak."""
        cfg = res["cfg"]
        npix = res.get("npix_executed") or res["B"] * res["H"] * res["W"]    # (cfg5: the haloed tile this rank ran)
        npix_alg = res["B"] * res["H"] * res["W"] / (world if res["workload"] == "cfg5" else 1)
        L, C_ = cfg["num_encoder_layers"], cfg["num_channels"]
        hC = C_ * cfg["hidden_ratio"]
        # Dominant kernel: two launches per encoder block (conv1, conv2), or ONE when the block runs fused
        # (block_fused_kernel: both convolutions, hidden tensor on-chip) -- per-launch work and bytes double, the
        # fractions are the same ratios either way.
        per = 1 if res.get("fused") else 2
        n_launch = per * L
        conv_launch_ms = res["conv_ms"] / n_launch
        conv_flops = conv_flops_per_launch(cfg, npix_alg) * (2 // per)
        alg_bytes = 6.0 * C_ * npix_alg * (2 // per)
        if res.get("fused"):   # read zb 2C + zf 4C, write zf 4C + zb 2C: the hidden tensor never leaves the SM
            design_bytes = 12.0 * C_ * npix
        else:
            design_bytes = 0.5 * ((2 * C_ + 2 * hC) + (2 * hC + 4 * C_ + 4 * C_ + 2 * C_)) * npix
        t_tensor = conv_flops / (peaks["bf16_sustained"] * 1e12)
        t_hbm = alg_bytes / (peaks["hbm"] * 1e9)
        tf = conv_flops / (conv_launch_ms * 1e-3) / 1e12
        gbs_alg = alg_bytes / (conv_launch_ms * 1e-3) / 1e9
        gbs_design = design_bytes / (conv_launch_ms * 1e-3) / 1e9
        total_flops = algorithmic_flops_per_lr_px(cfg) * res["B"] * res["H"] * res["W"]
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):          # DRAM bytes per launch from the committed ncu capture of this workload
            with open(tpath) as f:
                tj = json.load(f).get(res["workload"] + ("_fused" if res.get("fused") else ""))
            if tj:
                traffic, traffic_src = tj["traffic_bytes_per_launch"], tj["source"]
        n_gpus = world if res["workload"] == "cfg5" else 1
        common = {
            "kernel": ("block_fused_kernel (conv1 -> FiLM -> SiLU -> conv2 -> residual, one CTA-pair kernel per encoder block, tcgen05)"
                       if res.get("fused") else "conv_tc_kernel (3x3 implicit GEMM, tcgen05)"),
            "traffic": traffic, "traffic_source": traffic_src,
            "flops_per_launch": conv_flops, "bytes_per_launch": alg_bytes, "design_bytes_per_launch": design_bytes,
            "ms_per_launch": conv_launch_ms,
            "launches_per_step": n_launch, "conv_share_of_step": res["conv_ms"] / res["ms_step"],
            "tensor": {"achieved": tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                       "frac": tf / peaks["bf16_sustained"], "frac_of_burst_peak": tf / peaks["bf16_burst"]},
            "hbm": {"achieved": gbs_alg, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs_alg / peaks["hbm"],
                    "basis": "algorithmic bytes 6C per LR px per convolution (SURVEY 8(d))"},
            "hbm_design": {"achieved": gbs_design, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs_design / peaks["hbm"],
                           "basis": ("bytes this design moves: fp32 residual stream + 16-bit shadow (12C per block; the hidden "
                                     "tensor stays on the SM)") if res.get("fused") else
                                    "bytes this design moves: fp32 residual stream + 16-bit shadow + hidden round trip"},
            "whole_step_tflops_per_gpu": total_flops / n_gpus / (res["ms_step"] * 1e-3) / 1e12,
            "whole_step_frac_of_burst_peak": total_flops / n_gpus / (res["ms_step"] * 1e-3) / 1e12 / peaks["bf16_burst"],
            "peak_source": peaks["source"] + "; tensor = sustained 16-bit dense (kernel timed inside a long step)",
        }
        if t_hbm > t_tensor:
            return {"bound": "hbm", "achieved": gbs_alg, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": gbs_alg / peaks["hbm"], **common}
        return {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                "frac": tf / peaks["bf16_sustained"], **common}

    def measure_unet_ops():
        """The 0.3.0 U-Net operators that are not 3x3 convolutions (SURVEY 8(f) rank 3), each against its HBM roofline:
        algorithmic bytes = every input and output element once, fp32.  Inputs are larger than L2 (126 MB)."""
        from ultrazoom_b200 import unet as N

        g = torch.Generator().manual_seed(5)
        out = {}

        def timed(fn, nbytes, iters=10):
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            return {"ms": ms, "algorithmic_bytes": nbytes, "gb_per_s": nbytes / ms / 1e6}

        C = 96
        x = torch.randn(1, 540, 960, C, generator=g).to(dev)
        z = torch.randn(1, 540, 960, C, generator=g).to(dev)
        w = (torch.randn(C, 2 * C, 1, 1, generator=g) / (2 * C) ** 0.5).to(dev)
        a = torch.tensor(0.25)
        for math in ("tf32", "fp32"):
            out[f"adaptive_residual_mix_c96_960x540_{math}"] = timed(lambda: N.adaptive_residual_mix(x, z, w, a, math), 3 * x.numel() * 4)
        xi = torch.randn(1, 1080, 1920, 48, generator=g).to(dev)
        wc = (torch.randn(96, 48, 2, 2, generator=g) / (4 * 48) ** 0.5).to(dev)
        for math in ("tf32", "fp32"):
            out[f"pixel_crush_f2_48to96_1920x1080_{math}"] = timed(lambda: N.pixel_crush(xi, wc, 2, math),
                                                                   (xi.numel() + 540 * 960 * 96) * 4)
        xs = torch.randn(1, 540, 960, 192, generator=g).to(dev)
        out["pixel_shuffle_nhwc_r2_192to48_960x540"] = timed(lambda: N.pixel_shuffle_nhwc(xs, 2), 2 * xs.numel() * 4)
        out["crop_feature_maps_c96_960x540_to_956x536"] = timed(lambda: N.crop_feature_maps(x, (536, 956)), 2 * 536 * 956 * C * 4)
        # one decoder stage end to end (DecoderBlock + SubpixelConv2d x2, reference model.py:975-1001): three 3x3 convolutions
        # on conv_tc_kernel (96 -> 192 -> 96, 96 -> 4 x 48), the gated mix, the NHWC shuffle; random-init weights
        torch.manual_seed(9)
        blk = N.SR2XBlock(C, 2, 48).to(dev)
        rec = timed(lambda: blk.forward(x), 0, iters=5)
        flops = 2 * 9 * (C * 2 * C * 2 + C * 4 * 48) * 540 * 960
        out["sr2x_block_c96_to_c48_960x540"] = {"ms": rec["ms"], "conv_tflops": flops / rec["ms"] / 1e9,
                                                "note": "composite: 3 tcgen05 3x3 convolutions + mix + shuffle + the casts between them"}
        return out

    def measure_small_kernels():
        """The non-encoder kernels of the path at the headline shape, one launch each through the per-kernel C-ABI entry
        points (ultrazoom_b200.ops): HBM roofline over algorithmic bytes (inputs and outputs once)."""
        from ultrazoom_b200 import ops
        model_name, B, H, W, _ = WORKLOADS["cfg2"]
        cfg = MODEL_CONFIGS[model_name]
        Cc, r = cfg["num_channels"], cfg["upscale_ratio"]
        Cp = ops.padded_channels(Cc)
        g = torch.Generator().manual_seed(0)
        x = torch.rand(B, 3, H, W, generator=g).to(dev)
        zb = torch.randn(B, H, W, Cp, generator=g).to(torch.float16).to(dev)
        wh = ops.pack_conv_weight(torch.randn(3 * r * r, Cc, 3, 3, generator=g) * 0.02, dev)
        ws, bs = torch.randn(Cc, 3, 1, 1, generator=g), torch.randn(Cc, generator=g)
        y = torch.empty(B, 3, H * r, W * r, device=dev)
        npx = B * H * W
        peaks_hbm = load_peaks()["hbm"]

        def timed(fn, nbytes, iters=10):
            for _ in range(3):
                fn()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / iters
            return {"ms": ms, "algorithmic_bytes": nbytes, "gb_per_s": nbytes / ms / 1e6,
                    "frac_of_hbm_peak": nbytes / ms / 1e6 / peaks_hbm}

        return {
            "what": f"one launch each at the headline shape ({B} x {W}x{H}, {Cc} channels, r = {r}); the timed call includes the "
                    "ctypes wrapper's own output allocation",
            "head_conv_shuffle_bicubic_skip_clamp": timed(
                lambda: ops.head_shuffle_add(zb, wh, r, x=x, y=y, skip_mode=2, clamp01=True), npx * (2 * Cp + 12 + 12 * r * r)),
            "stem_nchw_to_nhwc_fp32_and_16bit": timed(lambda: ops.stem_pack(x, ws, bs), npx * (12 + 6 * Cp)),
            "bicubic_standalone": timed(lambda: ops.bicubic(x, r), npx * (12 + 12 * r * r)),
        }

    main_res = measure(args.workload, args.steps, args.warmup, not args.no_e2e, True, dump=bool(args.dump_outputs))
    # The north_star's efficiency target is stated on MewZoom-4X-Ctrl and its hard multi-GPU case is the spatial split:
    # the default line carries those as first-class records (own clocks; 4X-Ctrl with its own e2e) under "also".
    also = {}
    if args.workload == "cfg2" and not args.no_also:
        k = args.steps
        also["cfg4a"] = measure("cfg4a", k, args.warmup, not args.no_e2e, True)
        also["cfg3"] = measure("cfg3", k, args.warmup, False, True)
        also["cfg5"] = measure("cfg5", k, args.warmup, False, True)
        # the same headline workload with the other 16-bit operand type (same tcgen05 rate and bytes; see operands_for)
        other = "float16" if main_res["operands"] == "bfloat16" else "bfloat16"
        also["cfg2_fp16" if other == "float16" else "cfg2_bf16"] = measure("cfg2", k, args.warmup, False, True, operands=other)
    unet_ops = measure_unet_ops() if (args.workload == "cfg2" and not args.no_also and world == 1) or args.unet_ops else None
    small = measure_small_kernels() if args.workload == "cfg2" and not args.no_also and world == 1 else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    res = main_res
    model_name, cfg, B, H, W, desc = res["model_name"], res["cfg"], res["B"], res["H"], res["W"], res["desc"]
    ms_step, value, e2e, clocks = res["ms_step"], res["value"], res["e2e"], res["clocks"]
    L = cfg["num_encoder_layers"]
    launches_per_step = (1 if res.get("fused") else 2) * L + 2 + (1 if cfg["control_features"] else 0)
    roofline = roofline_of(res, peaks)
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:   # reported at N = 1 only
        threads = os.cpu_count() or 1
        sh, sw = H, W
        while sh * sw > 540 * 960:
            sh, sw = sh // 2, sw // 2
        mpx, dt = cpu_port_sample(model_name, sh, sw, threads)
        cpu_baseline = {"value": mpx, "unit": "Mpx/s", "cores": threads, "kind": "port",
                        "sample": f"1 frame {sw}x{sh} of the workload, fp32 oracle, {dt:.1f} s"}
    line = {
        "metric": "output_mpx_per_s", "value": value, "unit": "Mpx/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": res["scaling"],
        "vs_baseline": None, "dtype": "f16" if res["operands"] == "float16" else "bf16", "data": "synthetic",
        "config": config_of(args.workload, world, args, res["operands"]),
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e,
        "gpu_launches": launches_per_step * args.steps, "clocks": clocks,
        "ms_per_frame": ms_step / B,
    }
    if res.get("e2e_uint8"):
        line["e2e_uint8"] = res["e2e_uint8"]
    if "tiling" in res:
        line["tiling"] = res["tiling"]
    if also:
        line["also"] = {}
        for name, ar in also.items():
            rec = {"workload": ar["desc"] + (f" -- {ar['operands']} tensor-core operands" if name.startswith("cfg2_") else ""),
                   "value": ar["value"], "unit": "Mpx/s", "scaling": ar["scaling"],
                   "steps": ar["steps"], "ms_per_frame": ar["ms_step"], "roofline": roofline_of(ar, peaks),
                   "clocks": ar["clocks"], "e2e": ar["e2e"], "e2e_uint8": ar.get("e2e_uint8"), "config": config_of(ar["workload"], world, args, ar["operands"]),
                   "dtype": "f16" if ar["operands"] == "float16" else "bf16"}
            if "tiling" in ar:
                rec["tiling"] = ar["tiling"]
            line["also"][name] = rec
    if unet_ops:
        for rec in unet_ops.values():
            if "gb_per_s" in rec:
                rec["frac_of_hbm_peak"] = rec["gb_per_s"] / peaks["hbm"]
        line.setdefault("also", {})["unet_ops"] = {
            "what": "0.3.0 U-Net operators beside the 3x3 convolutions (SURVEY 8(f) rank 3): one launch each, fp32 NHWC feature "
                    "maps larger than L2, HBM roofline over algorithmic bytes (every input and output element once); "
                    "tf32 = tcgen05 kind::tf32 GEMM from the fp32 maps (default), fp32 = the exact SIMT twin",
            "hbm_peak_gb_per_s": peaks["hbm"], "ops": unet_ops}
    if small:
        line.setdefault("also", {})["small_kernels"] = small
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
