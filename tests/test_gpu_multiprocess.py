"""GPU, two processes / two GPUs (skipped on a one-GPU box): the multi-process half of the spatial split (SURVEY.md
8(e), partitioning 2) that a single process cannot exercise -- a NON-owner rank opens the owner's frame through the CUDA
IPC handle (mz_ipc_frame_open) with its own GPU current and its head kernels store the cores of its tiles straight into
the owner's memory over NVLink (run_tile_into -> mz_upscale_window); the copy form (put_core) likewise.  The assembled
frame equals the un-tiled result bit for bit.  Control plane: gloo on 127.0.0.1 (64-byte handle + barriers); there is
no collective on the data path."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, mode: str, out_path: str):
    import torch.distributed as dist

    from ultrazoom_b200 import MODEL_CONFIGS, MewZoom
    from ultrazoom_b200.sharding import (frames_for_rank, halo_radius, plan_tiles, put_core, run_tile, run_tile_into,
                                         share_frame)

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        cfg = dict(MODEL_CONFIGS["MewZoom-4X-Ctrl"])
        cfg["num_encoder_layers"] = 3
        torch.manual_seed(51)                                           # every rank builds the same replica
        m = MewZoom(**cfg).to(dev).eval()
        g = torch.Generator().manual_seed(52)
        H, W, r = 70, 300, 4
        io8 = mode == "uint8"
        x = torch.rand(1, 3, H, W, generator=g)
        if io8:
            x = (x * 255).to(torch.uint8)
        x, c = x.to(dev), torch.rand(1, 3, generator=g).to(dev)
        plan = plan_tiles(H, W, 2, 2, halo_radius(3), align_w=128)
        shared = share_frame((1, 3, H * r, W * r), torch.uint8 if io8 else torch.float32, 0, rank, dev)
        for i in frames_for_rank(len(plan), rank, world):               # tiles 0, 2 on rank 0; 1, 3 on rank 1
            if mode == "copy":
                put_core(shared.tensor, run_tile(m.upscale, x, c, plan[i], r), plan[i], r)
            else:
                run_tile_into(m, x, c, plan[i], r, shared.tensor)
        torch.cuda.synchronize()
        dist.barrier()                                                  # every rank's stores have landed
        if rank == 0:
            full = m.upscale(x, c)
            ok = bool(torch.equal(shared.tensor, full))
            with open(out_path, "w") as f:
                f.write("ok" if ok else f"mismatch {(shared.tensor.float() - full.float()).abs().max().item()}")
        dist.barrier()
        shared.close()
    finally:
        dist.destroy_process_group()


def _refresh_worker(rank: int, world: int, port: int, out_path: str):
    import torch.distributed as dist

    from ultrazoom_b200 import MODEL_CONFIGS, MewZoom
    from ultrazoom_b200.sharding import share_frame, upscale_tiled_refresh

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        results = []
        for name, L, k in (("MewZoom-4X-Ctrl", 4, 2), ("MewZoom-2X-Ctrl", 5, 1)):
            cfg = dict(MODEL_CONFIGS[name])
            cfg["num_encoder_layers"] = L
            r = cfg["upscale_ratio"]
            torch.manual_seed(71)
            m = MewZoom(**cfg).to(dev).eval()
            g = torch.Generator().manual_seed(72)
            H, W = 60, 300
            x, c = torch.rand(1, 3, H, W, generator=g).to(dev), torch.rand(1, 3, generator=g).to(dev)
            shared = share_frame((1, 3, H * r, W * r), torch.float32, 0, rank, dev)
            for rows, cols in ((1, 2), (2, 2)):                          # one tile per rank / two tiles per rank
                upscale_tiled_refresh(m, x, c, r, L, rows, cols, k, shared.tensor, rank, world, align_w=128)
                torch.cuda.synchronize()
                dist.barrier()
                if rank == 0:
                    results.append(bool(torch.equal(shared.tensor, m.upscale(x, c))))
                    shared.tensor.zero_()
                    torch.cuda.synchronize()
                dist.barrier()
            shared.close()
        if rank == 0:
            with open(out_path, "w") as f:
                f.write("ok" if all(results) and len(results) == 4 else f"mismatch {results}")
    finally:
        dist.destroy_process_group()


def test_halo_refresh_across_two_gpus(tmp_path):
    """Periodic halo refresh between PROCESSES: every rank reads the halo strips of the fp32 stream and its 16-bit shadow
    out of its neighbours' IPC-mapped stage buffers (one-sided gets over NVLink, ordered by two 1-element all-reduces per
    refresh), cores land in rank 0's IPC frame; the result equals the un-tiled frame bit for bit, with one and with two
    tiles per rank."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp

    out = str(tmp_path / "result.txt")
    mp.spawn(_refresh_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert open(out).read() == "ok"


@pytest.mark.parametrize("mode", ["fused", "copy", "uint8"])
def test_non_owner_rank_fills_the_owners_frame(tmp_path, mode):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp

    out = str(tmp_path / "result.txt")
    mp.spawn(_worker, args=(2, _free_port(), mode, out), nprocs=2, join=True)
    assert open(out).read() == "ok"
