"""Work partitioning for multi-GPU runs -- one process per GPU, NO collective on the hot path.

Two partitionings (SURVEY.md section 8(e)):
  * frame stream: frame i of a stream goes to rank ``i % world`` (``frames_for_rank``);
  * spatial tiles with halo: one large image is cut into a cols x rows grid of LR tiles, each extended
    by the network's receptive-field radius ``halo_radius(L) = 2L + 1`` LR pixels (every block has two
    3x3 convs, the head one more); each rank runs the whole network on its haloed tile with ordinary
    image-border semantics and keeps only the core (``plan_tiles`` / ``upscale_tiled``).
    Tiles touching a true image border take no halo on that side, so zero padding (convs) and clamped
    taps (bicubic) there are exactly the full-image ones.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, List, Optional, Sequence, Tuple

import torch
from torch import Tensor


def halo_radius(num_encoder_layers: int) -> int:
    """LR-pixel halo that makes tiled inference exact: 2 convs per block + the head conv.

    The bicubic skip only needs 2 LR pixels, which this always covers."""
    return 2 * num_encoder_layers + 1


def bind_process_to_gpu(device_index: int) -> Optional[List[int]]:
    """One process per GPU with HOST buffers: pin the calling thread (and the threads it starts later) to the CPUs
    next to GPU ``device_index`` (NVML's ideal-CPU set: the GPU's NUMA node), so that the pinned staging buffers it
    allocates afterwards are node-local and the H2D / D2H copies of eight ranks do not all cross one socket's memory
    controller and the inter-socket link.  Call it first thing in the rank, before any pinned allocation.  Returns the
    CPU list, or None when NVML / the device is not available (nothing is changed then)."""
    try:
        import os

        import pynvml

        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(device_index)
        h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(props.uuid)).encode())
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return sorted(os.sched_getaffinity(0))
    except Exception:       # noqa: BLE001 -- a placement hint: never fatal
        return None


def frames_for_rank(num_frames: int, rank: int, world: int) -> List[int]:
    assert world > 0 and 0 <= rank < world, f"bad rank {rank} / world {world}"
    return list(range(rank, num_frames, world))


@dataclass(frozen=True)
class Tile:
    index: int
    # core region in LR pixels (what this tile contributes to the output)
    y0: int
    y1: int
    x0: int
    x1: int
    # haloed region actually fed to the network
    hy0: int
    hy1: int
    hx0: int
    hx1: int


def _splits(n: int, parts: int) -> List[Tuple[int, int]]:
    base, extra = divmod(n, parts)
    out, s = [], 0
    for i in range(parts):
        e = s + base + (1 if i < extra else 0)
        out.append((s, e))
        s = e
    return out


def _splits_aligned(n: int, parts: int, halo: int, align: int) -> List[Tuple[int, int]]:
    """Split [0, n) into ``parts`` cores such that every HALOED extent (core + halo on each interior side) needs as
    few ``align``-wide kernel tiles as possible and all parts need the same number: the convolution kernel works on
    128-pixel-wide tiles, so a 642-pixel haloed tile costs six of them where 640 cost five."""
    if parts == 1 or align <= 1:
        return _splits(n, parts)
    sides = [(1 if i > 0 else 0) + (1 if i < parts - 1 else 0) for i in range(parts)]
    t = 1
    while sum(max(t * align - halo * s, 0) for s in sides) < n:
        t += 1
    cap = [t * align - halo * s for s in sides]
    if min(cap) <= 0:
        return _splits(n, parts)
    excess = sum(cap) - n
    # hand the slack back evenly (never below one pixel per core); any core <= its cap keeps the tile count at t
    core = list(cap)
    i = 0
    while excess > 0:
        take = min(excess, max((core[i] - 1), 0), -(-excess // parts))
        core[i] -= take
        excess -= take
        i = (i + 1) % parts
    out, s0 = [], 0
    for c in core:
        out.append((s0, s0 + c))
        s0 += c
    assert s0 == n
    return out


ROW_ALIGN = 4   # the fused-block kernel ties its accumulator ring (4 blocks) to the image row: see plan_tiles


def plan_tiles(H: int, W: int, rows: int, cols: int, halo: int, align_w: int = 1, align_rows: int = ROW_ALIGN) -> List[Tile]:
    """``align_w`` = 128 sizes the columns for the convolution kernel's 128-pixel tiles (see ``_splits_aligned``).
    ``align_rows``: the first row of a haloed tile is moved up to a multiple of it (a few more halo rows are harmless).
    The fused encoder block sums the accumulators of rows 0 / 1 mod 4 in two parts; with tile origins on multiples of 4
    a row keeps its association inside a tile, so tiled inference stays BIT-identical to the un-tiled frame."""
    assert rows > 0 and cols > 0 and rows <= H and cols <= W, f"bad grid {rows}x{cols} for a {H}x{W} image"
    assert halo >= 0 and align_rows >= 1
    tiles = []
    for iy, (y0, y1) in enumerate(_splits(H, rows)):
        for ix, (x0, x1) in enumerate(_splits_aligned(W, cols, halo, align_w)):
            hy0 = max(0, y0 - halo)
            hy0 -= hy0 % align_rows
            tiles.append(Tile(iy * cols + ix, y0, y1, x0, x1, hy0, min(H, y1 + halo), max(0, x0 - halo), min(W, x1 + halo)))
    return tiles


def best_grid(H: int, W: int, n_tiles: int, halo: int, align_w: int = 1) -> Tuple[int, int]:
    """rows x cols = n_tiles grid with the least executed work: the haloed area, or with ``align_w`` the slowest tile's
    area with its width rounded up to whole kernel tiles (tiles run in parallel, one per GPU)."""
    best, best_cost = (1, n_tiles), None
    for rows in range(1, n_tiles + 1):
        if n_tiles % rows:
            continue
        cols = n_tiles // rows
        if rows > H or cols > W:
            continue
        plan = plan_tiles(H, W, rows, cols, halo, align_w)
        if align_w > 1:
            cost = max((t.hy1 - t.hy0) * (-(-(t.hx1 - t.hx0) // align_w) * align_w) for t in plan)
        else:
            cost = sum((t.hy1 - t.hy0) * (t.hx1 - t.hx0) for t in plan)
        if best_cost is None or cost < best_cost:
            best, best_cost = (rows, cols), cost
    return best


def run_tile(fn: Callable[[Tensor, Optional[Tensor]], Tensor], x: Tensor, c: Optional[Tensor], t: Tile,
             r: int) -> Tensor:
    """Run ``fn`` on the haloed tile and crop its HR core."""
    y = fn(x[:, :, t.hy0:t.hy1, t.hx0:t.hx1].contiguous(), c)
    oy, ox = (t.y0 - t.hy0) * r, (t.x0 - t.hx0) * r
    return y[:, :, oy:oy + (t.y1 - t.y0) * r, ox:ox + (t.x1 - t.x0) * r]


def stitch(out: Tensor, tile_out: Tensor, t: Tile, r: int) -> None:
    out[:, :, t.y0 * r:t.y1 * r, t.x0 * r:t.x1 * r] = tile_out


def upscale_tiled(fn: Callable[[Tensor, Optional[Tensor]], Tensor], x: Tensor, c: Optional[Tensor], r: int,
                  num_encoder_layers: int, rows: int, cols: int, tiles: Optional[Sequence[int]] = None,
                  out: Optional[Tensor] = None, align_w: int = 1) -> Tensor:
    """Tiled inference, exact w.r.t. the full-image result.  ``tiles`` selects which tile indices THIS
    caller computes (e.g. ``frames_for_rank(rows*cols, rank, world)``); the others are left untouched in
    ``out`` so ranks can fill disjoint parts of a shared / gathered buffer."""
    B, _, H, W = x.shape
    plan = plan_tiles(H, W, rows, cols, halo_radius(num_encoder_layers), align_w)
    if out is None:
        out = torch.zeros((B, 3, H * r, W * r), dtype=torch.float32, device=x.device)
    for t in plan:
        if tiles is not None and t.index not in tiles:
            continue
        stitch(out, run_tile(fn, x, c, t, r), t, r)
    return out


# ---- assembling the frame on one GPU: one-sided puts over NVLink, no collective (SURVEY.md 8(e)) --------------------
class SharedFrame:
    """The assembled HR frame of a one-process-per-GPU tiled run: allocated by the owner rank, mapped by every other rank
    of the node through a CUDA IPC handle opened with that rank's own GPU current (mz_ipc_frame_*), so that both the
    head kernel's stores (``run_tile_into``) and 2-D copies (``put_core``) reach it over NVLink.  ``.tensor`` is the
    (B,3,H,W) view on each rank; keep the object alive while anything is in flight, ``close()`` when done."""

    def __init__(self, shape, dtype: torch.dtype, owner: int, rank: int, device: torch.device, group=None):
        import ctypes as C

        import torch.distributed as dist

        from . import _native

        self.lib, self.owner = _native.load(), rank == owner
        self.ptr = C.c_void_p()
        numel = 1
        for d in shape:
            numel *= int(d)
        handle = C.create_string_buffer(64)
        with torch.cuda.device(device):
            if self.owner:
                nbytes = numel * torch.empty(0, dtype=dtype).element_size()
                _native.check(self.lib.mz_ipc_frame_create(nbytes, C.byref(self.ptr), handle))
            box = [handle.raw if self.owner else None]
            if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
                dist.broadcast_object_list(box, src=owner, group=group)   # control plane: 64 bytes, once
            if not self.owner:
                _native.check(self.lib.mz_ipc_frame_open(box[0], C.byref(self.ptr)))
        typestr = {torch.float32: "<f4", torch.uint8: "|u1", torch.uint16: "<u2"}[dtype]

        class _Mem:
            __cuda_array_interface__ = {"shape": tuple(int(d) for d in shape), "typestr": typestr,
                                        "data": (self.ptr.value, False), "version": 2}

        self.tensor = torch.as_tensor(_Mem())      # zero-copy view of the mapping (on the device CUDA reports for it)

    def close(self) -> None:
        if self.ptr:
            from . import _native

            self.tensor = None
            _native.check(self.lib.mz_ipc_frame_close(self.ptr, 1 if self.owner else 0))
            self.ptr = None


def share_frame(shape, dtype: torch.dtype, owner: int, rank: int, device: torch.device, group=None) -> SharedFrame:
    """Collective over the control plane (once, outside the timed loop): see ``SharedFrame``."""
    return SharedFrame(shape, dtype, owner, rank, device, group)


def put_core(frame: Tensor, tile_out: Tensor, t: Tile, r: int) -> None:
    """Write the HR core of tile ``t`` (``run_tile``'s result on this rank's GPU) into ``frame`` -- which may live on
    another GPU (``share_frame``) or in pinned host memory -- as 2-D copies on the current stream (mz_put_plane_async),
    one per image plane.  Nothing synchronises: order a later reader with an event or the timing barrier."""
    from . import _native

    lib = _native.load()
    B, C, h, w = tile_out.shape
    assert (h, w) == ((t.y1 - t.y0) * r, (t.x1 - t.x0) * r) and frame.shape[:2] == tile_out.shape[:2]
    assert tile_out.stride(3) == 1 and frame.stride(3) == 1 and frame.dtype == tile_out.dtype
    es = tile_out.element_size()
    stream = torch.cuda.current_stream(tile_out.device).cuda_stream
    for b in range(B):
        for ch in range(C):
            dst = frame[b, ch, t.y0 * r:t.y1 * r, t.x0 * r:t.x1 * r]
            src = tile_out[b, ch]
            _native.check(lib.mz_put_plane_async(dst.data_ptr(), dst.stride(0) * es, src.data_ptr(), src.stride(0) * es,
                                                 w * es, h, stream))


def run_tile_into(model, x: Tensor, c: Optional[Tensor], t: Tile, r: int, frame: Tensor) -> None:
    """``run_tile`` + ``put_core`` in one pass: the head kernel of the tile writes the core straight into ``frame``
    (``MewZoom.upscale_into`` -> mz_upscale_window); with a peer ``frame`` its stores are the NVLink transfer."""
    model.upscale_into(x[:, :, t.hy0:t.hy1, t.hx0:t.hx1], c, frame,
                       (t.y0 - t.hy0, t.y1 - t.hy0, t.x0 - t.hx0, t.x1 - t.hx0), (t.y0 * r, t.x0 * r))


# ---- periodic halo refresh (SURVEY.md 8(e) "per-layer halo exchange", made coarse; VERDICT r1 item 4) ---------------
# A tile that carries the full receptive-field halo (2L+1 = 81 LR pixels for 40 blocks) recomputes 44 % extra pixels on
# the 4 x 2 grid of a 1080p frame.  With a halo of only 2k+1 pixels the network runs k blocks at a time; after each
# group the outer 2k pixels of the halo are stale, and every tile refreshes its halo ring -- fp32 residual stream and
# 16-bit shadow -- with the values its neighbours computed for those pixels inside their cores.  k = 10: 3 exchanges of
# a few MB per neighbour, executed work 1.13 x instead of 1.44 x.  The exchanged values are the very numbers an
# un-tiled run computes (a pixel's result does not depend on the tile origin: tile rows start on multiples of ROW_ALIGN),
# so the assembled frame stays bit-identical.  This is the one place the path has a real exchange step: one-sided copies
# inside a process, NCCL point-to-point (grouped isend / irecv, no collective reduction) between processes.
def _intersect(a, b):
    y0, y1, x0, x1 = max(a[0], b[0]), min(a[1], b[1]), max(a[2], b[2]), min(a[3], b[3])
    return (y0, y1, x0, x1) if y0 < y1 and x0 < x1 else None


def refresh_rects(plan: Sequence[Tile]):
    """{(i, j): (y0, y1, x0, x1)}: the part of tile i's haloed region that lies in tile j's core (global LR
    coordinates) -- what i receives from j at every refresh.  Cores tile the frame, so for a fixed i the rectangles
    over j != i cover i's halo exactly once."""
    out = {}
    for a in plan:
        for b in plan:
            if a.index == b.index:
                continue
            r = _intersect((a.hy0, a.hy1, a.hx0, a.hx1), (b.y0, b.y1, b.x0, b.x1))
            if r is not None:
                out[(a.index, b.index)] = r
    return out


class _StageBuffer:
    """Workspace of one tile for staged execution, allocated so that OTHER processes of the node can map it (CUDA IPC):
    neighbours pull their halo strips straight out of it over NVLink.  ``tensor`` is the uint8 view ``upscale_stage`` takes."""

    def __init__(self, nbytes: int, device: torch.device):
        import ctypes as C

        from . import _native

        self.lib = _native.load()
        self.ptr = C.c_void_p()
        self.handle = C.create_string_buffer(64)
        self.nbytes = nbytes
        with torch.cuda.device(device):
            _native.check(self.lib.mz_ipc_frame_create(nbytes, C.byref(self.ptr), self.handle))

        class _Mem:
            __cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (self.ptr.value, False), "version": 2}

        self.tensor = torch.as_tensor(_Mem())          # zero-copy view (on the device CUDA reports for the allocation)
        self.base = (-self.ptr.value) % 1024          # offset of the 1024-byte-aligned workspace inside the allocation

    def close(self) -> None:
        if self.ptr:
            from . import _native

            self.tensor = None
            _native.check(self.lib.mz_ipc_frame_close(self.ptr, 1))
            self.ptr = None


def upscale_tiled_refresh(model, x: Tensor, c: Optional[Tensor], r: int, num_encoder_layers: int, rows: int, cols: int,
                          refresh_every: int, frame: Tensor, rank: int = 0, world: int = 1, group=None, align_w: int = 1,
                          state: Optional[dict] = None) -> dict:
    """Halo-tiled ``upscale`` of ONE frame with a halo refresh every ``refresh_every`` encoder blocks.  Tile i of the
    ``rows x cols`` grid belongs to rank ``i % world``; every tile's core lands in ``frame`` (``share_frame`` when the
    ranks are processes).  ``state`` (returned) caches the plan, tile crops, workspaces and peer mappings between calls.

    Refresh = ONE-SIDED GETS: every tile's workspace is mapped by its neighbours (CUDA IPC, opened with the puller's GPU
    current), and a tile pulls each halo rectangle of the fp32 stream and of the 16-bit shadow out of the neighbour's
    core with one 2-D copy (mz_put_plane_async: rows of (x1 - x0) * C elements at the two tiles' row pitches) over
    NVLink.  Two tiny stream-ordered all-reduces per refresh order the gets against the neighbours' kernels ("everyone
    has finished the group" / "everyone has finished pulling"); no data moves through a collective."""
    import ctypes as C

    import torch.distributed as dist

    from . import _native

    L, k = num_encoder_layers, refresh_every
    assert 1 <= k <= L, "refresh_every must be in [1, num_encoder_layers]"
    B, _, H, W = x.shape
    multi = world > 1
    lib = _native.load()
    if state is None:
        plan = plan_tiles(H, W, rows, cols, 2 * k + 1, align_w)
        mine = [t for t in plan if t.index % world == rank]
        rects = refresh_rects(plan)
        state = {"plan": plan, "mine": mine, "rects": rects, "buf": {}, "xt": {}, "peer": {}, "layout": {},
                 "token": torch.zeros(1, device=x.device)}
        eng = model._engine(x.device)
        for t in plan:                                  # workspace layout of EVERY tile (a peer's offsets are computed here)
            zf_o, zb_o, hid_o, cp, zp = C.c_size_t(), C.c_size_t(), C.c_size_t(), C.c_int32(), C.c_int32()
            _native.check(lib.mz_workspace_layout(eng.handle, B, t.hy1 - t.hy0, t.hx1 - t.hx0, C.byref(zf_o), C.byref(zb_o),
                                                  C.byref(hid_o), C.byref(cp), C.byref(zp)))
            state["layout"][t.index] = (zf_o.value, zb_o.value, hid_o.value, cp.value, zp.value)
        state["fused"] = bool(lib.mz_model_fused_block(eng.handle))
        for t in mine:
            xt = x[:, :, t.hy0:t.hy1, t.hx0:t.hx1].contiguous()
            state["xt"][t.index] = xt
            need = C.c_size_t()
            _native.check(lib.mz_workspace_bytes(eng.handle, B, xt.shape[2], xt.shape[3], C.byref(need)))
            state["buf"][t.index] = _StageBuffer(need.value + 1024, x.device)
        # base addresses (of the aligned workspace) of every tile some tile of mine pulls from
        local = {i: b.ptr.value + b.base for i, b in state["buf"].items()}
        if multi:
            gathered = [None] * world
            dist.all_gather_object(gathered, {i: (b.handle.raw, b.base) for i, b in state["buf"].items()}, group=group)
            with torch.cuda.device(x.device):
                for (i, j) in rects:
                    if i % world == rank and j % world != rank and j not in state["peer"]:
                        raw, base = gathered[j % world][j]
                        p = C.c_void_p()
                        _native.check(lib.mz_ipc_frame_open(raw, C.byref(p)))
                        state["peer"][j] = p.value + base
                        state.setdefault("mappings", []).append(p)
        state["addr"] = {**state["peer"], **local}
    plan, mine, rects, addr = state["plan"], state["mine"], state["rects"], state["addr"]
    by_index = {t.index: t for t in plan}
    bounds = list(range(0, L, k)) + [L]
    es16 = 2
    stream = torch.cuda.current_stream(x.device)

    def planes(idx: int, blocks_done: int):
        """(offset, channel pitch, element size) of the fp32 stream and of the current 16-bit stream of tile idx."""
        zf_o, zb_o, hid_o, cp, zp = state["layout"][idx]
        in_hidden = state["fused"] and (blocks_done & 1)
        return ((zf_o, cp, 4), (hid_o, cp, es16) if in_hidden else (zb_o, zp, es16))

    for g in range(len(bounds) - 1):
        l0, l1 = bounds[g], bounds[g + 1]
        if g > 0:
            if multi:
                dist.all_reduce(state["token"], group=group)          # every rank's group g-1 kernels precede its arrival
            with torch.cuda.device(x.device):
                for (i, j), rect in rects.items():
                    if i % world != rank:
                        continue                                        # tile i (mine) pulls rect out of tile j's core
                    ti, tj = by_index[i], by_index[j]
                    Wi, Wj, Hi, Hj = ti.hx1 - ti.hx0, tj.hx1 - tj.hx0, ti.hy1 - ti.hy0, tj.hy1 - tj.hy0
                    h, w = rect[1] - rect[0], rect[3] - rect[2]
                    for (so, sp, es), (do, dp, _) in zip(planes(j, l0), planes(i, l0)):
                        for b in range(B):
                            src = addr[j] + so + ((b * Hj + rect[0] - tj.hy0) * Wj + rect[2] - tj.hx0) * sp * es
                            dst = addr[i] + do + ((b * Hi + rect[0] - ti.hy0) * Wi + rect[2] - ti.hx0) * dp * es
                            # (rows of min(sp, dp) channels: the pitches agree -- same model, same padding)
                            _native.check(lib.mz_put_plane_async(dst, Wi * dp * es, src, Wj * sp * es, w * sp * es, h,
                                                                 stream.cuda_stream))
            if multi:
                dist.all_reduce(state["token"], group=group)          # nobody overwrites a core that is still being pulled
        for t in mine:
            model.upscale_stage(state["xt"][t.index], c, frame, (t.y0 - t.hy0, t.y1 - t.hy0, t.x0 - t.hx0, t.x1 - t.hx0),
                                (t.y0 * r, t.x0 * r), l0, l1, state["buf"][t.index].tensor)
    return state



def close_refresh_state(state: Optional[dict]) -> None:
    """Release what ``upscale_tiled_refresh`` cached: peer mappings first, then this rank's own workspaces (call it on
    every rank, after a barrier: a workspace must not disappear while a neighbour still maps it)."""
    if not state:
        return
    from . import _native

    lib = _native.load()
    for p in state.pop("mappings", []):
        _native.check(lib.mz_ipc_frame_close(p, 0))
    for b in state.pop("buf", {}).values():
        b.close()
