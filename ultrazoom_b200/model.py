"""MewZoom -- drop-in for ``ultrazoom.model.MewZoom`` (reference src/ultrazoom/model.py:43-192, 0.2.x
``upscale(x, c)`` signature per README.md:124) whose forward pass runs on hand-written sm_100a kernels.

The ``torch.nn`` sub-modules below only *hold* the parameters (same shapes, same default initialisation and
the same ``state_dict`` keys as the flat architecture BASELINE.json names, SURVEY.md Appendix C); they are
never called.  ``forward`` hands device pointers to the C ABI (include/mewzoom_b200.h) on the current CUDA
stream.  There is no CPU / eager fallback: a non-CUDA input or a missing native library raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
from torch import Tensor, nn

try:  # the reference mixes this in (model.py:37,43); keep from_pretrained/save_pretrained working
    from huggingface_hub import PyTorchModelHubMixin
except Exception:  # pragma: no cover - hub not installed

    class PyTorchModelHubMixin:  # type: ignore
        pass


from . import _native


def _is_nhwc(t: Tensor) -> bool:
    """``t`` holds interleaved pixels: (B,3,H,W) in ``channels_last`` strides -- what a numpy / PIL / video frame becomes
    through ``torch.from_numpy(frames).permute(0, 3, 1, 2)`` -- and not also plainly contiguous."""
    return t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()


_INT_IMAGE_DTYPES = (torch.uint8, torch.uint16)   # images the kernels read and write as integers (MZ_FLAG_IO_U8 / _U16)


def _input_image(x: Tensor, integer: bool):
    """``(x, flag)``: the image as the kernels read it -- uint8 / uint16 as it is, anything else as float32 -- kept
    interleaved when it is (``MZ_FLAG_X_NHWC``, no transpose), otherwise made contiguous NCHW."""
    nhwc = _is_nhwc(x)
    x = x.detach() if integer else x.detach().to(torch.float32)
    x = x.contiguous(memory_format=torch.channels_last if nhwc else torch.contiguous_format)
    return x, (_native.FLAG_X_NHWC if nhwc else 0)


def _output_flag(memory_format) -> int:
    assert memory_format in (torch.contiguous_format, torch.channels_last), (
        "memory_format must be torch.contiguous_format or torch.channels_last")
    return _native.FLAG_Y_NHWC if memory_format == torch.channels_last else 0


def _frame_layout(frame: Tensor):
    """``(flag, row pitch, image-or-plane pitch)`` of an assembled output frame (B,3,H',W'): interleaved (channels-last
    strides: ``stride(1) == 1``, ``stride(3) == 3``; rows and images at any pitch) or planar (``stride(3) == 1``, evenly
    spaced planes)."""
    if frame.stride(1) == 1 and frame.stride(3) == 3:
        return _native.FLAG_Y_NHWC, frame.stride(2), frame.stride(0)
    assert frame.stride(3) == 1, "frame must be planar (stride(3) == 1) or interleaved (stride(1) == 1, stride(3) == 3)"
    assert frame.stride(0) == 3 * frame.stride(1), "frame planes must be evenly spaced"
    return 0, frame.stride(2), frame.stride(1)


class FanOutProjection(nn.Module):
    """Parameter holder for the 1x1 stem (reference model.py:212-242)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        assert in_channels > 0, "Input channels must be greater than 0."
        assert in_channels < out_channels, "Output channels must be greater than input channels."
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=1)


class InvertedBottleneck(nn.Module):
    """Parameter holder for conv3x3 -> SiLU -> conv3x3 (reference model.py:731-778)."""

    def __init__(self, num_channels: int, hidden_ratio: int):
        super().__init__()
        assert num_channels > 0, "Number of channels must be greater than 0."
        assert hidden_ratio in {1, 2, 4}, "Hidden ratio must be either 1, 2, or 4."
        hidden = hidden_ratio * num_channels
        self.conv1 = nn.Conv2d(num_channels, hidden, kernel_size=3, padding=1, bias=False)
        self.conv2 = nn.Conv2d(hidden, num_channels, kernel_size=3, padding=1, bias=False)


class ControlModule(nn.Module):
    """Parameter holder for the per-layer FiLM control (restated; SURVEY.md Appendix C)."""

    def __init__(self, control_features: int, hidden_channels: int):
        super().__init__()
        assert control_features > 0, "Control features must be greater than 0."
        self.linear = nn.Linear(control_features, 2 * hidden_channels, bias=True)


class EncoderBlock(nn.Module):
    """One residual block (reference model.py:487-511 with the plain ResidualConnection :781-792)."""

    def __init__(self, num_channels: int, hidden_ratio: int, control_features: int):
        super().__init__()
        self.convnet = InvertedBottleneck(num_channels, hidden_ratio)
        if control_features > 0:
            self.control = ControlModule(control_features, hidden_ratio * num_channels)


class SubpixelConv2d(nn.Module):
    """Parameter holder for conv3x3 -> PixelShuffle (reference model.py:885-930)."""

    def __init__(self, in_channels: int, out_channels: int, upscale_ratio: int):
        super().__init__()
        assert upscale_ratio in {2, 3, 4}, "Upscale ratio must be either 2, 3, or 4."
        self.conv = nn.Conv2d(in_channels, out_channels * upscale_ratio**2, kernel_size=3, padding=1, bias=False)


class _Engine:
    """One native mz_model on one device (for one operand dtype) + its cached workspace.

    One workspace and one prepared-launch cache serve every call, so calls are serialised on the device: a call
    enqueued on a different CUDA stream than the previous one first waits for that call's kernels (an event), and the
    workspace is marked as used on every stream that touched it, so the caching allocator cannot hand it out while
    kernels still run (ADVICE r1: stream-level concurrency)."""

    def __init__(self, owner: "MewZoom", device: torch.device, operand_dtype: str):
        self.lib = _native.load()
        if self.lib.mz_device_count() == 0:
            raise RuntimeError("no sm_100 (B200) device visible; ultrazoom_b200 has no CPU or non-Blackwell fallback")
        self.device = device
        self.operand_dtype = operand_dtype
        cfg = _native.MzConfig(owner.upscale_ratio, owner.num_channels, owner.hidden_ratio,
                               owner.num_encoder_layers, owner.control_features, device.index or 0,
                               _native.dtype_code(operand_dtype), _native.STREAM_CODES[owner.residual_stream])
        handle = C.c_void_p()
        _native.check(self.lib.mz_model_create(C.byref(cfg), C.byref(handle)))
        self.handle = handle
        self.versions = None
        self.ws: Optional[Tensor] = None
        self.ws_stream = None          # the stream the workspace was allocated on
        self.last_stream = None        # cuda_stream of the previous call on this engine
        self.last_event: Optional[torch.cuda.Event] = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.mz_model_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def sync_weights(self, owner: "MewZoom") -> None:
        params = owner._flat_params()
        versions = tuple([(p.data_ptr(), p._version) for p in params])
        if versions == self.versions:
            return
        lib, h = self.lib, self.handle
        stream = torch.cuda.current_stream(self.device)
        on_device = False

        def put(kind: int, layer: int, t: Tensor) -> None:
            nonlocal on_device
            if t.is_cuda and t.device == self.device:
                # packed by a kernel on the current stream (mz_model_set_weight_dev): no round trip through the host
                a = t.detach().to(torch.float32).contiguous()
                _native.check(lib.mz_model_set_weight_dev(h, kind, layer, a.data_ptr(), a.numel(), stream.cuda_stream))
                on_device = True
            else:
                a = t.detach().to(device="cpu", dtype=torch.float32).contiguous()
                _native.check(lib.mz_model_set_weight(h, kind, layer, a.data_ptr(), a.numel()))

        with torch.cuda.device(self.device):
            put(_native.W_STEM_WEIGHT, 0, owner.stem.conv.weight)
            put(_native.W_STEM_BIAS, 0, owner.stem.conv.bias)
            for l, blk in enumerate(owner.encoder):
                put(_native.W_CONV1, l, blk.convnet.conv1.weight)
                put(_native.W_CONV2, l, blk.convnet.conv2.weight)
                if owner.control_features > 0:
                    put(_native.W_CTRL_WEIGHT, l, blk.control.linear.weight)
                    put(_native.W_CTRL_BIAS, l, blk.control.linear.bias)
            put(_native.W_HEAD, 0, owner.head.conv.weight)
            if on_device and self.operand_dtype == "float16" and not torch.cuda.is_current_stream_capturing():
                stream.synchronize()        # once per weight change: the device-side pack reports range errors by flag
                if self.saturated(reset=True):
                    raise AssertionError("a convolution weight exceeds the fp16 operand range (|w| > 65504 or not finite); "
                                         "build the model with operand_dtype='bfloat16' (or 'auto')")
        self.versions = versions

    def saturated(self, reset: bool = False) -> bool:
        """Has any COMPLETED kernel of this engine rounded a value beyond the fp16 range (mz_model_saturated)?"""
        flag = C.c_int32()
        _native.check(self.lib.mz_model_saturated(self.handle, 1 if reset else 0, C.byref(flag)))
        return bool(flag.value)

    def workspace(self, B: int, H: int, W: int, stream: "torch.cuda.Stream") -> Tensor:
        need = C.c_size_t()
        _native.check(self.lib.mz_workspace_bytes(self.handle, B, H, W, C.byref(need)))
        if self.ws is None or self.ws.numel() < need.value:
            self.ws = None     # (kernels still using the old buffer were recorded on it with record_stream)
            self.ws = torch.empty(need.value + 1024, dtype=torch.uint8, device=self.device)
            self.ws_stream = stream.cuda_stream
        elif stream.cuda_stream != self.ws_stream and not torch.cuda.is_current_stream_capturing():
            self.ws.record_stream(stream)
        return self.ws

    def begin(self, stream: "torch.cuda.Stream") -> None:
        """Order this call after the previous one when that ran on another stream (they share the workspace)."""
        if torch.cuda.is_current_stream_capturing():
            return      # (a capturing stream may not wait for an event recorded outside the capture; torch synchronises
                        # the device before a capture begins, so everything earlier has finished)
        if self.last_stream is not None and self.last_stream != stream.cuda_stream and self.last_event is not None:
            stream.wait_event(self.last_event)

    def end(self, stream: "torch.cuda.Stream") -> None:
        if torch.cuda.is_current_stream_capturing():
            return
        if self.last_event is None:
            self.last_event = torch.cuda.Event()
        self.last_event.record(stream)
        self.last_stream = stream.cuda_stream


class MewZoom(nn.Module, PyTorchModelHubMixin):
    """Fast single-image super-resolution with optional control conditioning (B200-native forward)."""

    AVAILABLE_UPSCALE_RATIOS = {2, 3, 4}

    AVAILABLE_HIDDEN_RATIOS = {1, 2, 4}

    def __init__(
        self,
        upscale_ratio: int,
        num_channels: int,
        hidden_ratio: int,
        num_encoder_layers: int,
        control_features: int = 0,
        operand_dtype: str = "float16",
        residual_stream: str = "auto",
    ):
        """``operand_dtype``: element type of the tensor-core operands ("float16" default, "bfloat16", or "auto").
        Both run at the same tcgen05 rate with fp32 accumulation; fp16's 10-bit mantissa keeps max|err| vs the fp32
        reference ~8x smaller (DESIGN.md, "Numerics"), but its range ends at 65504: every kernel that rounds a larger
        magnitude into an fp16 operand raises a flag (``saturated()``).  With "float16" a call that synchronises anyway
        (``upscale_host``, ``host_wait``, ``capture``) raises itself; every other call returns at once and the NEXT call
        on the model (any entry point, a graph's ``__call__`` included) raises -- a clipped result is never passed
        over in silence.  With "auto", ``forward``, ``upscale``, ``upscale_into`` and ``upscale_host`` are checked
        (one stream synchronisation) and a saturated one is re-run -- like all later calls -- with bfloat16 operands;
        stages, lanes and graphs cannot be re-run and raise as with "float16" (the model then runs with bfloat16).
        ``residual_stream``: "auto" | "float32" -- the residual stream lives in HBM as fp32 + a 16-bit shadow (the next
        block's tensor-core operand)."""
        super().__init__()
        if str(operand_dtype) != "auto":
            _native.dtype_code(operand_dtype)
        assert residual_stream in _native.STREAM_CODES, f"residual_stream must be one of {sorted(_native.STREAM_CODES)}"
        assert upscale_ratio in self.AVAILABLE_UPSCALE_RATIOS, (
            f"Upscale ratio must be one of {self.AVAILABLE_UPSCALE_RATIOS}, but got {upscale_ratio}.")
        assert hidden_ratio in self.AVAILABLE_HIDDEN_RATIOS, (
            f"Hidden ratio must be one of {self.AVAILABLE_HIDDEN_RATIOS}, but got {hidden_ratio}.")
        assert num_encoder_layers > 0, "Number of encoder layers must be greater than 0."
        assert control_features >= 0, "Control features must not be negative."

        self.stem = FanOutProjection(3, num_channels)
        self.encoder = nn.ModuleList(
            [EncoderBlock(num_channels, hidden_ratio, control_features) for _ in range(num_encoder_layers)])
        self.head = SubpixelConv2d(num_channels, 3, upscale_ratio)

        self.upscale_ratio = upscale_ratio
        self.num_channels = num_channels
        self.hidden_ratio = hidden_ratio
        self.num_encoder_layers = num_encoder_layers
        self.control_features = control_features
        self.operand_dtype = str(operand_dtype).replace("torch.", "")
        self.residual_stream = residual_stream
        self._engines: dict = {}
        self._flags_extra = 0
        self.u8_truncate = False          # uint8 results: floor(255 y) instead of floor(255 y + 0.5); not for uint16
        self._auto_dtype = "float16"      # operand_dtype="auto": what the next call runs with
        self._param_cache = None
        self._host_keep: dict = {}          # (device, lane) -> (engine, x, c, out) of the frame in flight on that lane
        self._host_clipped: set = set()     # (device, lane) whose frame was in flight when the range flag was found up

    # ---- reference model.py:94-115 ----
    @property
    def num_params(self) -> int:
        return sum(p.numel() for p in self.parameters())

    @property
    def num_trainable_params(self) -> int:
        return sum(p.numel() for p in self.parameters() if p.requires_grad)

    def freeze_parameters(self) -> None:
        for p in self.parameters():
            p.requires_grad = False

    # ---- reference model.py:117-139: checkpoints are written with weight-norm parametrizations in place ----
    def add_weight_norms(self) -> None:
        """Weight-normalise every convolution (stem, encoder, head), as the reference's training scripts do before
        ``load_state_dict`` (test_compare.py:36).  The kernels always see the baked ``weight``."""
        from torch.nn.utils.parametrizations import weight_norm
        from torch.nn.utils.parametrize import is_parametrized

        for module in self.modules():
            if isinstance(module, nn.Conv2d) and not is_parametrized(module):
                weight_norm(module)
        self._invalidate_params()

    def remove_parameterizations(self) -> None:
        """Bake and remove all parametrizations (reference model.py:131-139, called before ``eval()``)."""
        from torch.nn.utils.parametrize import is_parametrized, remove_parametrizations

        for module in self.modules():
            if is_parametrized(module):
                for name in list(module.parametrizations.keys()):
                    remove_parametrizations(module, name)
        self._invalidate_params()

    @staticmethod
    def convert_reference_state_dict(state_dict: dict) -> dict:
        """A reference training checkpoint's ``state_dict`` -> plain keys: strips the ``_orig_mod.`` prefixes of a
        compiled model (test_compare.py:38-41) and bakes weight-norm pairs ``parametrizations.weight.original0/1``
        (g, v) into ``weight = g * v / ||v||`` (norm over all dims but 0, as ``weight_norm(dim=0)`` defines it)."""
        sd = {k.replace("_orig_mod.", ""): v for k, v in state_dict.items()}
        out = {}
        for k, v in sd.items():
            if k.endswith(".parametrizations.weight.original0"):
                prefix = k[: -len(".parametrizations.weight.original0")]
                g, d = v.float(), sd[prefix + ".parametrizations.weight.original1"].float()
                norm = d.flatten(1).norm(dim=1).reshape(-1, *([1] * (d.dim() - 1)))
                out[prefix + ".weight"] = g * d / norm
            elif ".parametrizations." not in k:
                out[k] = v
        return out

    @classmethod
    def from_checkpoint(cls, checkpoint, **kwargs) -> "MewZoom":
        """Build a model from a reference training checkpoint -- a path or the loaded dict with ``upscaler_args`` and
        ``upscaler`` (test_compare.py:32-49) -- ready for ``.to("cuda").eval()``."""
        if not isinstance(checkpoint, dict):
            checkpoint = torch.load(checkpoint, map_location="cpu", weights_only=True)
        model = cls(**checkpoint["upscaler_args"], **kwargs)
        model.load_state_dict(cls.convert_reference_state_dict(checkpoint["upscaler"]))
        return model

    # ---- native plumbing ----
    def _flat_params(self) -> list:
        """The parameters as a flat list, cached: ``Module.parameters()`` walks the module tree on every call, which is
        most of the host time of a small frame.  Each entry remembers the ``_parameters`` dict and key it came from, so
        a replaced Parameter object (parametrizations, direct assignment) is noticed by an identity check."""
        cache = self._param_cache
        if cache is not None and all(d.get(n) is p for d, n, p in cache):
            return [p for _, _, p in cache]
        cache = [(m._parameters, n, p) for m in self.modules() for n, p in m._parameters.items() if p is not None]
        self._param_cache = cache
        return [p for _, _, p in cache]

    def _invalidate_params(self) -> None:
        self._param_cache = None
        for eng in self._engines.values():
            eng.versions = None

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self._invalidate_params()
        return out

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self._invalidate_params()
        return out

    def _operand_dtype_now(self) -> str:
        return self._auto_dtype if self.operand_dtype == "auto" else self.operand_dtype

    def _engine(self, device: torch.device, operand_dtype: Optional[str] = None) -> _Engine:
        dt = operand_dtype or self._operand_dtype_now()
        dt = "bfloat16" if _native.dtype_code(dt) == _native.DTYPE_BF16 else "float16"
        key = (device.type, device.index, dt)
        eng = self._engines.get(key)
        if eng is None:
            eng = _Engine(self, device, dt)
            self._engines[key] = eng
        eng.sync_weights(self)
        return eng

    def saturated(self, device: Optional[torch.device] = None, sync: bool = True, reset: bool = False) -> bool:
        """fp16 range guard: did a kernel round a magnitude beyond 65504 into an fp16 operand (the result of that call
        is then clipped, i.e. wrong)?  ``sync`` waits for the device first."""
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if sync:
            torch.cuda.synchronize(dev)
        eng = self._engines.get((dev.type, dev.index, "float16"))
        return eng.saturated(reset) if eng is not None else False

    def _range_guard(self, eng: _Engine, rerun: bool = False) -> bool:
        """The fp16 range policy of every entry point: True when no COMPLETED kernel of ``eng`` has clipped a value.

        Otherwise a result was clipped.  With "float16" this raises (the flag stays up until ``saturated(reset=True)``).
        With "auto" the model switches to bfloat16 operands for good and clears the flag; then a caller that can still
        repeat its own call (``rerun``: the flag is its own -- it synchronised the device before its launch -- and
        nothing clipped has reached the caller yet) gets False and repeats it, anyone else gets the error: a clipped
        result that was already handed out is never passed over silently.  The flag is one word per engine, so a frame
        still in flight on one of the engine's host lanes when it is found up is reported as clipped by its
        ``host_wait`` too."""
        if eng.operand_dtype != "float16" or not eng.saturated():
            return True
        if self.operand_dtype == "auto":
            eng.saturated(reset=True)
            self._auto_dtype = "bfloat16"
            if rerun:
                return False
        self._host_clipped.update(k for k, v in self._host_keep.items() if v[0] is eng)
        raise self._clipped_error()

    def _clipped_error(self) -> RuntimeError:
        if self.operand_dtype == "auto":
            return RuntimeError(
                "a call on this model rounded a value beyond the fp16 range (65504) into a tensor-core operand: its "
                "result was clipped.  The model now runs with bfloat16 operands ('auto'); repeat the call (a captured "
                "graph must be captured again).")
        return RuntimeError(
            "a call on this model rounded a value beyond the fp16 range (65504) into a tensor-core operand: its result "
            "was clipped.  Use operand_dtype='bfloat16' or 'auto' for this checkpoint (model.saturated(reset=True) "
            "clears the flag).")

    def set_conv_tune(self, which: int = -1, device: Optional[torch.device] = None, **kw) -> None:
        """Override the tcgen05 kernel's tunables (see mz_conv_tune); for benches and tests."""
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        eng = self._engine(dev)
        t = _native.tune(**kw)
        _native.check(eng.lib.mz_model_set_tune(eng.handle, which, C.byref(t)))

    def _image_flags(self, dtype: torch.dtype) -> int:
        """The element-type flags of an image: uint8 (rounded as ``u8_truncate`` says), uint16, or 0 for float32."""
        if dtype == torch.uint8:
            return _native.FLAG_IO_U8 | (_native.FLAG_U8_TRUNC if self.u8_truncate else 0)
        return _native.FLAG_IO_U16 if dtype == torch.uint16 else 0

    def _check_inputs(self, x: Tensor, c: Optional[Tensor]) -> Optional[Tensor]:
        assert x.dim() == 4 and x.shape[1] == 3, f"Expected input of shape (B, 3, H, W), got {tuple(x.shape)}."
        assert x.shape[0] > 0 and x.shape[2] > 0 and x.shape[3] > 0, "Input must not be empty."
        if self.control_features == 0:
            assert c is None, "This model has no control modules; c must be None."
            return None
        assert c is not None, "Control vector c is required for control models."
        if c.dim() == 1:
            c = c.unsqueeze(0)
        assert c.dim() == 2 and c.shape[1] == self.control_features, (
            f"Expected {self.control_features} control features, got {c.shape[-1]}.")
        assert c.shape[0] in (1, x.shape[0]), "Batch size of c must match x."
        return c

    def _run(self, x: Tensor, c: Optional[Tensor], flags: int, ws: Optional[Tensor] = None,
             memory_format=torch.contiguous_format) -> Tensor:
        c = self._check_inputs(x, c)
        if not x.is_cuda:
            raise RuntimeError("ultrazoom_b200.MewZoom runs on sm_100a CUDA kernels only; move the input to a "
                               "B200 (`x.cuda()`). There is no CPU fallback.")
        dev = x.device
        odt = x.dtype if x.dtype in _INT_IMAGE_DTYPES else torch.float32   # 8 / 16-bit images in and out: see upscale()
        if odt != torch.float32:
            assert flags & _native.FLAG_CLAMP01, (
                f"{str(odt).replace('torch.', '')} images are supported by upscale(), not forward()")
            flags |= self._image_flags(odt)
        x, xflag = _input_image(x, odt != torch.float32)
        flags |= xflag | _output_flag(memory_format)
        if c is not None:
            c = c.detach().to(device=dev, dtype=torch.float32).contiguous()
        B, _, H, W = x.shape
        r = self.upscale_ratio
        capturing = torch.cuda.is_current_stream_capturing()
        auto = self.operand_dtype == "auto" and not capturing
        while True:
            eng = self._engine(dev)
            if auto and eng.operand_dtype == "float16":
                torch.cuda.synchronize(dev)    # (the flag of an earlier asynchronous call is not this call's to absorb)
            if not capturing:
                self._range_guard(eng)
            y = torch.empty((B, 3, H * r, W * r), dtype=odt, device=dev, memory_format=memory_format)
            stream = torch.cuda.current_stream(dev)
            eng.begin(stream)
            w = ws if ws is not None else eng.workspace(B, H, W, stream)
            ws_ptr = (w.data_ptr() + 1023) // 1024 * 1024
            ws_bytes = w.numel() - (ws_ptr - w.data_ptr())
            _native.check(eng.lib.mz_upscale(
                eng.handle, x.data_ptr(), c.data_ptr() if c is not None else None,
                c.shape[0] if c is not None else 0, y.data_ptr(), B, H, W, ws_ptr, ws_bytes,
                flags | self._flags_extra, stream.cuda_stream))
            eng.end(stream)
            if auto and eng.operand_dtype == "float16":
                stream.synchronize()       # "auto": a saturated fp16 call is repeated with bfloat16 operands
                if not self._range_guard(eng, rerun=True):
                    continue
            return y

    # ---- reference model.py:149-179 ----
    def forward(self, x: Tensor, c: Optional[Tensor] = None, *, memory_format=torch.contiguous_format) -> Tensor:
        """bicubic(x) + residual network, un-clamped (reference model.py:149-164).  See ``upscale`` for the layouts."""
        return self._run(x, c, 0, memory_format=memory_format)

    @torch.inference_mode()
    def upscale(self, x: Tensor, c: Optional[Tensor] = None, *, memory_format=torch.contiguous_format) -> Tensor:
        """``clamp(forward(x, c), 0, 1)`` (reference model.py:166-179); the clamp is fused in the head kernel.

        A ``torch.uint8`` image (what ``decode_image`` returns, reference test_compare.py:53) is read as ``x / 255``
        (``ToDtype(float32, scale=True)``, test_compare.py:55-57) and the result comes back as uint8,
        ``floor(255 * y + 0.5)`` as ``save_image`` writes it (test_compare.py:89) -- or ``floor(255 * y)`` as
        ``ToPILImage`` does (README.md:81) when ``model.u8_truncate`` is set: a quarter of the image traffic.
        A ``torch.uint16`` image (16-bit PNG / TIFF, 10/12-bit video decoded to rgb48le) is read as ``x / 65535``, the
        exact quotient, and comes back as uint16, ``floor(65535 * y + 0.5)``: the fp32 result on ``x.float() / 65535``,
        quantised, at half the image traffic.  ``u8_truncate`` does not apply to it.

        Interleaved images need no transpose on either side: an ``x`` in ``channels_last`` strides (and not also plainly
        contiguous), e.g. ``torch.from_numpy(hwc_frames).permute(0, 3, 1, 2)``, is read as it is, and
        ``memory_format=torch.channels_last`` returns ``y`` in channels-last strides, so ``y.permute(0, 2, 3, 1)`` is a
        contiguous (B,rH,rW,3) array.  The default output is contiguous NCHW whatever the input's layout.  The results
        are bit-identical in every layout."""
        return self._run(x, c, _native.FLAG_CLAMP01, memory_format=memory_format)

    @torch.inference_mode()
    def test_compare(self, x: Tensor, c: Optional[Tensor] = None):
        """``(upscale(x, c), bicubic(x))``, both clamped to [0, 1]: what the reference's evaluation script asks of the
        0.2.x model (validate.py:97).  The bicubic image comes from the stand-alone bicubic kernel (mz_bicubic_f32)."""
        from . import ops

        scale = {torch.uint8: 255.0, torch.uint16: 65535.0}.get(x.dtype)
        return self.upscale(x, c), ops.bicubic(x.float() if scale is None else x.float() / scale,
                                               self.upscale_ratio).clamp_(0, 1)

    @torch.inference_mode()
    def upscale_into(self, x: Tensor, c: Optional[Tensor], frame: Tensor, window: tuple, at: tuple) -> None:
        """Halo-tiled inference without a tile output: ``upscale`` the LR tile ``x`` and write only its core -- the LR
        pixels ``window = (y0, y1, x0, x1)`` of the tile -- straight into ``frame`` (B,3,rH',rW'), whose HR pixel
        ``at = (fy, fx)`` receives the core's first pixel (mz_upscale_window).  ``frame`` may live on another GPU
        (``sharding.share_frame``): the head kernel's stores are then the transfer over NVLink.  ``frame`` is planar or
        interleaved (channels-last strides, any row and image pitch, e.g. a view into a wider HWC buffer)."""
        c = self._check_inputs(x, c)
        if not x.is_cuda:
            raise RuntimeError("ultrazoom_b200.MewZoom runs on sm_100a CUDA kernels only (no CPU fallback).")
        dev = x.device
        eng = self._engine(dev)
        auto = self.operand_dtype == "auto" and eng.operand_dtype == "float16"
        if auto:
            torch.cuda.synchronize(dev)        # (as in upscale: only this call's flag may be absorbed by its re-run)
        self._range_guard(eng)
        x_in, c_in = x, c
        odt = x.dtype if x.dtype in _INT_IMAGE_DTYPES else torch.float32
        flags = _native.FLAG_CLAMP01 | self._flags_extra | self._image_flags(odt)
        x, xflag = _input_image(x, odt != torch.float32)
        if c is not None:
            c = c.detach().to(device=dev, dtype=torch.float32).contiguous()
        B, _, H, W = x.shape
        r = self.upscale_ratio
        y0, y1, x0, x1 = window
        fy, fx = at
        assert frame.is_cuda and frame.dim() == 4 and frame.shape[0] == B and frame.shape[1] == 3, "frame must be (B,3,H',W')"
        assert frame.dtype == odt, f"frame must be {odt} for a {odt} input, got {frame.dtype}"
        yflag, row_pitch, img_pitch = _frame_layout(frame)
        flags |= xflag | yflag
        assert 0 <= fy and fy + (y1 - y0) * r <= frame.shape[2] and 0 <= fx and fx + (x1 - x0) * r <= frame.shape[3], (
            "the window does not fit into the frame at that position")
        if frame.device != dev:
            _native.check(eng.lib.mz_enable_peer_access(dev.index or 0, frame.device.index or 0))
        stream = torch.cuda.current_stream(dev)
        eng.begin(stream)
        ws = eng.workspace(B, H, W, stream)
        ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
        dst = frame[0, 0, fy, fx].data_ptr() if frame.numel() else 0
        _native.check(eng.lib.mz_upscale_window(
            eng.handle, x.data_ptr(), c.data_ptr() if c is not None else None, c.shape[0] if c is not None else 0,
            dst, row_pitch, img_pitch, B, H, W, y0, y1, x0, x1, ws_ptr,
            ws.numel() - (ws_ptr - ws.data_ptr()), flags, stream.cuda_stream))
        eng.end(stream)
        if auto:
            stream.synchronize()          # as in upscale: a saturated window is written again with bfloat16 operands
            if not self._range_guard(eng, rerun=True):
                self.upscale_into(x_in, c_in, frame, window, at)

    @torch.inference_mode()
    def upscale_stage(self, x: Tensor, c: Optional[Tensor], frame: Tensor, window: tuple, at: tuple, layer_begin: int,
                      layer_end: int, ws: Tensor) -> None:
        """``upscale_into`` cut into stages along the depth of the network (mz_upscale_stage): run the encoder blocks
        ``[layer_begin, layer_end)`` on the state kept in the caller's workspace ``ws`` (``stage_workspace``); the stem
        runs first when ``layer_begin == 0``, the head -- storing the window into ``frame`` -- last when ``layer_end ==
        num_encoder_layers``.  Between stages ``sharding.upscale_tiled_refresh`` overwrites the tile's halo with the
        neighbours' values (``stage_views``)."""
        c = self._check_inputs(x, c)
        assert x.is_cuda and x.dtype in (torch.float32, torch.uint8, torch.uint16), (
            "upscale_stage takes a CUDA image (float32, uint8 or uint16)")
        dev = x.device
        eng = self._engine(dev)
        self._range_guard(eng)            # (stages run asynchronously: a saturated stage is reported by the next call)
        integer = x.dtype in _INT_IMAGE_DTYPES
        flags = _native.FLAG_CLAMP01 | self._flags_extra | self._image_flags(x.dtype)
        x, xflag = _input_image(x, integer)
        if c is not None:
            c = c.detach().to(device=dev, dtype=torch.float32).contiguous()
        B, _, H, W = x.shape
        r = self.upscale_ratio
        y0, y1, x0, x1 = window
        fy, fx = at
        assert frame.is_cuda and frame.dim() == 4 and frame.shape[0] == B and frame.shape[1] == 3
        yflag, row_pitch, img_pitch = _frame_layout(frame)
        flags |= xflag | yflag
        if frame.device != dev:
            _native.check(eng.lib.mz_enable_peer_access(dev.index or 0, frame.device.index or 0))
        stream = torch.cuda.current_stream(dev)
        ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
        dst = frame[0, 0, fy, fx].data_ptr()
        _native.check(eng.lib.mz_upscale_stage(
            eng.handle, x.data_ptr(), c.data_ptr() if c is not None else None, c.shape[0] if c is not None else 0,
            dst, row_pitch, img_pitch, B, H, W, y0, y1, x0, x1, ws_ptr, ws.numel() - (ws_ptr - ws.data_ptr()),
            flags, stream.cuda_stream, layer_begin, layer_end))

    def stage_workspace(self, shape, device: torch.device) -> Tensor:
        """A private workspace for ``upscale_stage`` calls on a (B,3,H,W) tile (the state between stages lives in it)."""
        eng = self._engine(torch.device(device))
        need = C.c_size_t()
        _native.check(eng.lib.mz_workspace_bytes(eng.handle, shape[0], shape[2], shape[3], C.byref(need)))
        return torch.empty(need.value + 1024, dtype=torch.uint8, device=device)

    def stage_views(self, ws: Tensor, shape, blocks_done: int):
        """``(zf, z16)``: the fp32 residual stream (B,H,W,Cp) and its 16-bit shadow (B,H,W,pitch) inside ``ws`` after
        ``blocks_done`` encoder blocks, as tensors sharing the workspace's memory (mz_workspace_layout)."""
        eng = self._engine(ws.device)
        B, _, H, W = shape
        zf_o, zb_o, hid_o = C.c_size_t(), C.c_size_t(), C.c_size_t()
        cp, zp = C.c_int32(), C.c_int32()
        _native.check(eng.lib.mz_workspace_layout(eng.handle, B, H, W, C.byref(zf_o), C.byref(zb_o), C.byref(hid_o),
                                                  C.byref(cp), C.byref(zp)))
        base = (ws.data_ptr() + 1023) // 1024 * 1024 - ws.data_ptr()
        npix = B * H * W
        dt16 = torch.bfloat16 if eng.operand_dtype == "bfloat16" else torch.float16
        zf = ws[base + zf_o.value: base + zf_o.value + npix * cp.value * 4].view(torch.float32).view(B, H, W, cp.value)
        in_hidden = bool(eng.lib.mz_model_fused_block(eng.handle)) and (blocks_done & 1)
        off, pitch = (hid_o.value, cp.value) if in_hidden else (zb_o.value, zp.value)
        z16 = ws[base + off: base + off + npix * pitch * 2].view(dt16).view(B, H, W, pitch)
        return zf, z16

    def capture(self, x: Tensor, c: Optional[Tensor] = None, clamp: bool = True, *,
                memory_format=torch.contiguous_format) -> "GraphedUpscale":
        """Record one ``upscale`` (``clamp=False``: ``forward``) call at the shape of ``x`` into a CUDA graph.

        A frame of a few hundred pixels a side is launch-bound (2L + 3 kernels, most of them cluster launches of
        15-20 us of host time each); replaying the recorded graph removes the host from that loop.  The dependent-launch
        edges between the kernels are kept by the capture.  The graph reads its input in the layout of ``x`` and writes
        its output in ``memory_format`` (see ``upscale``).  See ``GraphedUpscale``."""
        return GraphedUpscale(self, x, c, _native.FLAG_CLAMP01 if clamp else 0, memory_format)

    @torch.inference_mode()
    def upscale_host(self, x: Tensor, c: Optional[Tensor] = None, out: Optional[Tensor] = None,
                     device: int = 0, lane: Optional[int] = None, *, memory_format=torch.contiguous_format) -> Tensor:
        """End-to-end call with HOST tensors: H2D copy, kernels, D2H copy (mz_upscale_host).

        ``lane=None``: synchronous; a batch is cut into chunks whose copies overlap the kernels of their neighbours.
        ``lane=0|1``: frame-stream form (mz_upscale_host_async) -- the call only enqueues and returns ``out`` at once;
        ``out`` is valid after ``host_wait(lane)``.  Alternating lanes double-buffers a stream of frames.  ``x``, ``c``
        and ``out`` should be pinned and must not be touched until the wait.  A frame clipped to the fp16 range raises
        in the synchronous call itself ("auto": it is repeated with bfloat16 operands), on a lane at ``host_wait``.

        Element types and layouts as in ``upscale`` (uint8 and uint16 frames come back as such): a channels-last ``x`` is
        copied as it is (no transpose on the CPU), and the result is interleaved with
        ``memory_format=torch.channels_last``.  A caller's ``out`` sets the output layout itself: it must be contiguous
        NCHW or contiguous channels-last, of the input's element type."""
        c = self._check_inputs(x, c)
        assert not x.is_cuda, "upscale_host takes host tensors"
        assert lane in (None, 0, 1), "lane must be None, 0 or 1"
        eng = self._engine(torch.device("cuda", device))
        if lane is None and self.operand_dtype == "auto" and eng.operand_dtype == "float16":
            torch.cuda.synchronize(torch.device("cuda", device))   # (as in upscale; lanes included)
        self._range_guard(eng)
        odt = x.dtype if x.dtype in _INT_IMAGE_DTYPES else torch.float32
        x, xflag = _input_image(x, odt != torch.float32)
        if c is not None:
            c = c.to(device="cpu", dtype=torch.float32).contiguous()
        B, _, H, W = x.shape
        r = self.upscale_ratio
        if out is None:
            out = torch.empty((B, 3, H * r, W * r), dtype=odt, memory_format=memory_format)
            yflag = _output_flag(memory_format)
        else:
            yflag = _native.FLAG_Y_NHWC if _is_nhwc(out) else 0
            assert out.is_contiguous() or yflag, "out must be contiguous NCHW or contiguous channels-last"
        assert tuple(out.shape) == (B, 3, H * r, W * r) and out.dtype == odt
        flags = _native.FLAG_CLAMP01 | self._flags_extra | xflag | yflag | self._image_flags(odt)
        cp, cr = (c.data_ptr(), c.shape[0]) if c is not None else (None, 0)
        if lane is None:
            _native.check(eng.lib.mz_upscale_host(eng.handle, x.data_ptr(), cp, cr, out.data_ptr(), B, H, W, flags))
            if not self._range_guard(eng, rerun=True):     # (the call has synchronised: "auto" repeats it with bf16)
                return self.upscale_host(x, c, out, device)
        else:
            # keep the (possibly converted) inputs alive until the wait, and the engine whose lane runs the frame
            self._host_keep[(device, lane)] = (eng, x, c, out)
            _native.check(eng.lib.mz_upscale_host_async(eng.handle, lane, x.data_ptr(), cp, cr, out.data_ptr(), B, H, W,
                                                        flags))
        return out

    def host_wait(self, lane: int = -1, device: int = 0) -> None:
        """Block until the frames enqueued with ``upscale_host(..., lane=...)`` on that lane (-1: both) are done; raises
        when one of them was clipped to the fp16 range (see ``_range_guard``).  It waits on the engine that ran each
        frame, which is not the current one when "auto" has switched to bfloat16 since the frame was enqueued."""
        lanes = (0, 1) if lane < 0 else (lane,)
        done = [self._host_keep.pop((device, ln)) for ln in lanes if (device, ln) in self._host_keep]
        engines = list({id(d[0]): d[0] for d in done}.values()) or [self._engine(torch.device("cuda", device))]
        for eng in engines:
            _native.check(eng.lib.mz_upscale_host_wait(eng.handle, lane))
        clipped = any((device, ln) in self._host_clipped for ln in lanes)
        self._host_clipped.difference_update((device, ln) for ln in lanes)
        for eng in engines:
            self._range_guard(eng)
        if clipped:
            raise self._clipped_error()


class GraphedUpscale:
    """``MewZoom.capture``: a CUDA graph of the whole call with fixed input and output buffers.

    ``g = model.capture(x, c); y = g(x2, c2)`` copies ``x2``/``c2`` (same shapes and dtypes as at capture) into the
    graph's input buffers, replays it on the current stream and returns the graph's output tensor ``g.y`` -- the same
    tensor on every call, so consume or clone it before the next replay.  ``g.replay()`` skips the copies (fill
    ``g.x`` / ``g.c`` yourself).  The graph reads the engine's packed weights in place: parameters changed after the
    capture are picked up by the next ordinary call (which re-packs them), not by a replay on its own."""

    def __init__(self, model: MewZoom, x: Tensor, c: Optional[Tensor], flags: int,
                 memory_format=torch.contiguous_format):
        c = model._check_inputs(x, c)
        if not x.is_cuda:
            raise RuntimeError("MewZoom.capture needs a CUDA input (there is no CPU fallback).")
        self.model = model
        # (the input buffer keeps the layout of x: the graph reads it as _run reads x; a replay copies either layout in)
        self.x = _input_image(x, x.dtype in _INT_IMAGE_DTYPES)[0].clone()
        self.c = None if c is None else c.detach().to(device=x.device, dtype=torch.float32).contiguous().clone()
        # The graph bakes in raw pointers: it owns everything they point at -- its input / output tensors, a PRIVATE
        # workspace (the engine's cached one is dropped and re-allocated when a later call needs a larger one) and the
        # engine itself (packed weights, FiLM parameters): the one the warm-up left current, which "auto" may have
        # switched to bfloat16.
        eng = model._engine(x.device)
        need = C.c_size_t()
        B, _, H, W = self.x.shape
        _native.check(eng.lib.mz_workspace_bytes(eng.handle, B, H, W, C.byref(need)))
        self.ws = torch.empty(need.value + 1024, dtype=torch.uint8, device=x.device)
        with torch.inference_mode():
            side = torch.cuda.Stream(device=x.device)
            side.wait_stream(torch.cuda.current_stream(x.device))
            with torch.cuda.stream(side):        # warm-up: packs the weights, prepares the launches
                model._run(self.x, self.c, flags, ws=self.ws, memory_format=memory_format)
            side.synchronize()
            self.engine = model._engine(x.device)
            model._range_guard(self.engine)      # a checkpoint that saturates is not recorded
            torch.cuda.current_stream(x.device).wait_stream(side)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.y = model._run(self.x, self.c, flags, ws=self.ws, memory_format=memory_format)

    def replay(self) -> Tensor:
        """Replay as it is: the 3-5 us path, so it does not consult the fp16 range flag.  A clipped replay is reported
        by the next ``__call__`` or call on the model, or read with ``model.saturated()``."""
        self.graph.replay()
        return self.y

    def __call__(self, x: Tensor, c: Optional[Tensor] = None) -> Tensor:
        """Copy ``x`` / ``c`` in and replay; raises first when an earlier replay was clipped to the fp16 range."""
        self.model._range_guard(self.engine)
        integer = x.dtype in _INT_IMAGE_DTYPES
        assert tuple(x.shape) == tuple(self.x.shape) and (x.dtype == self.x.dtype if integer else self.x.dtype == torch.float32), (
            f"Graph was captured for input {tuple(self.x.shape)} {self.x.dtype}, got {tuple(x.shape)} {x.dtype}.")
        self.x.copy_(x, non_blocking=True)
        if self.c is not None:
            assert c is not None, "Control vector c is required for control models."
            self.c.copy_(c.reshape(-1, self.c.shape[1]).expand_as(self.c), non_blocking=True)
        return self.replay()


class ONNXModel(nn.Module):
    """Wrapper whose forward is ``model.upscale`` (reference model.py:195-209)."""

    def __init__(self, model: MewZoom):
        super().__init__()
        self.model = model

    def forward(self, x: Tensor, c: Optional[Tensor] = None) -> Tensor:
        return self.model.upscale(x, c)
