"""ctypes binding of the C ABI in include/mewzoom_b200.h.

There is no fallback: if the shared library is missing it is built with nvcc, and if that fails, or
no sm_100 device is visible when a compute entry point is called, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmewzoom_b200.so")

ABI_VERSION = 4

MZ_OK = 0
MZ_ERR_INVALID = -1
MZ_ERR_CUDA = -2
MZ_ERR_UNSUPPORTED = -3
MZ_ERR_WORKSPACE = -4
MZ_ERR_STATE = -5

FLAG_CLAMP01 = 1
FLAG_SIMT_CONV = 2
FLAG_SKIP_FROM_BUFFER = 4
FLAG_IO_U8 = 8
FLAG_U8_TRUNC = 16
FLAG_X_NHWC = 32
FLAG_Y_NHWC = 64
FLAG_IO_U16 = 128

DTYPE_F16, DTYPE_BF16 = 0, 1
MATH_TF32, MATH_FP32 = 0, 1

W_STEM_WEIGHT, W_STEM_BIAS, W_CONV1, W_CONV2, W_CTRL_WEIGHT, W_CTRL_BIAS, W_HEAD = range(7)


STREAM_AUTO, STREAM_FP32 = 0, 1
STREAM_CODES = {"auto": STREAM_AUTO, "float32": STREAM_FP32}


class MzConfig(C.Structure):
    _fields_ = [
        ("upscale_ratio", C.c_int32),
        ("num_channels", C.c_int32),
        ("hidden_ratio", C.c_int32),
        ("num_encoder_layers", C.c_int32),
        ("control_features", C.c_int32),
        ("device", C.c_int32),
        ("operand_dtype", C.c_int32),
        ("residual_stream", C.c_int32),
    ]


class MzConvTune(C.Structure):
    _fields_ = [
        ("rows", C.c_int32),
        ("acc_stages", C.c_int32),
        ("kc", C.c_int32),
        ("halo_mode", C.c_int32),
        ("b_stages", C.c_int32),
        ("a_stages", C.c_int32),
        ("max_ctas", C.c_int32),
        ("cluster", C.c_int32),
        ("dbg", C.c_int32),
        ("pair", C.c_int32),
        ("resident", C.c_int32),
        ("epi_warps", C.c_int32),
        ("fuse", C.c_int32),
        ("block", C.c_int32),
        ("seg_rows", C.c_int32),
    ]


# name -> (restype, argtypes); every symbol include/mewzoom_b200.h declares.
_P = C.c_void_p
_I = C.c_int32
SIGNATURES = {
    "mz_last_error": (C.c_char_p, []),
    "mz_abi_version": (C.c_int, []),
    "mz_device_count": (C.c_int, []),
    "mz_model_create": (C.c_int, [C.POINTER(MzConfig), C.POINTER(_P)]),
    "mz_model_destroy": (None, [_P]),
    "mz_model_set_weight": (C.c_int, [_P, _I, _I, _P, C.c_size_t]),
    "mz_model_set_weight_dev": (C.c_int, [_P, _I, _I, _P, C.c_size_t, _P]),
    "mz_model_saturated": (C.c_int, [_P, _I, C.POINTER(_I)]),
    "mz_model_set_tune": (C.c_int, [_P, _I, C.POINTER(MzConvTune)]),
    "mz_model_enable_timing": (C.c_int, [_P, _I]),
    "mz_model_conv_stack_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "mz_workspace_bytes": (C.c_int, [_P, _I, _I, _I, C.POINTER(C.c_size_t)]),
    "mz_model_fused_block": (C.c_int, [_P]),
    "mz_block_fused": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "mz_upscale": (C.c_int, [_P, _P, _P, _I, _P, _I, _I, _I, _P, C.c_size_t, C.c_uint32, _P]),
    "mz_upscale_window": (C.c_int, [_P, _P, _P, _I, _P, C.c_int64, C.c_int64, _I, _I, _I, _I, _I, _I, _I, _P, C.c_size_t,
                                    C.c_uint32, _P]),
    "mz_upscale_stage": (C.c_int, [_P, _P, _P, _I, _P, C.c_int64, C.c_int64, _I, _I, _I, _I, _I, _I, _I, _P, C.c_size_t,
                                   C.c_uint32, _P, _I, _I]),
    "mz_workspace_layout": (C.c_int, [_P, _I, _I, _I, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t),
                                      C.POINTER(_I), C.POINTER(_I)]),
    "mz_enable_peer_access": (C.c_int, [_I, _I]),
    "mz_ipc_frame_create": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p), _P]),
    "mz_ipc_frame_open": (C.c_int, [_P, C.POINTER(C.c_void_p)]),
    "mz_ipc_frame_close": (C.c_int, [_P, _I]),
    "mz_upscale_host": (C.c_int, [_P, _P, _P, _I, _P, _I, _I, _I, C.c_uint32]),
    "mz_upscale_host_async": (C.c_int, [_P, _I, _P, _P, _I, _P, _I, _I, _I, C.c_uint32]),
    "mz_upscale_host_wait": (C.c_int, [_P, _I]),
    "mz_put_plane_async": (C.c_int, [_P, C.c_size_t, _P, C.c_size_t, C.c_size_t, C.c_size_t, _P]),
    "mz_bicubic_f32": (C.c_int, [_P, _P, _I, _I, _I, _I, _P]),
    "mz_stem_pack": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "mz_conv3x3": (C.c_int, [_P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, C.POINTER(MzConvTune), _P]),
    "mz_head_shuffle_add": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, C.POINTER(MzConvTune), _P]),
    "mz_pack_conv_weight": (C.c_int, [_P, _I, _I, _I, _I, _I, _P, C.POINTER(C.c_size_t)]),
    "mz_control_film": (C.c_int, [_P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "mz_adaptive_mix": (C.c_int, [_P, _P, _P, C.c_float, _P, _P, C.c_int64, _I, _I, _I, _I, _P]),
    "mz_pixel_crush": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "mz_quality_assessor": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "mz_pixel_shuffle_nhwc": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "mz_crop_feature_maps": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P]),
    "mz_probe_umma": (C.c_int, [_I, _I, _I, C.POINTER(C.c_float)]),
    "mz_probe_set_gap": (C.c_int, [_I, _I, _I]),
    "mz_probe_mma_rate": (C.c_int, [_I, _I, _I, _I, _I, _I, _I, C.POINTER(C.c_float)]),
    "mz_padded_channels": (C.c_int, [_I]),
    "mz_zb_pitch": (C.c_int, [_I]),
}

_lib = None
_lock = threading.Lock()


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first if necessary) the native library; raises RuntimeError on failure."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if build_if_missing:
            # build() is a digest comparison when the library is current: a stale .so after an edit under csrc/ is
            # rebuilt instead of loaded silently.  One process per GPU (torchrun): an inter-process lock keeps the
            # ranks from running nvcc into the same objects at once.  Without nvcc (a deployment box) a library that
            # is already there is loaded as it is.
            from . import build as _build

            try:
                _build.build_locked()
            except RuntimeError:
                if not os.path.exists(LIB_PATH):
                    raise
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing; run `python -m ultrazoom_b200.build`")
        try:
            lib = C.CDLL(LIB_PATH)
        except OSError as e:  # pragma: no cover - depends on the box
            raise RuntimeError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError => the library is stale
            fn.restype = res
            fn.argtypes = args
        if lib.mz_abi_version() != ABI_VERSION:
            raise RuntimeError(f"ABI mismatch: library reports {lib.mz_abi_version()}, binding expects {ABI_VERSION}")
        _lib = lib
        return lib


def last_error() -> str:
    return load().mz_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Non-zero status -> exception.  MZ_ERR_INVALID mirrors the reference's assert-style validation."""
    if rc == MZ_OK:
        return
    msg = last_error()
    if rc == MZ_ERR_INVALID:
        raise AssertionError(msg)
    raise RuntimeError(f"mewzoom_b200 error {rc}: {msg}")


def dtype_code(dt) -> int:
    """torch.float16 / 'f16' -> MZ_DTYPE_F16, torch.bfloat16 / 'bf16' -> MZ_DTYPE_BF16."""
    name = str(dt).replace("torch.", "")
    if name in ("float16", "f16", "fp16", "half"):
        return DTYPE_F16
    if name in ("bfloat16", "bf16"):
        return DTYPE_BF16
    raise AssertionError(f"Operand dtype must be float16 or bfloat16, {dt} given.")


def tune(**kw) -> MzConvTune:
    t = MzConvTune()
    for k, v in kw.items():
        setattr(t, k, int(v))
    return t
