"""CPU: the C-ABI library loads and exports every symbol include/mewzoom_b200.h declares (no compute
calls without a GPU), the Python boundary mirrors the reference's API and fails loudly without a B200."""
import ctypes
import os
import re

import pytest
import torch

from oracle import MODEL_CONFIGS as ORACLE_CONFIGS
from oracle import OracleMewZoom, make_oracle
from ultrazoom_b200 import MODEL_CONFIGS, ControlVector, MewZoom, ONNXModel, _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "mewzoom_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mz_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _native.load()
    names = _declared_symbols()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"
        assert n in _native.SIGNATURES, f"{n} has no ctypes signature"
    assert sorted(_native.SIGNATURES) == names
    assert lib.mz_abi_version() == _native.ABI_VERSION == 4


def test_padded_channels_and_error_plumbing():
    lib = _native.load()
    assert [lib.mz_padded_channels(c) for c in (48, 54, 96, 108, 192, 12, 27)] == [48, 64, 96, 128, 192, 16, 32]
    # invalid config -> MZ_ERR_INVALID with the reference's assertion wording (model.py:67-69)
    cfg = _native.MzConfig(5, 48, 2, 20, 0, 0, 0, 0)
    h = ctypes.c_void_p()
    rc = lib.mz_model_create(ctypes.byref(cfg), ctypes.byref(h))
    assert rc == _native.MZ_ERR_INVALID
    assert "Upscale ratio" in _native.last_error()
    with pytest.raises(AssertionError):
        _native.check(rc)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_gpu_fails_loudly_no_fallback():
    lib = _native.load()
    assert lib.mz_device_count() == 0
    cfg = _native.MzConfig(2, 48, 2, 20, 0, 0, 0, 0)
    h = ctypes.c_void_p()
    rc = lib.mz_model_create(ctypes.byref(cfg), ctypes.byref(h))
    assert rc in (_native.MZ_ERR_CUDA, _native.MZ_ERR_INVALID, _native.MZ_ERR_UNSUPPORTED) and not h.value
    m = MewZoom(**MODEL_CONFIGS["MewZoom-2X"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.upscale(torch.rand(1, 3, 8, 8))


def test_constructor_validation_matches_reference():
    with pytest.raises(AssertionError):
        MewZoom(5, 48, 2, 20)           # reference tests/test_model.py:69-73
    with pytest.raises(AssertionError):
        MewZoom(2, 48, 3, 20)           # model.py:738
    with pytest.raises(AssertionError):
        MewZoom(2, 48, 2, 0)
    with pytest.raises(AssertionError):
        MewZoom(2, 2, 2, 1)             # FanOutProjection model.py:218-222
    m = MewZoom(2, 16, 2, 2, control_features=3)
    x = torch.rand(2, 3, 8, 8)
    with pytest.raises(AssertionError):
        m._check_inputs(x, torch.rand(3, 3))      # tests/test_model.py:97-103
    with pytest.raises(AssertionError):
        m._check_inputs(x, torch.rand(2, 4))
    with pytest.raises(AssertionError):
        m._check_inputs(x, None)
    with pytest.raises(AssertionError):
        m._check_inputs(torch.rand(2, 1, 8, 8), torch.rand(2, 3))
    assert m._check_inputs(x, torch.rand(3)).shape == (1, 3)
    with pytest.raises(AssertionError):
        MewZoom(2, 16, 2, 2)._check_inputs(x, torch.rand(2, 3))


@pytest.mark.parametrize("name", sorted(MODEL_CONFIGS))
def test_state_dict_is_interchangeable_with_oracle(name):
    assert MODEL_CONFIGS[name] == ORACLE_CONFIGS[name]
    torch.manual_seed(0)
    m = MewZoom(**MODEL_CONFIGS[name])
    o = make_oracle(name, seed=0)
    sd_m, sd_o = m.state_dict(), o.state_dict()
    assert list(sd_m.keys()) == list(sd_o.keys())
    for k in sd_m:
        assert torch.equal(sd_m[k], sd_o[k]), k      # same default init, same construction order
    assert m.num_params == sum(p.numel() for p in o.parameters())
    assert m.num_trainable_params == m.num_params
    m.freeze_parameters()
    assert m.num_trainable_params == 0
    assert m.upscale_ratio == MODEL_CONFIGS[name]["upscale_ratio"]


def test_save_and_from_pretrained_round_trip(tmp_path):
    torch.manual_seed(3)
    m = MewZoom(3, 16, 2, 2, control_features=3)
    m.save_pretrained(str(tmp_path))
    assert (tmp_path / "config.json").exists() and (tmp_path / "model.safetensors").exists()
    m2 = MewZoom.from_pretrained(str(tmp_path))
    assert m2.upscale_ratio == 3 and m2.control_features == 3 and m2.num_encoder_layers == 2
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)


def test_control_vector():
    c = ControlVector(gaussian_blur=0.5, gaussian_noise=0.2, jpeg_compression=0.3).to_tensor()   # README.md:118-122
    assert c.dtype == torch.float32 and c.shape == (3,)
    assert c.tolist() == pytest.approx([0.5, 0.2, 0.3])
    with pytest.raises(AssertionError):
        ControlVector(gaussian_noise=-0.1)
    assert isinstance(ONNXModel(MewZoom(2, 16, 2, 1)), torch.nn.Module)


def test_reference_checkpoint_recipes():
    """The reference's loading recipe (test_compare.py:32-49: add_weight_norms -> load_state_dict of a compiled,
    weight-normed state dict -> remove_parameterizations) works on this class, and from_checkpoint does it in one."""
    torch.manual_seed(3)
    cfg = dict(upscale_ratio=2, num_channels=16, hidden_ratio=2, num_encoder_layers=2, control_features=3)
    trained = MewZoom(**cfg)
    trained.add_weight_norms()
    with torch.no_grad():
        for p in trained.parameters():
            p.add_(0.05 * torch.randn_like(p))
    baked = {k: v.detach().clone() for k, v in
             {"stem": trained.stem.conv.weight, "c1": trained.encoder[1].convnet.conv1.weight,
              "head": trained.head.conv.weight}.items()}
    ckpt = {"upscaler_args": cfg, "upscaler": {"_orig_mod." + k: v for k, v in trained.state_dict().items()}}
    assert any("parametrizations.weight.original0" in k for k in ckpt["upscaler"])

    # the reference's own sequence
    m = MewZoom(**ckpt["upscaler_args"])
    m.add_weight_norms()
    sd = dict(ckpt["upscaler"])
    for key in list(sd.keys()):
        sd[key.replace("_orig_mod.", "")] = sd.pop(key)
    m.load_state_dict(sd)
    m.remove_parameterizations()
    m.eval()
    assert not any("parametrizations" in k for k in m.state_dict())
    assert torch.allclose(m.stem.conv.weight, baked["stem"], atol=1e-6)
    assert torch.allclose(m.encoder[1].convnet.conv1.weight, baked["c1"], atol=1e-6)

    # one call
    m2 = MewZoom.from_checkpoint(ckpt)
    assert torch.allclose(m2.head.conv.weight, baked["head"], atol=1e-6)
    assert torch.allclose(m2.encoder[1].convnet.conv1.weight, baked["c1"], atol=1e-6)
    assert torch.equal(m2.encoder[0].control.linear.bias, trained.encoder[0].control.linear.bias)
    assert sorted(m2.state_dict()) == sorted(MewZoom(**cfg).state_dict())


def test_reference_import_paths_work_verbatim():
    """Reference README.md:69,102-103: `from ultrazoom.model import MewZoom`, `from ultrazoom.control import
    ControlVector` resolve to the B200-native classes (the `ultrazoom/` shim package)."""
    from ultrazoom.control import ControlVector as RefCV
    from ultrazoom.model import MewZoom as RefMewZoom
    from ultrazoom.model import ONNXModel as RefONNX

    assert RefMewZoom is MewZoom and RefCV is ControlVector and RefONNX is ONNXModel
    c = RefCV(gaussian_blur=0.5, gaussian_noise=0.2, jpeg_compression=0.3).to_tensor()       # README.md:118-122
    assert c.dtype == torch.float32 and c.tolist() == pytest.approx([0.5, 0.2, 0.3])


def test_parameter_cache_follows_replaced_parameters():
    """The flat parameter list the engine polls is cached; parametrizations and direct assignment replace Parameter
    objects and must be noticed (identity check), `.to()` / `load_state_dict` keep them."""
    m = MewZoom(2, 16, 2, 2, control_features=3)
    p0 = m._flat_params()
    assert len(p0) == len(list(m.parameters())) and all(a is b for a, b in zip(p0, m.parameters()))
    assert m._flat_params() is not p0 and all(a is b for a, b in zip(m._flat_params(), p0))
    m.add_weight_norms()
    p1 = m._flat_params()
    assert len(p1) == len(list(m.parameters())) > len(p0)
    m.remove_parameterizations()
    assert len(m._flat_params()) == len(p0)
    m.head.conv.weight = torch.nn.Parameter(torch.zeros_like(m.head.conv.weight))
    assert any(p is m.head.conv.weight for p in m._flat_params())
    assert MewZoom(2, 16, 2, 2, operand_dtype="auto").operand_dtype == "auto"
    with pytest.raises(AssertionError):
        MewZoom(2, 16, 2, 2, operand_dtype="float64")


def test_build_is_idempotent_under_the_lock():
    from ultrazoom_b200 import build as b

    assert b.build_locked() == b.LIB and os.path.exists(b.LIB)


def test_bench_arms_describe_one_workload():
    """VERDICT r1: the driver compares the `config` objects of `bench.py` and `bench.py --impl reference`; both come
    from one function, for every workload."""
    import argparse

    bench = _bench_module()
    args = argparse.Namespace(io="float32", residual_stream="auto", operands="float16", tune="")
    for w in bench.WORKLOADS:
        a, b = bench.config_of(w, 1, args), bench.config_of(w, 1, args)
        assert a == b and {"workload", "batch_per_gpu", "lr_h", "lr_w", "parallelism"} <= set(a)
    assert "halo-padded tile" in bench.config_of("cfg5", 8, args)["parallelism"]
    # --operands auto (the default of both arms): bf16 for the 20-layer 2X model -- the type BASELINE configs[1] names --
    # fp16 for the deeper models, where bf16 misses BASELINE's 2e-2 (tests/test_gpu_fullsize.py)
    auto = argparse.Namespace(io="float32", residual_stream="auto", operands="auto", tune="")
    assert bench.config_of("cfg2", 1, auto)["mma_operands"] == "bfloat16"
    assert all(bench.config_of(w, 1, auto)["mma_operands"] == "float16" for w in ("cfg3", "cfg4a", "cfg4b", "cfg5"))
    assert bench.config_of("cfg2", 1, auto, "float16")["mma_operands"] == "float16"


def test_current_library_is_found_without_writing(monkeypatch):
    """bench.py may run from a read-only tree: a current library is returned without a lock file or a directory."""
    import builtins

    from ultrazoom_b200 import build as b

    b.build_locked()
    real_open = builtins.open

    def read_only_open(path, mode="r", *a, **kw):
        if set(mode) & set("wax+"):
            raise PermissionError(f"read-only tree: {path}")
        return real_open(path, mode, *a, **kw)

    def no_makedirs(path, *a, **kw):
        raise PermissionError(f"read-only tree: {path}")

    monkeypatch.setattr(builtins, "open", read_only_open)
    monkeypatch.setattr(b.os, "makedirs", no_makedirs)
    assert b.build_locked() == b.LIB


def _bench_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs: a small output is written whole, a large one as a fixed sample with its flat indices; float32,
    within 64 MB, the same files for the same output."""
    import numpy as np

    bench = _bench_module()
    small = torch.rand(1, 3, 8, 10)
    bench.dump_output(str(tmp_path / "a"), "upscale", small)
    got = np.load(tmp_path / "a" / "upscale.npy")
    assert got.dtype == np.float32 and np.array_equal(got, small.numpy())
    assert not (tmp_path / "a" / "upscale_index.npy").exists()

    big = (torch.arange(2 * 3 * 1030 * 1024) % 251).to(torch.uint8).reshape(2, 3, 1030, 1024)
    for d in ("b", "c"):
        bench.dump_output(str(tmp_path / d), "upscale", big)
    vals, idx = np.load(tmp_path / "b" / "upscale.npy"), np.load(tmp_path / "b" / "upscale_index.npy")
    assert vals.dtype == np.float32 and idx.dtype == np.float64 and vals.shape == idx.shape == (bench.DUMP_MAX_ELEMENTS,)
    block = -(-big.numel() // bench.DUMP_MAX_ELEMENTS)                 # the sample spans the whole output
    assert np.all(np.diff(idx) > 0) and 0 <= idx[0] < block and big.numel() - block <= idx[-1] < big.numel()
    assert np.array_equal(vals, big.reshape(-1)[torch.from_numpy(idx).long()].float().numpy())
    assert sum(os.path.getsize(p) for p in (tmp_path / "b").iterdir()) <= 64 << 20
    for name in ("upscale.npy", "upscale_index.npy"):
        assert (tmp_path / "b" / name).read_bytes() == (tmp_path / "c" / name).read_bytes()
