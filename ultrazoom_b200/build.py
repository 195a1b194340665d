"""Build the sm_100a shared library in-tree: ultrazoom_b200/lib/libmewzoom_b200.so.

    python -m ultrazoom_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the tree.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libmewzoom_b200.so")
STAMP = os.path.join(LIBDIR, "libmewzoom_b200.sha256")
# (source, extra defines, object name).  conv_tc.cu is compiled once per epilogue mode 0..2 (its template instantiations
# dominate the build time), once (part 4) for its host side, once per interleaved image layout of the head (parts
# 5..7), once per layout of the 16-bit image head (parts 8..11) and once per layout of the RGBA head (parts 12..19); see
# the MZ_TC_PART comment in the file.
SOURCES = [(f"{n}.cu", [], f"{n}.o") for n in ("host_util", "small_kernels", "yuv420", "api", "model", "probe", "block_fused", "unet_ops", "unet_tc")] + [
    ("conv_tc.cu", [f"-DMZ_TC_PART={part}"], f"conv_tc_p{part}.o") for part in (0, 1, 2, 4, *range(5, 20))
]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if os.path.exists(cand):
        return cand
    found = shutil.which("nvcc")
    if not found:
        raise RuntimeError("nvcc not found; the sm_100a library cannot be built")
    return found


def _digest() -> str:
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)) + ["../../include/mewzoom_b200.h"]:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(name.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current() -> bool:
    """The library exists and was built from the present sources and flags."""
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and is_current():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    digest = _digest()
    nvcc = _nvcc()

    def compile_one(unit) -> str:
        src, defines, objname = unit
        obj = os.path.join(OBJDIR, objname)
        cmd = [nvcc, *NVCC_FLAGS, *defines, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {unit[0]} {unit[1]}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with cf.ThreadPoolExecutor(max_workers=min(os.cpu_count() or 4, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    r = subprocess.run([nvcc, "-shared", "-o", LIB, *objs, "-cudart", "static"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(STAMP, "w") as f:
        f.write(digest)
    return LIB


def build_locked(force: bool = False, verbose: bool = False) -> str:
    """build() under an inter-process file lock (one process per GPU: every rank calls this at import).

    A current library is returned without taking the lock, so that a built tree is only read: it may be read-only."""
    import fcntl

    if not force and is_current():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    with open(os.path.join(LIBDIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return build(force=force, verbose=verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
