"""Build librpsf_b200.so in-tree with nvcc for sm_100a (no torch involved).

    python -m regularizepsf_b200.csrc.build [--force]

One translation unit per patch size (rpsf_inst.cu, -DRPSF_P=...) compiled in parallel, plus the
C-ABI layer; linked with the static CUDA runtime so the library has no dependency beyond the
driver.  The .so lands in regularizepsf_b200/ (git-ignored, but it travels with gpurun).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
OBJ = os.path.join(HERE, "_build")
LIB = os.path.join(PKG, "librpsf_b200.so")
SIZES = (16, 32, 64, 128, 256, 512)
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-std=c++17", "-O3", "-lineinfo", "-Xcompiler", "-fPIC"] + ARCH
HEADERS = ["rpsf_fft.cuh", "rpsf_bands.cuh", "rpsf_kernels.cuh", "rpsf_saturation.cuh", "rpsf_stream.cuh", "rpsf_builder.cuh", "rpsf_adjoint.cuh", "rpsf_kgrad.cuh", "rpsf_construct_grad.cuh", "rpsf_ops.h", os.path.join("..", "..", "include", "rpsf_b200.h")]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found; the CUDA extension cannot be built")
    return exe


def _stale(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd: list[str]) -> None:
    proc = subprocess.run(cmd, cwd=HERE, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("command failed: " + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)


def build(force: bool = False, verbose: bool = False) -> str:
    """Build the library."""
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    deps = [os.path.join(HERE, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    objs = []
    for p in SIZES:
        obj = os.path.join(OBJ, f"inst_p{p}.o")
        objs.append(obj)
        if force or _stale(obj, deps + [os.path.join(HERE, "rpsf_inst.cu")]):
            jobs.append([nvcc, *COMMON, f"-DRPSF_P={p}", "-c", "rpsf_inst.cu", "-o", obj])
    api = os.path.join(OBJ, "api.o")
    objs.append(api)
    if force or _stale(api, deps + [os.path.join(HERE, "rpsf_api.cu")]):
        jobs.append([nvcc, *COMMON, "-c", "rpsf_api.cu", "-o", api])
    if verbose:
        for j in jobs:
            print(" ".join(j))
    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4) or 1) as pool:
        list(pool.map(_run, jobs))
    if jobs or force or not os.path.exists(LIB):
        _run([nvcc, "-shared", *ARCH, "-cudart", "static", "-o", LIB, *objs])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
