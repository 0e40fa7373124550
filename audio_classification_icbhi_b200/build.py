"""Builds liblogmel_b200.so in-tree with nvcc for sm_100a (no torch, no pybind: a plain C ABI).

    python -m audio_classification_icbhi_b200.build [--force]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "liblogmel_b200.so")
SOURCES = ["logmel_capi.cu"]
DEPS = ["logmel_capi.cu", "logmel_kernel.cuh", "logmel_aux.cuh", "resample.cuh", "lm_f2.cuh", "fft_gen.cuh", os.path.join("..", "..", "include", "logmel_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xptxas", "-v",
    "-shared", "-Xcompiler", "-fPIC",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")


def regenerate_fft() -> None:
    """fft_gen.cuh is generated text; regenerate it so the committed copy cannot drift."""
    out = subprocess.run([sys.executable, os.path.join(CSRC, "gen_fft.py")], check=True,
                         capture_output=True, text=True).stdout
    path = os.path.join(CSRC, "fft_gen.cuh")
    if not os.path.exists(path) or open(path).read() != out:
        with open(path, "w") as f:
            f.write(out)


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force: bool = False, verbose: bool = True) -> str:
    regenerate_fft()
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc(), *NVCC_FLAGS, "-o", LIB_PATH, *[os.path.join(CSRC, s) for s in SOURCES]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose:
        for line in (res.stdout + res.stderr).splitlines():
            if "registers" in line or "spill" in line or "error" in line or "warning" in line:
                print("[nvcc]", line.strip())
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
