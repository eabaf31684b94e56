"""Builds libsage_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_PKG, "csrc", "sage_b200.cu")
_DEPS = [os.path.join(_PKG, "csrc", f) for f in ("sage_b200.cu", "kernels.cuh", "device_common.cuh", "fdr.cuh")] + [
    os.path.join(os.path.dirname(_PKG), "include", "sage_b200.h")]
_OUT = os.path.join(_PKG, "lib", "libsage_b200.so")

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false", "-Xcompiler", "-fPIC", "-shared"]


def library_path() -> str:
    return os.environ.get("SAGE_B200_LIB") or _OUT   # SAGE_B200_LIB: load a specific build (A/B measurements)


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(os.path.dirname(_OUT), exist_ok=True)
    if not force and os.path.exists(_OUT) and all(os.path.getmtime(_OUT) >= os.path.getmtime(d) for d in _DEPS):
        return _OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", _OUT, _SRC]
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    subprocess.check_call(cmd, env=env)
    return _OUT


_SYNTH_SRC = os.path.join(_PKG, "csrc", "synth_expand.cpp")
_SYNTH_OUT = os.path.join(_PKG, "lib", "libsage_synth.so")


def synth_library_path() -> str:
    return _SYNTH_OUT


def build_synth_library(force: bool = False) -> str:
    """Host-only helper of synth.py (synthetic benchmark / test data; no CUDA, not on the search path)."""
    os.makedirs(os.path.dirname(_SYNTH_OUT), exist_ok=True)
    if not force and os.path.exists(_SYNTH_OUT) and os.path.getmtime(_SYNTH_OUT) >= os.path.getmtime(_SYNTH_SRC):
        return _SYNTH_OUT
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    subprocess.check_call(["/usr/bin/g++", "-O3", "-std=c++17", "-fopenmp", "-shared", "-fPIC", "-o", _SYNTH_OUT, _SYNTH_SRC], env=env)
    return _SYNTH_OUT


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
    print(build_synth_library(force=True))
