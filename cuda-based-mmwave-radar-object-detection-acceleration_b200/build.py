"""Builds libmmw_radar_b200.so (the CUDA kernels + the C ABI) in-tree with nvcc for sm_100a.

The library is plain CUDA runtime code (no torch, no cuFFT): nvcc cross-compiles it without a
GPU, and the built .so travels with the tree to the GPU box.
"""
from __future__ import annotations

import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libmmw_radar_b200.so")
SOURCES = ["mmw_api.cu", "mmw_pipeline.cu", "mmw_detect.cu", "mmw_legacy.cu", "mmw_cluster.cu"]
HEADERS = [
    os.path.join(CSRC, "fft_regs.cuh"),
    os.path.join(CSRC, "mmw_common.cuh"),
    os.path.join(ROOT, "include", "mmw_radar.h"),
    os.path.join(ROOT, "include", "mmw_legacy.h"),
]
# the reference caller compiled UNMODIFIED from /root/reference by oracle/Makefile; linked here against
# our library to prove the drop-in (oracle/_ref is git-ignored and only exists where it was built)
REF_CALLER_OBJ = os.path.join(ROOT, "oracle", "_ref", "cudaBenchMarking.o")
DROPIN_BIN = os.path.join(ROOT, "oracle", "_ref", "dropin_acceleration")


def _nvcc() -> str:
    for cand in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc"), shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _host_cxx() -> str:
    # the image exports CXX=/opt/gcc/bin/g++ (a wrapper); the distro compiler is the safe host compiler for nvcc
    return "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else (shutil.which("g++") or "g++")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    cmd = [
        _nvcc(), "-ccbin", _host_cxx(),
        "-gencode", "arch=compute_100a,code=sm_100a",
        "-lineinfo", "-O3", "-std=c++17",
        "-Xptxas", "-v" if verbose else "-O3",
        "-shared", "-Xcompiler", "-fPIC",
        "-o", LIB,
    ] + [os.path.join(CSRC, s) for s in SOURCES] + ["-ldl"]      # dlopen of libnccl.so.2 (mmw_group_create); NCCL itself is not linked
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return LIB


def build_dropin() -> str | None:
    """Links the reference's unmodified cudaBenchMarking.o against our library (drop-in proof)."""
    if not os.path.exists(REF_CALLER_OBJ):
        return None
    build()
    if os.path.exists(DROPIN_BIN) and os.path.getmtime(DROPIN_BIN) > max(os.path.getmtime(LIB), os.path.getmtime(REF_CALLER_OBJ)):
        return DROPIN_BIN
    cmd = [_host_cxx(), "-m64", "-O3", "-o", DROPIN_BIN, REF_CALLER_OBJ, LIB, "-Wl,-rpath," + PKG]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("drop-in link failed:\n" + res.stdout + res.stderr)
    return DROPIN_BIN


if __name__ == "__main__":
    print(build(force=True, verbose=True))
    print(build_dropin())
