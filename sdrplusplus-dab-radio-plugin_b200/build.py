"""Build libdabgpu.so (CUDA, sm_100a only) in-tree with nvcc.  nvcc cross-compiles without a GPU."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libdabgpu.so")
SOURCES = ["dabgpu.cu"]
HEADERS = ["common.cuh", "tables.cuh", "viterbi.cuh", "viterbi_lanes.cuh", "viterbi_lane_core.h", "chan.cuh", "dabplus.cuh", "ofdm.cuh", "ofdm_demod.cuh", "ofdm_host.cuh", "wideband.cuh", os.path.join("..", "..", "include", "dabgpu.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17", "--shared",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for f in SOURCES + HEADERS:
        p = os.path.join(CSRC, f)
        if os.path.exists(p) and os.path.getmtime(p) > t:
            return True
    return False


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    res = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libdabgpu.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


ROOT = os.path.dirname(HERE)
ADAPTER_SRC = os.path.join(ROOT, "tests", "host", "adapter_check.cpp")
ADAPTER_BIN = os.path.join(ROOT, "tests", "host", "_bin", "adapter_check")


def build_adapter_check(force: bool = False) -> str:
    """g++ build of the C++ adapter test driver (host/dab_adapters.hpp over the C ABI), linked against libdabgpu.so."""
    deps = [ADAPTER_SRC, os.path.join(HERE, "host", "dab_adapters.hpp"), os.path.join(ROOT, "include", "dabgpu.h")]
    if not force and os.path.exists(ADAPTER_BIN) and all(os.path.getmtime(d) <= os.path.getmtime(ADAPTER_BIN) for d in deps):
        return ADAPTER_BIN
    os.makedirs(os.path.dirname(ADAPTER_BIN), exist_ok=True)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-Wall", "-Wextra", "-o", ADAPTER_BIN, ADAPTER_SRC,
           "-L" + CSRC, "-ldabgpu", "-Wl,-rpath," + CSRC, "-lpthread"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("g++ failed building tests/host/adapter_check")
    return ADAPTER_BIN


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
