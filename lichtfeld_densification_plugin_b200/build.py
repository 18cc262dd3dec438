"""Build recipe for csrc/libldp_b200.so: plain nvcc, sm_100a only, in-tree output.

    python -m lichtfeld_densification_plugin_b200.build
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libldp_b200.so")
SOURCES = ["ldp_api.cu"]                      # unity build: includes ldp_sample.cu / ldp_geometry.cu
DEPS = ["ldp_api.cu", "ldp_sample.cu", "ldp_front.cu", "ldp_geometry.cu", "ldp_output.cu", "ldp_select.cu", "ldp_voxel.cu", "ldp_outlier.cu", "ldp_device.cuh", os.path.join("..", "..", "include", "ldp_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.isfile(nvcc):
        raise RuntimeError("nvcc not found")
    return nvcc


def is_stale() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    cmd = [find_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH] + SOURCES
    proc = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
