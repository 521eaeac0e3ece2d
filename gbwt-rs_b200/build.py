"""Builds libgbwt_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python gbwt-rs_b200/build.py [--force]

nvcc cross-compiles without a GPU. The shared object is git-ignored but travels to the GPU box with the
repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libgbwt_b200.so")
SOURCES = [os.path.join(CSRC, f) for f in ("cabi.cu", "find_mixed.cu", "find_window.cu", "layout_builder.cpp", "sds_loader.cpp", "layout_writer.cpp", "locate.cu", "ranges.cu", "build.cu")]
HEADERS = [os.path.join(CSRC, f) for f in ("kernels.cuh", "find_lean.cuh", "find_mixed.h", "find_window.h", "record_scan.cuh", "layout.h", "layout_builder.h", "sds_loader.h", "layout_writer.h", "locate.h", "ranges.h", "build.h", "record_encode.h")] + \
          [os.path.join(os.path.dirname(HERE), "include", f) for f in ("gbwt_b200.h", "gbwt_b200_ranges.h", "gbwt_b200_build.h")]


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def command(out: str = OUT, extra=()):
    return [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
            "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fPIC,-fopenmp,-O3,-fvisibility=hidden,-Wall", "-Xptxas", "-v",
            "-shared", "-o", out, *extra, *SOURCES, "-lgomp", "-ldl"]


def is_stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(f) > t for f in SOURCES + HEADERS + [os.path.abspath(__file__)])


def build(force: bool = False, verbose: bool = False) -> str:
    if force or is_stale():
        proc = subprocess.run(command(), capture_output=True, text=True)
        if proc.returncode != 0:
            sys.stderr.write(proc.stdout + proc.stderr)
            raise RuntimeError("nvcc failed")
        log = os.path.join(HERE, "build_ptxas.log")
        with open(log, "w") as f:
            f.write(proc.stdout + proc.stderr)
        if verbose:
            sys.stderr.write(proc.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
