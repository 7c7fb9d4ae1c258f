"""Builds libmbe.so in-tree with nvcc for sm_100a (the only target)."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libmbe.so")
SOURCES = ["mbe.cu"]


def deps():
    """Every file the library is compiled from: all .cu / .cuh here plus the public header."""
    files = glob.glob(os.path.join(HERE, "*.cu")) + glob.glob(os.path.join(HERE, "*.cuh"))
    return sorted(files) + [os.path.join(HERE, "..", "..", "include", "mbe.h")]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in deps())


def build(force: bool = False, verbose: bool = False, out: str = None) -> str:
    if out is None and not force and not is_stale():
        return LIB
    cmd = [
        nvcc_path(), "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC,-pthread",
        "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
        "--expt-relaxed-constexpr", "--extended-lambda",
        "-Xptxas", "-v" if verbose else "-O3",
        "-o", out or LIB,
    ] + [os.path.join(HERE, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return out or LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
