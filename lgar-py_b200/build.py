"""In-tree build of liblgar_b200.so with nvcc for sm_100a (no JIT cache: the .so travels with
the source tree to the GPU box)."""
from __future__ import annotations

import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB = os.path.join(_HERE, "liblgar_b200.so")
SOURCES = ["lgar_capi.cu", "lgar_backward_launch.cu"]
HEADERS = ["lgar_device.cuh", "lgar_forward.cuh", "lgar_backward.cuh", "lgar_pow.cuh", "lgar_pow_tables.h", "lgar_var.cuh", "lgar_rounded.cuh",
           "../../include/lgar_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--threads", "2",
    # no FMA contraction: every product and sum rounds separately, like the reference's torch ops
    "--fmad=false",
    "-Xcompiler", "-fPIC", "-shared",
]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    for f in SOURCES + HEADERS + ["../build.py"]:
        p = os.path.join(CSRC, f)
        if os.path.exists(p) and os.path.getmtime(p) > t:
            return True
    return False


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    flags = list(NVCC_FLAGS)
    if verbose:
        flags += ["-Xptxas", "-v"]
    flags += os.environ.get("LGAR_EXTRA_NVCC_FLAGS", "").split()  # developer A/B switches
    cmd = ["nvcc", *flags, "-o", os.environ.get("LGAR_BUILD_OUT", LIB), *[os.path.join(CSRC, s) for s in SOURCES]]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building liblgar_b200.so")
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
