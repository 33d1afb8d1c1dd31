"""Build libtrb_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m torchregister_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.path.join(OUT_DIR, "libtrb_b200.so")
SOURCES = ["abi.cu", "affine.cu", "affine_tma.cu", "affine_persist.cu", "warp_tma.cu", "edge.cu", "flow.cu", "flow_direct.cu", "jacobian.cu", "transform.cu", "lncc.cu", "nmi.cu", "nmi_src.cu", "instnorm.cu", "thinconv.cu"]
# every header under csrc/ plus the public C header: editing any of them makes the library stale
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inc"))) + [os.path.join("..", "..", "include", "trb.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found; libtrb_b200.so must be prebuilt (python -m torchregister_b200.build)")


def is_stale() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.isfile(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    os.makedirs(OUT_DIR, exist_ok=True)
    env = dict(os.environ)
    # the image exports CC/CXX pointing at a gcc wrapper without OpenMP specs; nvcc only needs g++
    extra = ["-DTRB_TIMING"] if os.environ.get("TRB_TIMING") else []
    extra += ["-D" + d for d in os.environ.get("TRB_DEFINES", "").split() if d]
    cmd = [_nvcc()] + NVCC_FLAGS + extra + ["-ccbin", shutil.which("g++") or "g++", "-o", LIB_PATH] + \
          [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    log = res.stdout + res.stderr
    with open(os.path.join(OUT_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed (see %s)" % os.path.join(OUT_DIR, "build.log"))
    if verbose:
        print(log)
    return LIB_PATH


if __name__ == "__main__":
    p = build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(p)
