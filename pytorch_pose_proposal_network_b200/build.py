"""Compile libppn_decode.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m pytorch_pose_proposal_network_b200.build [--force]

The .so lands next to this file so that it travels with the source tree; there is no JIT
cache and no CPU fallback — if the library is missing, loading the package's ops raises.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB_PATH = os.path.join(PKG_DIR, "libppn_decode.so")
SOURCES = ["ppn_kernels.cu", "ppn_encode.cu", "ppn_head.cu", "ppn_loss.cu", "ppn_eval.cu", "ppn_proposals.cu", "ppn_augment.cu", "ppn_flip.cu", "ppn_capi.cu"]
HEADERS = [os.path.join(CSRC, "ppn_device.cuh"), os.path.join(CSRC, "ppn_kernels.h"),
           os.path.join(INCLUDE, "ppn_decode.h"), os.path.join(INCLUDE, "ppn_decode_bench.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",                  # numpy never fuses a*b+c; neither may we
    "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libppn_decode.so cannot be built")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > built for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    cmd = [nvcc_path(), *NVCC_FLAGS, "-I", INCLUDE, "-I", CSRC,
           *[os.path.join(CSRC, s) for s in SOURCES], "-o", LIB_PATH, "-lcudart"]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    log = os.path.join(PKG_DIR, "csrc", "build.log")
    with open(log, "w") as f:
        f.write(" ".join(cmd) + "\n" + proc.stdout + proc.stderr)
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout + proc.stderr)
    if proc.returncode != 0:
        raise RuntimeError(f"nvcc failed (exit {proc.returncode}); see {log}")
    return LIB_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
