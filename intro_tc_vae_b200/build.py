"""Build libtcelbo.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo snapshot).

    python -m intro_tc_vae_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
LIB_PATH = os.path.join(PKG_DIR, "libtcelbo.so")
SOURCES = ["tc_kernels.cu", "tc_bwd_ds.cu", "tc_colvar.cu", "tc_materialized.cu", "tc_rowops.cu", "tc_abi.cu"]
HEADERS = ["tc_common.cuh", "tc_kernels.h", "tc_layout.h", "tc_rowops.h", "tc_instr.h", "tc_materialized.h"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3",
    "-shared", "-cudart", "shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libtcelbo.so cannot be built (there is no CPU fallback)")


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(INCLUDE, "tcelbo.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA sources into intro_tc_vae_b200/libtcelbo.so; returns its path."""
    if not force and not _stale():
        return LIB_PATH
    extra = os.environ.get("TCELBO_NVCC_FLAGS", "").split()          # extra nvcc flags, e.g. -Xptxas -warn-spills
    cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-I", INCLUDE, "-I", CSRC]
    cmd += [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout + res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
