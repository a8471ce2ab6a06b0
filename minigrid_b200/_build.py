"""Builds minigrid_b200/libminigrid_b200.so in-tree with nvcc for sm_100a (no torch headers: the library is
a plain C-ABI shared object, see include/minigrid_b200.h)."""
from __future__ import annotations

import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_PKG, "csrc")
LIB_PATH = os.path.join(_PKG, "libminigrid_b200.so")
SOURCES = ["mg_abi.cu", "mg_step.cu", "mg_step_window.cu", "mg_reset.cu", "mg_state.cu", "mg_wrappers.cu", "mg_host_expand.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--threads", "0"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: minigrid_b200 needs the CUDA toolkit to build its extension")


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)] + [os.path.join(os.path.dirname(_PKG), "include", "minigrid_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB_PATH
    cmd = [nvcc_path(), *NVCC_FLAGS, "-shared", "-o", LIB_PATH] + [os.path.join(_CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return LIB_PATH


if __name__ == "__main__":
    build(force=True, verbose=True)
