"""Builds libxvec_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python speaker-recognition-x-vectors_b200/build.py [--force] [--verbose]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libxvec_b200.so")
SOURCES = ["capi.cu", "tdnn_gemm.cu", "tdnn_stack.cu", "fc_small.cu", "pool.cu", "mfcc.cu"]
HEADERS = ["ptx.cuh", "gemm_tile.cuh", "xvec_internal.h", os.path.join("..", "..", "include", "xvec_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
              "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


DEBUG_LIB = os.path.join(HERE, "libxvec_b200_debug.so")


def needs_build(lib: str = LIB) -> bool:
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, debug: bool = False) -> str:
    """debug=True builds libxvec_b200_debug.so with -DXVEC_DEBUG (per-tile clock stamps and epilogue/mainloop skip switches
    for tools/trace_tiles.py etc.; select it with XVEC_LIB=...)."""
    if debug:
        if not force and not needs_build(DEBUG_LIB):
            return DEBUG_LIB
        return _build_to(DEBUG_LIB, list(NVCC_FLAGS) + ["-DXVEC_DEBUG"], verbose, "_dbg")
    if not force and not needs_build():
        return LIB
    return _build_to(LIB, list(NVCC_FLAGS), verbose, "")


def _build_to(lib: str, flags, verbose: bool, suffix: str) -> str:
    flags = flags + (["-Xptxas", "-v"] if verbose else [])
    objs = []
    for s in SOURCES:
        obj = os.path.join(CSRC, s.replace(".cu", suffix + ".o"))
        cmd = [_nvcc()] + flags + ["-c", os.path.join(CSRC, s), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
        if r.returncode:
            raise RuntimeError(f"nvcc failed on {s}")
        objs.append(obj)
    cmd = [_nvcc(), "-shared", "-o", lib] + objs + ["-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, debug="--debug" in sys.argv))
