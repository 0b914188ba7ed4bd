"""Builds libimp_gpu.so in-tree with nvcc for sm_100a. Cross-compiles without a GPU."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libimp_gpu.so")
SOURCES = ["imp_kernels.cu", "imp_k_strip.cu", "imp_k_blur.cu", "imp_k_cubic.cu", "imp_k_gather.cu", "imp_gpu.cu", "imp_transfer.cpp", "imp_planner.cpp", "imp_ops.cpp"]
HEADERS = ["imp_plan.h", "imp_pixel.cuh", "imp_gather.cuh", "imp_internal.h", "imp_tiles.cuh", "imp_blur.cuh", "imp_cubic.cuh", "imp_gathertile.cuh",
           os.path.join("..", "..", "include", "imp_gpu.h"), os.path.join("..", "..", "include", "imp_ops.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",                      # every float op rounds once, like the reference's C (DESIGN.md §Exactness)
    "-Xcompiler", "-fPIC,-ffp-contract=off",
    "--shared", "-cudart", "static", "-diag-suppress", "128",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libimp_gpu.so cannot be built (there is no CPU fallback)")


OBJ = os.path.join(HERE, "build")
COMPILE_FLAGS = [f for f in NVCC_FLAGS if f != "--shared"]


def _deps(src: str):
    return [os.path.join(CSRC, src)] + [os.path.join(CSRC, h) for h in HEADERS]


def _obj(src: str) -> str:
    return os.path.join(OBJ, os.path.splitext(src)[0] + ".o")


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def stale() -> bool:
    return _newer(LIB, [d for s in SOURCES for d in _deps(s)])


LIB_DBG = os.path.join(HERE, "libimp_gpu_dbg.so")


def build(force: bool = False, verbose: bool = False, debug: bool = False) -> str:
    """One object per source (compiled in parallel, only when its source or a header changed), then one link.
    debug=True: the same sources with -DIMP_DEBUG_BOUNDS (imp_tiles.cuh) -> libimp_gpu_dbg.so, for the bounds-check test."""
    global OBJ
    if debug:
        return _build_debug(force)
    if not force and not stale():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    todo = [s for s in srcs if force or _newer(_obj(s), _deps(s))]
    procs = []
    for s in todo:
        cmd = [nvcc()] + COMPILE_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", _obj(s), os.path.join(CSRC, s)]
        procs.append((s, subprocess.Popen(cmd, cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    for s, pr in procs:
        out, err = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n" + out + err)
        if verbose:
            print(err)
    link = [nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-cudart", "static", "-o", LIB] + [_obj(s) for s in srcs]
    res = subprocess.run(link, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    return LIB


def _build_debug(force: bool) -> str:
    deps = [d for s in SOURCES for d in _deps(s)]
    if not force and not _newer(LIB_DBG, deps):
        return LIB_DBG
    obj = os.path.join(HERE, "build", "dbg")
    os.makedirs(obj, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    procs = []
    for s in srcs:
        o = os.path.join(obj, os.path.splitext(s)[0] + ".o")
        procs.append((s, o, subprocess.Popen([nvcc()] + COMPILE_FLAGS + ["-DIMP_DEBUG_BOUNDS", "-c", "-o", o, os.path.join(CSRC, s)],
                                             cwd=CSRC, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    for s, o, pr in procs:
        out, err = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc (debug) failed on {s}:\n" + out + err)
    link = [nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-cudart", "static", "-o", LIB_DBG] + [o for _, o, _ in procs]
    res = subprocess.run(link, cwd=CSRC, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link (debug) failed:\n" + res.stdout + res.stderr)
    return LIB_DBG


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug="--debug" in sys.argv))
