"""Build the C-ABI CUDA library in-tree: slam_experiments_b200/libhm_matcher.so.

nvcc cross-compiles sm_100a without a GPU.  The built .so is git-ignored but
travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "libhm_matcher.so")
SOURCES = ["hm_api.cu", "hm_popc.cu", "hm_tc.cu", "hm_epilogue.cu", "hm_orb.cu", "hm_small.cu"]
HEADERS = ["hm_common.cuh", "hm_tcgen05.cuh", "hm_orb_pattern.inc"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(ROOT, "include", "hm_matcher.h")]
    return any(os.path.getmtime(d) > t for d in deps)


FAST_SRC = os.path.join(CSRC, "hmfast.c")
FAST_SO = os.path.join(HERE, "_hmfast.so")


def build_hmfast(force: bool = False) -> str:
    """Host-side helper (CPython C API, gcc): bulk cv2.DMatch construction.  Optional: the Python
    side falls back to calling the DMatch type when it is missing."""
    import sysconfig
    if not force and os.path.exists(FAST_SO) and os.path.getmtime(FAST_SO) >= os.path.getmtime(FAST_SRC):
        return FAST_SO
    inc = sysconfig.get_paths()["include"]
    subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-I", inc, "-o", FAST_SO, FAST_SRC])
    return FAST_SO


def build(force: bool = False, verbose: bool = False) -> str:
    try:
        build_hmfast(force)
    except Exception as e:  # pragma: no cover - optional accelerator
        print(f"warning: _hmfast not built ({e}); DMatch construction falls back to Python", file=sys.stderr)
    if not force and not is_stale():
        return SO
    cmd = [
        nvcc_path(), "-O3", "-std=c++17", "-lineinfo",
        "-gencode", "arch=compute_100a,code=sm_100a",
        "--cudart", "static", "-shared", "-Xcompiler", "-fPIC,-fvisibility=hidden",
        "-I", os.path.join(ROOT, "include"), "-I", CSRC,
        "-o", SO,
    ] + [os.path.join(CSRC, f) for f in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return SO


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(SO)
