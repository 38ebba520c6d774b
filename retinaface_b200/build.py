"""In-tree build of librf_b200.so with nvcc for sm_100a (no JIT cache: the .so travels with the tree)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "librf_b200.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]
# (source, extra flags).  postproc.cu spells every rounding explicitly; -fmad=false is the belt to
# that pair of braces (bit-exact decode / IoU, see the header comment there).
SOURCES = [
    ("engine.cu", []),
    ("plan_fp.cu", []),
    ("plan_i8.cu", []),
    ("plan_tile.cu", []),
    ("comm.cu", []),
    ("jpeg.cu", []),
    ("postproc.cu", ["-fmad=false"]),
    ("preprocess.cu", ["-fmad=false"]),
    ("align.cu", ["-fmad=false"]),
    ("calibrate.cu", []),
    ("model.cpp", []),
    ("frontend.cpp", []),
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: librf_b200 cannot be built (there is no CPU fallback)")


def _deps_mtime() -> float:
    t = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(root):
            if f.endswith((".h", ".cuh")):
                t = max(t, os.path.getmtime(os.path.join(root, f)))
    return t


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = _deps_mtime()
    objs = []
    rebuilt = False
    cc = nvcc()
    for src, extra in SOURCES:
        sp = os.path.join(CSRC, src)
        op = os.path.join(OBJ, src.rsplit(".", 1)[0] + ".o")
        objs.append(op)
        if force or not os.path.exists(op) or os.path.getmtime(op) < max(os.path.getmtime(sp), hdr_t):
            cmd = [cc] + ARCH + COMMON + extra + ["-c", sp, "-o", op]
            if verbose:
                print(" ".join(cmd), file=sys.stderr)
            subprocess.check_call(cmd)
            rebuilt = True
    if rebuilt or not os.path.exists(LIB):
        cmd = [cc] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)
    return LIB


def build_host(force: bool = False) -> str:
    """C++ host side: the RetinaFace class shell + the main.cpp-style driver, linked against librf_b200.so."""
    host = os.path.join(HERE, "host")
    exe = os.path.join(HERE, "rf_main")
    srcs = [os.path.join(host, f) for f in ("RetinaFace.cpp", "main.cpp")]
    deps = srcs + [os.path.join(host, f) for f in ("RetinaFace.h", "cv_compat.hpp")] + [LIB]
    if force or not os.path.exists(exe) or os.path.getmtime(exe) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-std=c++14", "-O2", "-I", host, "-I", os.path.join(os.path.dirname(HERE), "include")] + srcs +
                              ["-o", exe, "-L", HERE, "-lrf_b200", "-Wl,-rpath,$ORIGIN"])
    return exe


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
