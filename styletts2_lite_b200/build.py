"""Builds the C-ABI library in-tree with nvcc for sm_100a (no torch C++ ABI coupling).

    python -m styletts2_lite_b200.build [--force]

Output: styletts2_lite_b200/lib/libst2_b200.so (git-ignored, travels with gpurun snapshots).
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(HERE, "build")
LIB = os.path.join(LIBDIR, "libst2_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = ["decoder.cu", "predictor.cu", "api_units.cu", "kernels_norm.cu", "kernels_misc.cu", "kernels_source.cu",
           "length_regulator.cu", "vocos.cu", "conv_simt.cu", "conv_tc.cu", "conv_fused.cu", "conv_pipe.cu", "conv_row.cu", "kernels_lstm.cu", "postprocess.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr",
              "-I", INCLUDE]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _digest() -> str:
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(INCLUDE, "st2_b200.h"), __file__]
    for f in files:
        with open(f, "rb") as fh:
            h.update(f.encode())
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_current() -> bool:
    stamp = LIB + ".sha256"
    return os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and is_current():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src):
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(12, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static",
                                                  "-Xcompiler", "-fPIC"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(LIB + ".sha256", "w") as fh:
        fh.write(_digest())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
