"""Builds gretel_b200/libhanselx.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
SOURCES = ["api.cu", "ingest.cu", "ingest_umma.cu", "ingest_long.cu", "ingest_lumma.cu", "recover.cu", "wire.cu", "probe.cu", "coverage.cu", "support.cu", "score.cu", "bootstrap.cu", "bampack.cpp"]
LIB_PATH = os.path.join(_HERE, "libhanselx.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",                 # fp64 recovery arithmetic must round like the CPU oracle
    # no -march for the host compiler: the x86-64 baseline has no FMA, so host fp64 (the EM of hx_em_abundance) is not
    # contracted and rounds like the Python oracle
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    # sources only: build_lib writes csrc/ptxas.log after the library, which must not make it stale
    deps = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))
            if f.endswith((".cu", ".cuh", ".cpp", ".h"))]
    deps.append(os.path.join(_ROOT, "include", "hanselx.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build_lib(force=False, verbose=False):
    if not force and not needs_build():
        return LIB_PATH
    extra = os.environ.get("HX_NVCC_DEFS", "").split()
    cmd = [nvcc_path()] + NVCC_FLAGS + extra + ["-I", os.path.join(_ROOT, "include"), "-I", os.path.join(_HERE, "csrc"),
                                       "-o", LIB_PATH] + [os.path.join(_HERE, "csrc", s) for s in SOURCES] + ["-lz"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libhanselx.so")
    with open(os.path.join(_HERE, "csrc", "ptxas.log"), "w") as fh:
        fh.write(res.stderr)
    return LIB_PATH


if __name__ == "__main__":
    build_lib(force=True, verbose=True)
