"""Builds libb200llama.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with
the repo snapshot to the GPU box)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libb200llama.so")
SOURCES = ["plan.cu"]


def _deps():
    d = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    d.append(os.path.join(HERE, "..", "include", "b200llama.h"))
    return d


NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # Java never contracts a*b+c; the kernels reproduce the CPU path's float order exactly.
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread", "-shared", "-Xptxas", "-v",
]


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in _deps()) or os.path.getmtime(__file__) > t


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, *NVCC_FLAGS, "-o", LIB, *[os.path.join(CSRC, s) for s in SOURCES], "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building libb200llama.so")
    with open(os.path.join(CSRC, "ptxas.log"), "w") as f:
        f.write(r.stderr)
    return LIB


TOK_LIB = os.path.join(CSRC, "libb200tok.so")
TOK_SRC = os.path.join(CSRC, "tokenizer.cpp")


def build_tokenizer(force: bool = False) -> str:
    """libb200tok.so: the native BPE tokenizer (CPU only, plain g++)."""
    hdr = os.path.join(HERE, "..", "include", "b200tok.h")
    if not force and os.path.exists(TOK_LIB) and os.path.getmtime(TOK_LIB) >= max(os.path.getmtime(TOK_SRC), os.path.getmtime(hdr)):
        return TOK_LIB
    cxx = os.environ.get("CXX", "g++")
    r = subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-o", TOK_LIB, TOK_SRC], capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building libb200tok.so")
    return TOK_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_tokenizer(force="--force" in sys.argv))
