"""Builds aeonflux_b200/csrc/libaeonflux_b200.so with nvcc for sm_100a (in-tree, so the .so travels to the GPU box)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(CSRC, "libaeonflux_b200.so")
SOURCES = ["afx_b200.cu", "api_impl.inc", "engine.cuh", "fe.cuh", "ge.cuh", "sc.cuh", "keccak.cuh", "sha512.cuh", "program.hpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared"]


def stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(os.path.dirname(HERE), "include", "aeonflux_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not stale():
        return SO
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO, os.path.join(CSRC, "afx_b200.cu")]
    subprocess.check_call(cmd, cwd=CSRC)
    return SO


def build_microbench():
    tools = os.path.join(os.path.dirname(HERE), "tools")
    out = os.path.join(tools, "microbench")
    src = os.path.join(tools, "microbench.cu")
    if not os.path.exists(out) or os.path.getmtime(src) > os.path.getmtime(out):
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-o", out, src])
    return out
