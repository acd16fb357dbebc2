"""Builds libentreepy_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

    python -m entreepy_b200.build            # build if sources are newer than the library
    python -m entreepy_b200.build --force

The library lands in entreepy_b200/lib/ so that it travels with the repo snapshot to the
GPU box (built artefacts are git-ignored, not gpurun-ignored).
"""
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIBDIR, "libentreepy_b200.so")
CLI = os.path.join(PKG, "bin", "entreepy")

SOURCES = ["et_host.cpp", "et_hist.cu", "et_pack.cu", "et_unpack.cu", "et_api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-Wall,-Wextra,-fvisibility=hidden",
    "-Xptxas", "-v",
]


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA kernels cannot be built (there is no CPU fallback)")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(os.path.dirname(CLI), exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh", ".inc"))]
    deps.append(os.path.join(PKG, "..", "include", "entreepy_b200.h"))
    if force or _stale(LIB, deps):
        cmd = [nvcc(), *NVCC_FLAGS, "-shared", "-o", LIB, *srcs]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed building libentreepy_b200.so")
        open(os.path.join(LIBDIR, "ptxas.log"), "w").write(res.stdout + res.stderr)
    cli_src = os.path.join(CSRC, "cli", "main.cpp")
    if os.path.exists(cli_src) and (force or _stale(CLI, [cli_src, LIB])):
        cmd = ["g++", "-O2", "-std=c++17", "-Wall", "-Wextra", "-o", CLI, cli_src,
               "-L" + LIBDIR, "-lentreepy_b200", "-Wl,-rpath,$ORIGIN/../lib"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("g++ failed building the entreepy CLI")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
