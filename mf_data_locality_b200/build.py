"""In-tree build of the CUDA C-ABI library (libbp4.so) for sm_100a and of the C++ host
library mirroring the reference's operator/solver surface (libbp4_host.so)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIB = os.path.join(HERE, "libbp4.so")
HOSTLIB = os.path.join(HERE, "libbp4_host.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--threads", "0"]


def _nccl_dir():
    """site-packages/nvidia/nccl of the interpreter's environment (the NCCL torch loads)"""
    for p in sys.path:
        d = os.path.join(p, "nvidia", "nccl")
        if os.path.isdir(os.path.join(d, "lib")):
            return d
    return None


def _nccl_include():
    d = _nccl_dir()
    return ["-I", os.path.join(d, "include")] if d and os.path.exists(os.path.join(d, "include", "nccl.h")) else []


NCCL_INC = _nccl_include()


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _sources(d, exts):
    return [os.path.join(d, f) for f in sorted(os.listdir(d)) if f.endswith(exts)]


def build_cuda(force=False, verbose=False):
    srcs = _sources(CSRC, (".cu",))
    deps = _sources(CSRC, (".cu", ".cuh", ".h")) + [os.path.join(ROOT, "include", "bp4.h")]
    if not force and not _newer(LIB, deps):
        return LIB
    objs = []
    procs = []
    for s in srcs:
        o = os.path.join(CSRC, os.path.basename(s) + ".o")
        extra = os.environ.get("BP4_NVCC_EXTRA", "").split()
        cmd = ["nvcc"] + NVCC_FLAGS + NCCL_INC + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        procs.append((cmd, subprocess.Popen(cmd)))
        objs.append(o)
    for cmd, p in procs:
        if p.wait() != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    # link the NCCL that torch bundles (torch.distributed loads it too: one NCCL per process);
    # fall back to the system library
    nccl = []
    d = _nccl_dir()
    if d and os.path.exists(os.path.join(d, "lib", "libnccl.so.2")):
        nccl = ["-L", os.path.join(d, "lib"), "-l:libnccl.so.2", "-Xlinker", "-rpath", "-Xlinker",
                os.path.join(d, "lib")]
    cmd = ["nvcc", "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + \
          (nccl or ["-lnccl"]) + ["-lcudart"]
    subprocess.check_call(cmd)
    return LIB


def build_host(force=False):
    """the C++ host mirror: one shared library per run_cg_solver plugin + the four CLI executables"""
    inc = os.path.join(ROOT, "include")
    plugins = (("plain", [], "benchmark_precond"),
               ("merged", ["-DBP4_PLUGIN_MERGED"], "benchmark_precond_merged"),
               ("plain_device", ["-DBP4_PLUGIN_PLAIN_DEVICE"], "benchmark_precond_device"),
               ("merged_device", ["-DBP4_PLUGIN_MERGED_DEVICE"], "benchmark_precond_merged_device"))
    deps = _sources(HOST, (".cc", ".h")) + [os.path.join(inc, "bp4.h")] + \
        [os.path.join(HERE, plug, "bench.cc") for _, _, plug in plugins]
    common = ["/usr/bin/g++", "-O3", "-std=c++17", "-fPIC", "-pthread", "-Wall", "-I", inc]
    link = ["-L", HERE, "-lbp4", "-Wl,-rpath,$ORIGIN"]
    outs = []
    jobs = []
    for name, macro, plug in plugins:
        lib = os.path.join(HERE, f"libbp4_host_{name}.so")
        exe = os.path.join(HERE, plug, "bench")
        outs += [lib, exe]
        if force or _newer(lib, deps):
            jobs.append(common + macro + ["-shared", "-o", lib, os.path.join(HOST, "host_capi.cc")] + link)
        if force or _newer(exe, deps):
            jobs.append(common + ["-o", exe, os.path.join(HERE, plug, "bench.cc")] +
                        ["-L", HERE, "-lbp4", "-Wl,-rpath,$ORIGIN/.."])
    procs = [(j, subprocess.Popen(j)) for j in jobs]
    for j, p in procs:
        if p.wait() != 0:
            raise RuntimeError("host build failed: " + " ".join(j))
    return outs


def build_all(force=False, verbose=False):
    build_cuda(force, verbose)
    build_host(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
