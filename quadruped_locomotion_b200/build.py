"""Build libqlb.so (the C-ABI library) in-tree with nvcc for sm_100a."""
from __future__ import annotations

import glob
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libqlb.so")
SOURCES = ["qlb_api.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "--fmad=true", "-ldl"]


def _stale(lib: str) -> bool:
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    # every kernel header is included by qlb_api.cu: any edit under csrc/ or include/ makes the library stale
    deps = glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")) + \
        glob.glob(os.path.join(ROOT, "include", "*.h")) + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, extra=(), out: str | None = None) -> str:
    """Compile libqlb.so.  extra: more nvcc flags (e.g. -DQLB_DBAS_MAX_ROUNDS=1 for a kernel variant); out: where the
    library goes (default: in the package, where capi loads it from)."""
    lib = LIB if out is None else os.path.abspath(out)
    if not force and not _stale(lib):
        return lib
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + list(extra) + ["-I" + os.path.join(ROOT, "include"), "-I" + CSRC, "-o", lib] + \
          [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return lib


DEMO = os.path.join(PKG, "host", "tick_demo")
QP_DEMO = os.path.join(PKG, "host", "qp_demo")


def build_host_demo(force: bool = False, verbose: bool = False, which: str = "tick_demo") -> str:
    """Compile a C++ adapter demo (host code only, links libqlb.so)."""
    exe = os.path.join(PKG, "host", which)
    src = exe + ".cpp"
    hdrs = [os.path.join(PKG, "host", h) for h in ("qlb_adapter.hpp", "qlb_qp_adapter.hpp", "qlb_batch_adapter.hpp")]
    build()
    if not force and os.path.exists(exe) and os.path.getmtime(exe) > max([os.path.getmtime(f) for f in [src, LIB] + hdrs]):
        return exe
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(PKG, "host"),
           "-o", exe, src, "-L" + PKG, "-lqlb", "-Wl,-rpath," + PKG, "-Wl,-rpath,/usr/local/cuda/lib64"]
    if which == "nccl_demo":   # the multi-GPU demo talks to the CUDA runtime and NCCL itself
        cmd += ["-I/usr/local/cuda/include", "-L/usr/local/cuda/lib64", "-lcudart", "-lnccl", "-pthread"]
    if which == "threads_demo":
        cmd += ["-I/usr/local/cuda/include", "-L/usr/local/cuda/lib64", "-lcudart", "-pthread"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return exe


if __name__ == "__main__":
    extra = ["-Xptxas", "-v"] if "-v" in sys.argv else []
    print(build(force=True, verbose=True, extra=extra))
    print(build_host_demo(force=True, verbose=True))
    print(build_host_demo(force=True, verbose=True, which="qp_demo"))
    print(build_host_demo(force=True, verbose=True, which="swing_demo"))
    for extra_demo in ("params_demo", "batch_demo", "nccl_demo", "threads_demo", "controller_demo"):
        print(build_host_demo(force=True, verbose=True, which=extra_demo))
