"""Builds the native pieces in-tree with nvcc for sm_100a (no JIT cache, no fallback arch).

  lib/libgraphembed_b200.so   CUDA kernels + the C ABI of include/graph_embed_b200.h
  lib/ge_dropin_demo          C++ program using the header-only drop-in (host/include/embed.hpp)

`python graph-embed_b200/build.py [-v]` or `build_all()` from __graft_entry__.build().
"""
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIB = os.path.join(LIBDIR, "libgraphembed_b200.so")
SOURCES = ["ge_capi.cu", "ge_flat.cu", "ge_flat_sym.cu", "ge_onchip.cu", "ge_multilevel.cu", "ge_galerkin.cu", "ge_coarsen.cu", "ge_components.cu", "ge_edges.cu", "ge_radii.cu", "ge_multi.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-O2,-Wall,-Wno-unknown-pragmas", "--expt-relaxed-constexpr"]


def nvcc():
    path = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(path):
        raise RuntimeError("nvcc not found; the CUDA extension cannot be built")
    return path


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(verbose=False, force=False):
    os.makedirs(LIBDIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(ROOT, "include", "graph_embed_b200.h"))
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            jobs.append([nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o])
    if jobs:  # the translation units are independent: compile them side by side
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=len(jobs)) as pool:
            list(pool.map(subprocess.check_call, jobs))
    if force or _stale(LIB, objs):
        subprocess.check_call([nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB]
                              + objs + ["-cudart", "static", "-ldl"])
    return LIB


def build_dropin_demo():
    """Compiles a C++ caller against the header-only drop-in to prove the reference-facing API."""
    src = os.path.join(PKG, "host", "examples", "dropin_demo.cpp")
    if not os.path.exists(src):
        return None
    out = os.path.join(LIBDIR, "ge_dropin_demo")
    deps = [src, LIB] + [os.path.join(PKG, "host", "include", f)
                         for f in os.listdir(os.path.join(PKG, "host", "include"))]
    if _stale(out, deps):
        subprocess.check_call(["g++", "-std=c++14", "-O2", "-I", os.path.join(PKG, "host", "include"),
                               "-I", os.path.join(PKG, "host", "compat"),
                               "-I", os.path.join(ROOT, "include"), src, "-o", out,
                               "-L", LIBDIR, "-lgraphembed_b200", "-Wl,-rpath,$ORIGIN", "-ldl", "-lpthread"])
    return out


def build_all(verbose=False, force=False):
    lib = build_library(verbose=verbose, force=force)
    build_dropin_demo()
    return lib


if __name__ == "__main__":
    print(build_all(verbose="-v" in sys.argv, force="-f" in sys.argv))
