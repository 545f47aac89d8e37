"""Builds libnmch_b200.so (the C-ABI shared library) in-tree with nvcc for sm_100a.

The library is the product: there is no Python/CPU fallback.  `build()` is what
__graft_entry__.build() calls; it cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libnmch_b200.so")
LIB_CHECKED = os.path.join(PKG, "libnmch_b200_checked.so")     # -DNMCHB_CHECKS: device asserts + guard bands
BIN = os.path.join(ROOT, "bin")

NVCC = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]
CU_SOURCES = ["engine.cu", "fe_kernels.cu", "em_kernels.cu", "xorwow.cu", "group.cu", "qe_kernels.cu", "greeks_kernels.cu"]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _deps():
    out = [os.path.join(ROOT, "include", "nmch_b200.h")]
    for f in os.listdir(CSRC):
        if f.endswith((".cu", ".cuh", ".cpp", ".hpp", ".h")):
            out.append(os.path.join(CSRC, f))
    return out


def build(force: bool = False, verbose: bool = False, only_if_missing: bool = False) -> str:
    """Compile every CUDA source for sm_100a into nmch_b200/libnmch_b200.so.

    only_if_missing: never rebuild an existing library (what tests use: a snapshot copied to another machine may not
    preserve modification times, and rebuilding a library that the running process has loaded is unsafe)."""
    if only_if_missing and os.path.exists(LIB):
        return LIB
    if force or _newer(LIB, _deps()):
        objs = []
        os.makedirs(os.path.join(PKG, "build"), exist_ok=True)
        for src in CU_SOURCES:
            obj = os.path.join(PKG, "build", src.replace(".cu", ".o"))
            s = os.path.join(CSRC, src)
            if force or _newer(obj, _deps()):
                cmd = [NVCC, *ARCH, *COMMON, "-I", os.path.join(ROOT, "include"), "-c", s, "-o", obj]
                if verbose:
                    print(" ".join(cmd))
                subprocess.run(cmd, check=True)
            objs.append(obj)
        cmd = [NVCC, *ARCH, "-shared", "-o", LIB, *objs, "-ldl"]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return LIB


def build_checked(force: bool = False, verbose: bool = False, only_if_missing: bool = False) -> str:
    """The checked build of the same sources and ABI (nmch_b200/libnmch_b200_checked.so): -DNMCHB_CHECKS turns on the
    device-side asserts and puts guard bands around every device buffer (csrc/device_common.cuh, csrc/engine.cu).
    It stands in for compute-sanitizer, which is closed on the B200 pool; tests/test_gpu_checked_build.py loads it
    through NMCH_B200_LIB and runs the ragged / 64-bit-index / shard / multi-tile cases."""
    if only_if_missing and os.path.exists(LIB_CHECKED):
        return LIB_CHECKED
    if force or _newer(LIB_CHECKED, _deps()):
        out_dir = os.path.join(PKG, "build", "checked")
        os.makedirs(out_dir, exist_ok=True)
        objs = []
        for src in CU_SOURCES:
            obj = os.path.join(out_dir, src.replace(".cu", ".o"))
            if force or _newer(obj, _deps()):
                cmd = [NVCC, *ARCH, *COMMON, "-DNMCHB_CHECKS", "-I", os.path.join(ROOT, "include"), "-c",
                       os.path.join(CSRC, src), "-o", obj]
                if verbose:
                    print(" ".join(cmd))
                subprocess.run(cmd, check=True)
            objs.append(obj)
        cmd = [NVCC, *ARCH, "-shared", "-o", LIB_CHECKED, *objs, "-ldl"]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return LIB_CHECKED


def build_cli(force: bool = False, verbose: bool = False, only_if_missing: bool = False):
    """Compile the C++ method API + the NMCH / exploration CLIs (host C++ over the C ABI)."""
    build(force=force, verbose=verbose, only_if_missing=only_if_missing)
    src_dir = os.path.join(ROOT, "src")
    if not os.path.isdir(src_dir):
        return []
    os.makedirs(BIN, exist_ok=True)
    cxx = "/usr/bin/g++"
    outs = []
    api = [os.path.join(src_dir, "NMCH", "methods", f) for f in ("NMCH.cpp", "NMCH_FE.cpp", "NMCH_EM.cpp", "NMCH_QE.cpp")]
    api += [os.path.join(src_dir, "NMCH", "utils", "utils.cpp")]
    for name in ("nmch", "exploration"):
        main = os.path.join(src_dir, "NMCH", "test", f"{name}.cpp")
        exe = os.path.join(BIN, "NMCH" if name == "nmch" else "exploration")
        deps = api + [main, LIB]
        if not all(os.path.exists(d) for d in deps):
            continue
        if only_if_missing and os.path.exists(exe):
            outs.append(exe)
            continue
        if force or _newer(exe, deps):
            cmd = [cxx, "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), main, *api, "-o", exe,
                   "-L", PKG, "-lnmch_b200", "-pthread", f"-Wl,-rpath,{PKG}", "-Wl,-rpath,$ORIGIN/../nmch_b200"]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True)
        outs.append(exe)
    return outs


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_checked(force="--force" in sys.argv, verbose=True))
    print(build_cli(force="--force" in sys.argv, verbose=True))
