"""Build recipe for the sm_100a shared library (and nothing else).

`python -m geometric_mapping_b200.build` compiles csrc/gm_capi.cu (which includes the kernel
headers) into csrc/libgm_b200.so with nvcc.  The library is built IN-TREE so that it travels to
the GPU box with the repo snapshot.  -fmad=false is part of the numerical contract: see
csrc/gm_stages.cuh.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libgm_b200.so")
SOURCES = ["gm_capi.cu"]
HEADERS = ["gm_device.cuh", "gm_sort.cuh", "gm_stages.cuh", "gm_ransac.cuh", "gm_polyline.cuh", "gm_compress.cuh", "gm_primitives.cuh", "gm_map.cuh", "gm_comm.cuh", "gm_register.cuh", "../../include/gm_capi.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",  # no implicit FMA contraction: integer decisions depend on unfused float math
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "-shared",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SOURCES
    env = dict(os.environ)
    # the image exports CXX=/opt/gcc/bin/g++; let nvcc use the distro host compiler
    env.pop("CXX", None)
    env.pop("CC", None)
    res = subprocess.run(cmd, cwd=CSRC, env=env, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


HOST_DIR = os.path.join(HERE, "host")
HOST_BIN = os.path.join(HOST_DIR, "geometric_mapping_node")
HOST_SOURCES = ["geometric_mapping_node.cpp", "tunnel_processing.cpp", "paramHandler.cpp"]


def build_host(force: bool = False) -> str:
    """C++ host shim + ROS-free node harness (mirrors the reference's node) linked against the library."""
    build()
    deps = [os.path.join(HOST_DIR, f) for f in HOST_SOURCES + ["tunnel_processing.hpp", "paramHandler.hpp", "gm_types.hpp"]]
    if not force and os.path.exists(HOST_BIN) and all(os.path.getmtime(d) <= os.path.getmtime(HOST_BIN) for d in deps + [LIB]):
        return HOST_BIN
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-O2", "-std=c++17", "-Wall", "-Wextra", "-o", HOST_BIN] + HOST_SOURCES + [
        "-L" + CSRC, "-lgm_b200", "-Wl,-rpath,$ORIGIN/../csrc"]
    res = subprocess.run(cmd, cwd=HOST_DIR, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return HOST_BIN


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_host(force="--force" in sys.argv))
