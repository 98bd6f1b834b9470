"""Build recipe of the native library: nvcc cross-compiles every kernel for sm_100a into one in-tree shared
object, poppy_b200/libpoppy_cuda.so (device kernels + the extern "C" layer of include/poppy_cuda.h + the C++
host stages behind include/poppy_host.h). No JIT, no torch extension: the .so travels with the tree."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(ROOT, "csrc")
LIB = os.path.join(ROOT, "libpoppy_cuda.so")

CUDA_SOURCES = [
    "poppy_cuda.cu",
    "device/kernels_geometry.cu",
    "device/kernels_warp.cu",
    "device/kernels_pyramid.cu",
    "device/kernels_unsharp.cu",
    "margin.cu",
    "denoise.cu",
]
HOST_SOURCES = [
    "host/delaunay.cpp",
    "host/morph_images.cpp",
    "host/host_abi.cpp",
    "host/writer.cpp",
]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-fmad=false",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
# host stages: no implicit FMA contraction (the Delaunay predicates mirror a non-FMA build of cv::Subdiv2D)
CXX_FLAGS = ["-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wall", "-pthread"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the morph renderer cannot be built without the CUDA toolkit")
    return exe


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _all_inputs():
    deps = [os.path.abspath(__file__)]
    for base, _, files in os.walk(CSRC):
        deps += [os.path.join(base, f) for f in files if f.endswith((".cu", ".cuh", ".cpp", ".hpp", ".h"))]
    inc = os.path.join(os.path.dirname(ROOT), "include")
    deps += [os.path.join(inc, f) for f in os.listdir(inc)]
    return deps


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libpoppy_cuda.so if any source is newer. Returns the library path."""
    if not force and not _newer(LIB, _all_inputs()):
        return LIB
    objdir = os.path.join(ROOT, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    objs = []
    for src in CUDA_SOURCES:
        obj = os.path.join(objdir, src.replace("/", "_") + ".o")
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src in HOST_SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(objdir, src.replace("/", "_") + ".o")
        objs.append(obj)
        cmd = ["g++", *CXX_FLAGS, "-I", os.path.join(os.path.dirname(ROOT), "include"), "-c", path, "-o", obj]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for cmd, p in procs:
        out, _ = p.communicate()
        log.append("$ " + " ".join(cmd) + "\n" + out)
        if p.returncode != 0:
            raise RuntimeError("build failed:\n" + log[-1])
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB, *objs, "-lcudart", "-lpthread"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log.append("$ " + " ".join(link) + "\n" + r.stdout)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + log[-1])
    with open(os.path.join(objdir, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
