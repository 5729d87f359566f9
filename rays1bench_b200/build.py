"""Builds the sm_100a artefacts in-tree (they travel to the GPU box with the repo snapshot):

  rays1bench_b200/librays1_b200.so   C-ABI library: CUDA kernels + reference-shaped host layer (include/rays1_b200.h)
  rays1bench_b200/rays1_b200         drop-in executable (`[-w] [-n N]`, src/latest/rayweek1.cpp:930-988 of the reference)

nvcc cross-compiles without a GPU.  `python rays1bench_b200/build.py [--force] [-v]` (run by path: importing the package
needs the library this script builds) or `build()` from __graft_entry__, which always recompiles.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librays1_b200.so")
EXE = os.path.join(HERE, "rays1_b200")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC,-Wall,-Wno-unused-function"]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")
    return nvcc


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def sources():
    names = sorted(os.listdir(CSRC))
    return [os.path.join(CSRC, n) for n in names] + [os.path.join(os.path.dirname(HERE), "include", "rays1_b200.h")]


def build(force=False, verbose=False):
    nvcc = _nvcc()
    srcs = sources()
    extra = ["-Xptxas", "-v"] if verbose else []
    if force or _stale(LIB, srcs):
        cmd = [nvcc, *ARCH, *COMMON, *extra, "-shared", "-o", LIB, os.path.join(CSRC, "r1_core.cu"), os.path.join(CSRC, "r1_bvh_device.cu"),
               os.path.join(CSRC, "r1_move.cu"), os.path.join(CSRC, "rays1_host.cpp"),
               "-lcudart", "-ldl"]
        subprocess.run(cmd, check=True)
    if force or _stale(EXE, srcs + [LIB]):
        cmd = [nvcc, *ARCH, *COMMON, "-o", EXE, os.path.join(CSRC, "rays1_main.cpp"), "-L" + HERE, "-lrays1_b200",
               "-Xlinker", "-rpath,$ORIGIN"]
        subprocess.run(cmd, check=True)
    return LIB, EXE


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
    print(EXE)
