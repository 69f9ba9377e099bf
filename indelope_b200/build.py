"""Build the in-tree native libraries.

  libindelope_cuda.so  -- CUDA kernels + the C ABI of include/indelope_cuda.h   (nvcc, sm_100a only)
  libindelope_host.so  -- C++ host stand-in of include/indelope_host.h          (g++, zlib)
  indelope             -- the command line of the reference (src/indelope.nim:553-608) over the two libraries

Both are written next to this file so that they travel to the GPU box with the repo snapshot.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
INC = os.path.join(ROOT, "include")
CSRC = os.path.join(HERE, "csrc")
CUDA_LIB = os.path.join(HERE, "libindelope_cuda.so")
HOST_LIB = os.path.join(HERE, "libindelope_host.so")
CLI_BIN = os.path.join(HERE, "indelope")

CUDA_SRCS = ["pipeline.cu", "sweep.cu", "bamdev.cu", "fastadev.cu"]
HOST_SRCS = ["host/synth_sweep.cpp", "host/pack_vcf.cpp", "host/bamio.cpp"]
CLI_SRCS = ["host/indelope_main.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math",
              "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _deps(subdir_srcs):
    deps = [os.path.join(CSRC, s) for s in subdir_srcs]
    for d, _, fs in os.walk(CSRC):
        deps += [os.path.join(d, f) for f in fs if f.endswith((".cuh", ".h", ".hpp"))]
    deps += [os.path.join(INC, f) for f in os.listdir(INC)]
    return deps


def nvcc_path():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def build_host(force=False, verbose=False):
    if force or _newer(HOST_LIB, _deps(HOST_SRCS)):
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-I", INC] + [os.path.join(CSRC, s) for s in HOST_SRCS] + ["-o", HOST_LIB, "-lz", "-lpthread"]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return HOST_LIB


def build_cuda(force=False, verbose=False):
    if force or _newer(CUDA_LIB, _deps(CUDA_SRCS)):
        cmd = [nvcc_path()] + NVCC_FLAGS + os.environ.get("IDL_NVCC_EXTRA", "").split() + ["-I", INC, "-I", CSRC] + [os.path.join(CSRC, s) for s in CUDA_SRCS] + ["-o", CUDA_LIB]
        if verbose:
            print(" ".join(cmd))
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(HERE, "build_cuda.log")
        with open(log, "w") as f:
            f.write(r.stdout + r.stderr)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed")
    return CUDA_LIB


def build_cli(force=False, verbose=False):
    """the `indelope` binary; finds both libraries next to itself ($ORIGIN)"""
    if force or _newer(CLI_BIN, _deps(CLI_SRCS) + [HOST_LIB, CUDA_LIB]):
        cmd = ["g++", "-O2", "-std=c++17", "-Wall", "-I", INC] + [os.path.join(CSRC, s) for s in CLI_SRCS] + [
            "-o", CLI_BIN, "-L", HERE, "-lindelope_host", "-lindelope_cuda", "-lpthread", "-Wl,-rpath,$ORIGIN"]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return CLI_BIN


def build_all(force=False, verbose=False):
    build_host(force, verbose)
    build_cuda(force, verbose)
    build_cli(force, verbose)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose=True)
