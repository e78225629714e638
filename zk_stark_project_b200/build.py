"""Builds libzkb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libzkb200.so")
SOURCES = ["zkb200.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-diag-suppress", "550"]


def needs_build():
    """True when the library is missing or older than a file it is compiled from: any file in csrc/, or the public header
    that csrc/host.hpp includes."""
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(CSRC, "..", "..", "include", "zkb200.h")]
    return any(os.path.getmtime(f) > t for f in files)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose=True))
