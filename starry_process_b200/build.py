"""Builds ``libspb200.so`` (hand-written sm_100a CUDA behind the C ABI of include/spb200.h) in-tree.

    python -m starry_process_b200.build [--force]

nvcc cross-compiles without a GPU.  The library is placed next to this file so that it travels
with a repository snapshot; it is git-ignored.
"""
import glob
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libspb200.so")
STAMP = os.path.join(HERE, ".libspb200.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
]
# kernels that must reproduce the reference's unfused multiply/add sequences bit-for-bit
NO_FMA = {"moments.cu", "wigner.cu"}


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _digest():
    h = hashlib.sha256()
    for f in _sources() + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + sorted(
            glob.glob(os.path.join(CSRC, "*.h"))) + [
            os.path.join(HERE, "..", "include", "spb200.h"), __file__]:
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "nvcc")
    dig = _digest()
    if (not force and os.path.exists(LIB) and os.path.exists(STAMP)
            and open(STAMP).read().strip() == dig):
        return LIB
    _compile(nvcc, LIB, os.path.join(HERE, "build"), verbose)
    with open(STAMP, "w") as fh:
        fh.write(dig)
    return LIB


def _compile(nvcc, LIB, objdir, verbose):
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in _sources():
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        flags = list(NVCC_FLAGS)
        if os.path.basename(src) in NO_FMA:
            flags += ["-fmad=false"]
        if verbose:
            flags += ["-Xptxas", "-v"]
        cmd = [nvcc] + flags + ["-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0 or verbose:
            sys.stderr.write(out.decode())
        if pr.returncode != 0:
            failed = True
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                "-cudart", "static"]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
