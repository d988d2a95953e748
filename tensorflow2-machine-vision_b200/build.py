"""Builds libb200det.so in-tree with nvcc for sm_100a (no torch extension machinery: plain C ABI)."""
import glob
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libb200det.so")
STAMP = os.path.join(HERE, "csrc", ".build_stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",            # decision paths must never contract a*b+c (detmath.h also pins this per op)
    "-ftz=false", "-prec-div=true", "-prec-sqrt=true",
    "-Xcompiler", "-fPIC,-O2,-ffp-contract=off,-fno-fast-math",
    "--threads", "0",
]


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def _digest():
    h = hashlib.sha256()
    for p in _sources() + sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + sorted(glob.glob(os.path.join(CSRC, "*.h"))) + [
        os.path.join(HERE, "..", "include", "b200det.h"), __file__]:
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    return h.hexdigest()


def build(force=False, verbose=False):
    """Compile every CUDA source into one shared library.  Returns the library path."""
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig:
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in _sources():
        obj = os.path.join(HERE, "build", os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("== %s ==\n%s\n" % (os.path.basename(src), out))
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libb200det.so")
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link of libb200det.so failed")
    with open(STAMP, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
