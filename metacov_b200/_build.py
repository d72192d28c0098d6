"""Build recipe of the native library (nvcc, sm_100a only, in-tree).

``python metacov_b200/_build.py`` produces ``metacov_b200/libmetacov_b200.so``
from ``metacov_b200/csrc`` (CUDA kernels + C-ABI + host BAM reader).  The
reference builds two Cython extensions against pysam's htslib instead
(reference setup.py:12-33); here there is one shared library with a plain C ABI
(include/metacov_b200.h) loaded through ctypes.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB = os.path.join(HERE, "libmetacov_b200.so")
BUILD_DIR = os.path.join(ROOT, "build")

CUDA_SOURCES = ["mcov_api.cu", "stats_sort.cu", "experimental.cu", "synth.cu", "bam_gpu.cu", "sam_gpu.cu", "basecount.cu", "alleles.cu", "compare.cu"]
CXX_SOURCES = ["bamio.cpp", "transport.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-I" + INCLUDE,
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the CUDA extension cannot be built")


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    deps += [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]
    deps.append(os.path.abspath(__file__))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile the library if it is missing or older than its sources."""
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    extra = os.environ.get("MCOV_NVCC_EXTRA", "").split()      # tuning hook, e.g. -DMCOV_TT_STAGES=4
    os.makedirs(BUILD_DIR, exist_ok=True)
    objs = []
    for src in CUDA_SOURCES + CXX_SOURCES:
        obj = os.path.join(BUILD_DIR, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)
        objs.append(obj)
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-lz", "-gencode", "arch=compute_100a,code=sm_100a"]
    if verbose:
        print(" ".join(cmd), file=sys.stderr)
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
