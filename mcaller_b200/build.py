"""Builds libmcaller_b200.so (hand-written sm_100a CUDA, C ABI in include/mcaller_b200.h) in-tree with nvcc."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmcaller_b200.so")
SOURCES = ["api.cu", "scan.cu", "records.cu", "windows.cu", "classify.cu", "synth.cu", "aggregate.cu", "fastq.cu", "format.cu", "train.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--use_fast_math=false",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-shared"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "mcaller_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, out=None):
    if out is None and not force and not needs_build():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"]
    extra = os.environ.get("MC_NVCC_EXTRA", "").split()          # e.g. "-DMC_SCAN_WARPS=10 -DMC_SCAN_MIN_CTAS=2" for tuning runs
    cmd = [_nvcc()] + flags + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out or LIB] + srcs
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode:
        sys.stderr.write(res.stdout)
    if res.returncode:
        raise RuntimeError("nvcc failed building libmcaller_b200.so")
    return out or LIB


if __name__ == "__main__":
    build(force=True, verbose="-v" in sys.argv)
    print(LIB)
