"""Build libpypore_b200.so in-tree with nvcc for sm_100a (B200).

    python -m pypore_b200.build [--force] [--verbose]

The shared library is a plain C-ABI object (include/pypore_b200.h); it links
only against the CUDA runtime, not against torch.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpypore_b200.so")
SOURCES = ["api.cu"]
HEADERS = ["common.cuh", "threshold.cuh", "prefix.cuh", "split.cuh", "split_flow.cuh", "stats.cuh", "filter.cuh", "hmm.cuh",
           os.path.join("..", "..", "include", "pypore_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # no FMA contraction anywhere: the split decisions are compared bit-exactly
    # against the reference's separate fp64 multiply/add/divide (SURVEY App. D)
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "shared",
]


def nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def up_to_date():
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return all(os.path.getmtime(d) <= t for d in deps if os.path.exists(d))


def build(force=False, verbose=False, defines=(), out=None):
    """`defines` / `out` build an experimental variant next to the product library (development only;
    select it with PYPORE_B200_LIB)."""
    if out is None and not force and up_to_date():
        return LIB
    cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-D" + d for d in defines] + \
          [os.path.join(CSRC, f) for f in SOURCES] + ["-o", out or LIB]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[6:] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, defines=defs,
                out=outs[0] if outs else None))
