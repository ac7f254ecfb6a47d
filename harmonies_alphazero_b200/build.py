"""Builds csrc/*.cu into harmonies_alphazero_b200/libharmonies_b200.so for sm_100a.

Plain nvcc, no torch linkage: the library is a C-ABI shared object (include/harmonies_b200.h)
that only needs the CUDA runtime (linked statically).  nvcc cross-compiles without a GPU.
"""

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libharmonies_b200.so")
SOURCES = ["hz_abi.cu", "hz_engine.cu", "hz_mcts.cu", "hz_evalcache.cu", "hz_symmetry.cu", "hz_heads.cu", "hz_tower.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--fmad=false",   # PUCT / Dirichlet arithmetic must round like the reference's numpy
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(os.path.dirname(HERE), "include", "harmonies_b200.h"),
        os.path.abspath(__file__),
    ]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile (if stale) and return the library path."""
    if not force and not needs_build():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    extra = os.environ.get("HZ_NVCC_EXTRA", "").split()      # experiments only (e.g. -DHZ_EXPAND_MIN_BLOCKS=5)
    cmd = [_nvcc()] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-shared", "-o", LIB] + srcs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed building libharmonies_b200.so")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
