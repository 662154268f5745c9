"""In-tree build of libragmeup_b200.so (sm_100a only).

``python -m ragmeup_b200.build`` or ``__graft_entry__.build()``.  nvcc cross-compiles without a
GPU; the .so is written next to the sources so it travels with the tree (it is git-ignored).
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libragmeup_b200.so")
STAMP = os.path.join(CSRC, ".build_stamp")
SOURCES = ["rmu_common.cu", "rmu_index.cu", "rmu_gemm.cu", "rmu_encoder.cu", "rmu_bm25.cu", "rmu_bm25_host.cu"]
# every header under csrc/ takes part in the up-to-date check (a list kept by hand once missed rmu_attention.cuh / rmu_scan.cuh)
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))) + [os.path.join("..", "..", "include", "ragmeup_b200.h")]

# -compress-all: by default the fatbinary is compressed only past a size threshold, so which object files came out
# compressed depended on how many kernel instantiations they held
NVCC_FLAGS = [
    "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--diag-suppress", "550", "-Xfatbin", "-compress-all",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _digest() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        p = os.path.join(CSRC, f)
        if os.path.exists(p):
            with open(p, "rb") as fh:
                h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source into one shared library; returns its path."""
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP):
        with open(STAMP) as f:
            if f.read().strip() == dig:
                return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    objs = []
    procs = []
    for s in srcs:
        o = s[:-3] + ".o"
        objs.append(o)
        cmd = [_nvcc(), *NVCC_FLAGS, "-c", s, "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    with open(STAMP, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
