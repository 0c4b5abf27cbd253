"""Build ``csrc/libpnp_b200.so`` in-tree with nvcc for sm_100a (B200) only.

    python -m dt4image_restoration_b200.build [--force] [--verbose]

The library has no torch dependency (plain C-ABI, see ``include/pnp_b200.h``); nvcc cross-compiles it on
a machine without a GPU.  The ``.so`` is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libpnp_b200.so")
STAMP = os.path.join(CSRC, ".build_stamp")
SOURCES = ["api.cu", "psnr.cu", "ssim.cu", "fftprox.cu", "unet.cu", "policy.cu", "policy_observe.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "-Xptxas", "-v",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _digest() -> str:
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    names = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    names.append(os.path.join("..", "..", "include", "pnp_b200.h"))
    for n in names:
        with open(os.path.join(CSRC, n), "rb") as f:
            h.update(n.encode())
            h.update(f.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for s in _sources():
        o = os.path.join(CSRC, s.replace(".cu", ".o"))
        objs.append(o)
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {s} ====\n{out}")
        failed |= p.returncode != 0
    with open(os.path.join(CSRC, "build.log"), "w") as f:
        f.write("\n".join(log))
    if failed or verbose:
        sys.stderr.write("\n".join(log))
    if failed:
        raise RuntimeError("nvcc failed, see csrc/build.log")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB, *objs, "-lcudart"]
    subprocess.check_call(cmd)
    with open(STAMP, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
