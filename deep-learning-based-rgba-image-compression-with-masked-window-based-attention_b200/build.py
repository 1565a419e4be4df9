"""In-tree nvcc build of libmwa_b200.so (sm_100a only).

    python -m <package>.build        or        __graft_entry__.build()

The shared library exports the C ABI declared in include/mwa_b200.h, links the CUDA runtime
statically and depends on nothing else (no torch types cross the boundary).  It is written next
to this file so that it travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libmwa_b200.so")
STAMP = os.path.join(PKG_DIR, "build", "stamp.txt")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]
# per-file extra flags: the rounding kernels must round like torch's separate fp32 ops (no FMA contraction)
EXTRA = {"round.cu": ["-fmad=false"], "alpha.cu": ["-fmad=false"], "rate.cu": ["-fmad=false"]}
SOURCES = ["abi.cu", "round.cu", "gdn.cu", "gdn_tc.cu", "mwa.cu", "mwa_sp.cu", "mwa_small.cu", "mwa_bwd.cu", "gate.cu", "alpha.cu", "conv_tc.cu", "msssim.cu", "rans.cu", "rans_dev.cu", "rate.cu"]


def _nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built")
    return exe


def _digest() -> str:
    h = hashlib.sha256()
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(CSRC, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    with open(os.path.join(PKG_DIR, "..", "include", "mwa_b200.h"), "rb") as f:
        h.update(f.read())
    h.update(repr((ARCH, COMMON, EXTRA, SOURCES)).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link libmwa_b200.so.  Returns the library path."""
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(STAMP):
        with open(STAMP) as f:
            if f.read().strip() == digest:
                return LIB_PATH
    nvcc = _nvcc()
    objdir = os.path.join(PKG_DIR, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *EXTRA.get(src, []), "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    for src, cmd, p in procs:
        out, _ = p.communicate()
        log.append(f"$ {' '.join(cmd)}\n{out}")
        if p.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError(f"nvcc failed on {src}")
    link = [nvcc, *ARCH, "-shared", "--cudart", "static", "-o", LIB_PATH, *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log.append(f"$ {' '.join(link)}\n{r.stdout}")
    if r.returncode != 0:
        sys.stderr.write(log[-1])
        raise RuntimeError("link failed")
    with open(os.path.join(objdir, "build.log"), "w") as f:
        f.write("\n".join(log))
    with open(STAMP, "w") as f:
        f.write(digest)
    if verbose:
        print("\n".join(log))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
