"""Build recipe for the in-tree CUDA library (sm_100a only).

``python -m damvsnet_b200.build`` (or ``__graft_entry__.build()``) compiles
``csrc/*.cu`` with nvcc into ``damvsnet_b200/_C/libdamvs_b200.so``.  nvcc
cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box
with the working-tree snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB = os.path.join(OUT_DIR, "libdamvs_b200.so")
STAMP = os.path.join(OUT_DIR, "build.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest() -> str:
    h = hashlib.sha256()
    files = sources() + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))
    files.append(os.path.join(HERE, "..", "include", "damvs.h"))
    for f in files:
        h.update(f.encode())
        h.update(open(f, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OUT_DIR, exist_ok=True)
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig:
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    log = []
    procs = []
    for src in sources():
        obj = os.path.join(OUT_DIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {os.path.basename(src)}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    link = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    with open(os.path.join(OUT_DIR, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    with open(STAMP, "w") as f:
        f.write(dig)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
