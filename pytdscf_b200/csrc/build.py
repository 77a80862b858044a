"""Build libtdvp_b200.so in-tree with nvcc for sm_100a (no GPU needed: nvcc cross-compiles).

    python pytdscf_b200/csrc/build.py [--force]

The shared library is placed next to the Python package (pytdscf_b200/libtdvp_b200.so); it is
git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
SOURCES = ["api.cu", "zgemm.cu", "zgemm_tma.cu", "contract.cu", "krylov.cu", "qr.cu", "svd.cu"]
HEADERS = ["common.cuh", "handle.cuh", "contract.cuh", "zgemm_plan.h", os.path.join("..", "..", "include", "tdvp_b200.h")]
OUT = os.path.join(PKG, "libtdvp_b200.so")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
]


def _digest() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        p = os.path.join(HERE, f)
        if os.path.exists(p):
            h.update(open(p, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = True) -> str:
    stamp = OUT + ".sha256"
    dig = _digest()
    if not force and os.path.exists(OUT) and os.path.exists(stamp) and open(stamp).read().strip() == dig:
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    objs = []
    os.makedirs(os.path.join(HERE, "_obj"), exist_ok=True)
    procs = []
    for src in SOURCES:
        sp = os.path.join(HERE, src)
        if not os.path.exists(sp):
            continue
        obj = os.path.join(HERE, "_obj", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", sp, "-o", obj]
        if verbose:
            print("[build]", " ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            print(f"[build] {src} FAILED:\n{out}", file=sys.stderr)
        elif out.strip() and verbose:
            print(out)
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT, *objs, "-lcudart"]
    if verbose:
        print("[build]", " ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    with open(stamp, "w") as f:
        f.write(dig)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
