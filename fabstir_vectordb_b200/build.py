"""In-tree build of libfvdb_b200.so (hand-written sm_100a CUDA; nvcc cross-compiles without a GPU).

    python -m fabstir_vectordb_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "libfvdb_b200.so")
STAMP = os.path.join(HERE, ".libfvdb_b200.stamp")

SOURCES = ["engine.cu", "exact_scan.cu", "layout.cu", "kmeans.cu", "tc_scan.cu", "synth.cu", "chunk_codec.cu"]
HEADERS = ["common.cuh", "kernels.cuh", "tc_scan.cuh", "tc_ptx.cuh", "tc_scan_wide.cuh"]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-fvisibility=hidden",
    "-ccbin", "/usr/bin/g++",
    "--fmad=true",  # fast kernels use FMA freely; reference-order arithmetic uses __f*_rn intrinsics
]


def _digest() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(fh.read())
    for f in ("fvdb.h", "fvdb_synth.h", "fvdb_chunk.h"):
        with open(os.path.join(ROOT, "include", f), "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    dig = _digest()
    if not force and os.path.exists(SO) and os.path.exists(STAMP):
        with open(STAMP) as fh:
            if fh.read().strip() == dig:
                return SO
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(out.decode(errors="replace"))
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"nvcc failed on {src}\n")
    if failed:
        raise RuntimeError("libfvdb_b200 build failed")
    link = [NVCC, "-shared", "-o", SO, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
            "-ccbin", "/usr/bin/g++", "-cudart", "static"]
    subprocess.check_call(link)
    with open(STAMP, "w") as fh:
        fh.write(dig)
    return SO


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(path)
