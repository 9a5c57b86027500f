"""In-tree build of libdeepbedmap_b200.so with nvcc for sm_100a (no torch extension machinery:
the library is a plain C-ABI shared object loaded through ctypes)."""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libdeepbedmap_b200.so")
TUNING_LIB = os.path.join(HERE, "libdeepbedmap_b200_tuning.so")
STAMP = os.path.join(HERE, "build", "stamp.txt")

SOURCES = ["ops.cu", "gemm_f32.cu", "gemm_bf16.cu", "umma_conv3x3.cu", "umma_trunk.cu", "umma_flat.cu", "umma_local.cu", "umma_deform.cu", "stem.cu", "deform_f32.cu", "train_ops.cu", "gen_api.cu", "disc_api.cu"]
TUNING_SOURCES = ["debug_bench.cu"]   # libdeepbedmap_b200_tuning.so: microbenchmarks, never loaded by the product
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    cand = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; cannot build libdeepbedmap_b200.so")
    return cand


def _digest() -> str:
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(INCLUDE, "deepbedmap_b200.h")]
    for f in files:
        with open(f, "rb") as fh:
            h.update(f.encode())
            h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into one shared library. Returns the library path."""
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == digest:
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-I", INCLUDE, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    subprocess.run(cmd, check=True)
    for src in TUNING_SOURCES:   # links against the product library for the shared helpers (set_error, check_launch)
        cmd = [nvcc, *NVCC_FLAGS, "-shared", "-I", INCLUDE, os.path.join(CSRC, src), "-o", TUNING_LIB, "-L", HERE,
               "-ldeepbedmap_b200", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"]
        subprocess.run(cmd, check=True)
    with open(STAMP, "w") as fh:
        fh.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
