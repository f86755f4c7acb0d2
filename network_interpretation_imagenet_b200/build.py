"""Builds libnib.so (the C-ABI CUDA library, include/nib.h) in-tree with nvcc for sm_100a.

The library is the product: there is no Python/CPU fallback, `network_interpretation_imagenet_b200._lib`
raises if it is missing.  nvcc cross-compiles without a GPU, so this runs in the CPU container too.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libnib.so")
BUILD_DIR = os.path.join(PKG_DIR, "build")
SOURCES = ["api.cu", "mask_synth.cu", "score.cu", "conv_simt.cu", "conv_x3.cu", "conv_tc.cu", "net.cu", "gp.cu", "segment.cu", "ski.cu", "ski_kron.cu", "comm.cu", "localize.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest() -> str:
    h = hashlib.sha256()
    for root in (CSRC, os.path.join(os.path.dirname(PKG_DIR), "include")):
        for name in sorted(os.listdir(root)):
            with open(os.path.join(root, name), "rb") as f:
                h.update(name.encode())
                h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a and link libnib.so. Returns the library path."""
    os.makedirs(BUILD_DIR, exist_ok=True)
    stamp = os.path.join(BUILD_DIR, "digest.txt")
    digest = _digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB_PATH
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(BUILD_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
