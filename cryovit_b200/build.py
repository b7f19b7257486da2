"""Build the sm_100a CUDA library in-tree (cryovit_b200/lib/libcryovit_b200.so).

nvcc cross-compiles without a GPU; the resulting .so is git-ignored but travels to the GPU box.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "csrc"
LIBDIR = ROOT / "lib"
LIB = LIBDIR / "libcryovit_b200.so"
SOURCES = ["host_common.cu", "gemm.cu", "vit_elementwise.cu", "attention.cu", "attention_tcgen05.cu", "head_elementwise.cu", "gn_fold.cu", "conv_halo.cu", "conv_wpackn.cu", "conv_wpack.cu", "conv_rows8.cu", "conv_rows.cu", "wgrad.cu", "wgrad_mn.cu", "wgrad_narrow.cu", "wgrad_tc.cu", "train_elementwise.cu", "det_reduce.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
] + os.environ.get("CVIT_NVCC_EXTRA", "").split()  # e.g. -DFA_POLY_EVERY=4 for A/B builds of one kernel


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (cand == "nvcc" or Path(cand).exists()):
            return cand
    raise RuntimeError("nvcc not found")


def _digest() -> str:
    h = hashlib.sha256()
    for f in sorted(CSRC.iterdir()):
        if f.suffix in (".cu", ".cuh", ".h"):
            h.update(f.name.encode())
            h.update(f.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> Path:
    LIBDIR.mkdir(exist_ok=True)
    stamp = LIBDIR / "build.sha256"
    digest = _digest()
    if not force and LIB.exists() and stamp.exists() and stamp.read_text().strip() == digest:
        return LIB
    nvcc = _nvcc()
    objdir = LIBDIR / "obj"
    objdir.mkdir(exist_ok=True)

    def compile_one(src: str) -> Path:
        obj = objdir / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
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
    cmd = [nvcc, "-shared", "-o", str(LIB), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp.write_text(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
