"""Build libpcgc_b200.so in-tree with nvcc for sm_100a (no JIT, no torch extension machinery).

``python -m pcgcv1_b200.build [--force] [--verbose]``.  nvcc cross-compiles without a GPU; the
resulting .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libpcgc_b200.so")
SOURCES = ["api.cu", "conv_ffma.cu", "umma_conv.cu", "umma_win.cu", "entropy.cu", "gpu_coder.cu", "train.cu", "topk.cu", "voxelize.cu", "metrics.cu", "meshsample.cu", "coder.cpp", "pointio.cpp", "meshio.cpp"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function,-ffp-contract=off", "--expt-relaxed-constexpr"]


def _deps_mtime() -> float:
    m = 0.0
    for root in (CSRC, os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(root):
            if f.endswith((".cu", ".cuh", ".h", ".cpp")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


# entropy.cu holds the device copy of the likelihood -> integer CDF path (det_math.h, cdf_norm.h) whose results must equal the host
# copy's bit for bit: no mul+add contraction there (the host objects are built with -ffp-contract=off).
# metrics.cu computes the per-point D1 / D2 values in NumPy's arithmetic (every multiply and add rounded on its own); so does
# meshsample.cu for the face weights, the sample points and their grid cells, which a NumPy restatement reproduces bit for bit.
PER_FILE = {"entropy.cu": ["-fmad=false"], "metrics.cu": ["-fmad=false"], "meshsample.cu": ["-fmad=false"]}


def _compile(src: str, verbose: bool) -> str:
    obj = os.path.join(OBJ, src + ".o")
    cmd = [NVCC] + FLAGS + PER_FILE.get(src, []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)      # a ptxas blow-up must not hang the build
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    if verbose:
        sys.stderr.write(r.stderr)
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _deps_mtime():
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-lcuda"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
