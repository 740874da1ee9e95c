"""Build librnamsm_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python rna-msm_b200/build.py [--force] [--verbose]

The shared object lands in ``rna-msm_b200/lib/`` (git-ignored, but shipped to the GPU box with
the repo snapshot).  One nvcc invocation per translation unit, run in parallel.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "librnamsm_b200.so")
SOURCES = ["api.cu", "elementwise.cu", "simt_f32.cu", "umma_gemm.cu", "col_attn_umma.cu", "col_attn_fa.cu", "col_attn_probs.cu", "row_attn_short.cu", "peer.cu", "contact.cu", "ingest.cu", "score.cu", "sample.cu", "jacobian.cu", "windows.cu", "coevolution.cu", "fold.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _deps():
    out = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    out.append(os.path.join(os.path.dirname(HERE), "include", "rnamsm_b200.h"))
    return out


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    objs = []
    for src, obj, r in results:
        if verbose or r.returncode != 0:
            sys.stderr.write(f"--- {src}\n{r.stdout}{r.stderr}\n")
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(obj)
    cmd = [NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    a = ap.parse_args()
    print(build(a.force, a.verbose))
