"""Build libsclens_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsclens_b200.so")
SOURCES = ["sparse.cu", "normalize.cu", "gemm_umma.cu", "eigen.cu", "tridiag.cu", "sytrd.cu", "sy2sb.cu", "sb2st.cu", "backtrans.cu", "refine.cu", "subspace.cu", "pipeline.cu", "denoise.cu", "preprocess.cu", "umap.cu", "leiden.cu", "capi.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-diag-suppress", "177"]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(HERE, "..", "include", "sclens_b200.h"))
    objdir = os.path.join(CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    jobs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            jobs.append([NVCC, *FLAGS, "-c", s, "-o", o])

    def run(cmd):
        if verbose:
            print(" ".join(cmd), flush=True)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        return r

    with ThreadPoolExecutor(max_workers=min(8, max(1, len(jobs)))) as ex:
        list(ex.map(run, jobs))
    objs = [os.path.join(objdir, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        run([NVCC, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
             "-lcusolver", "-ldl", "-Xlinker", "-rpath,/usr/local/cuda/lib64"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
