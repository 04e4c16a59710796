"""apply_umap on one GPU: per-stage device times of scl_op_umap at N x r = 777 x 10 (the z785 golden's pca_n1),
68 000 x 7 and 500 000 x 10, one JSON line per shape.  kNN rate = N^2 d FMAs per second against the FP32 FMA issue
rate measured in the same run (scripts/fma_rate.cu: eight independent fmaf chains per thread), host comparison = sklearn brute-force
NearestNeighbors on the same input (host CPU).  UMAP.jl: not measured (no Julia here).

    python scripts/umap_bench.py [--out profiles/r3_umap_bench.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def measured_fma_rate():
    """FP32 FMA/s of the card, measured now by scripts/fma_rate.cu (built into a temporary directory)."""
    import tempfile
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "fma_rate")
        subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-O3", "-gencode", "arch=compute_100a,code=sm_100a",
                               os.path.join(ROOT, "scripts", "fma_rate.cu"), "-o", exe])
        return float(subprocess.check_output([exe]).decode().strip())


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": pl, "max_sm_clock": clk}
    except Exception as e:   # noqa: BLE001
        return {"gpu": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="777x10,68000x7,500000x10")
    a = ap.parse_args()
    from sclens_b200 import Handle
    info_card = card()
    peak = measured_fma_rate()
    lines = []
    with Handle() as h:
        for spec in a.sizes.split(","):
            N, d = map(int, spec.split("x"))
            if N == 777:
                z = np.load(os.path.join(ROOT, "tests", "golden", "z785_oracle.npz"))
                s = z["sig_id"]
                X = (z["signal_evec"][:, s] * np.sqrt(z["signal_ev"][s])[None, :]).astype(np.float32)
            else:
                rng = np.random.default_rng(N)
                C = rng.normal(0, 0.05, (20, d))
                X = (C[rng.integers(0, 20, N)] + rng.normal(0, 0.01, (N, d))).astype(np.float32)
            h.umap(X, 15, 2, n_epochs=10)                          # warm-up (module load, pools)
            t0 = time.perf_counter()
            P, info = h.umap(X, 15, 2)
            wall = time.perf_counter() - t0
            tk = info.t_knn_ms / 1e3
            rec = {"shape": f"{N}x{d}", "N": N, "d": d, "k": 15, "nc": 2, "n_epochs": 300, "metric": "cosine",
                   "apply_umap_s_host_wall": wall, "t_knn_ms": info.t_knn_ms, "t_graph_ms": info.t_graph_ms,
                   "t_init_ms": info.t_init_ms, "t_layout_ms": info.t_layout_ms,
                   "layout_ms_per_epoch": info.t_layout_ms / 300, "graph_nnz": info.graph_nnz,
                   "spectral_iters": info.spectral_iters, "init_fallback": info.init_fallback,
                   "knn_fma_per_s": float(N) * N * d / tk, "fp32_fma_per_s_measured": peak,
                   "knn_share_of_measured_fma_rate": (float(N) * N * d / tk) / peak if peak else None, **info_card}
            if N <= 68000:
                from sklearn.neighbors import NearestNeighbors
                Xn = X / np.maximum(np.linalg.norm(X, axis=1, keepdims=True), 1e-30)
                t0 = time.perf_counter()
                NearestNeighbors(n_neighbors=16, algorithm="brute", metric="cosine").fit(Xn).kneighbors(Xn)
                rec["host_cpu_sklearn_brute_knn_s"] = time.perf_counter() - t0
            else:
                rec["host_cpu_sklearn_brute_knn_s"] = "not measured (N too large for the host run)"
            rec["umap_jl_s"] = "not measured"
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
