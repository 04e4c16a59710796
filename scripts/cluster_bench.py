"""Clustering on one GPU: per-stage device times of scl_op_leiden (one batch of the 16-resolution start grid) and of the
whole resolution search scl_op_cluster, on the fuzzy graph of the umap_bench.py inputs (68 000 x 7 and 500 000 x 10,
k = 15, cosine), one JSON line per shape.  Rates: copies x levels per second (sum over trials and iterations of the levels
run, over the Leiden time).  Host comparison: one networkx Louvain trial (resolution 1) at 68 000 on the host CPU.
The card's name and power limit are read in the same run.

    python scripts/cluster_bench.py [--out profiles/r4_cluster_bench.json] [--sizes 68000x7:50,500000x10:10]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from umap_bench import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="68000x7:50,500000x10:10", help="NxD:trials,...")
    ap.add_argument("--no-host", action="store_true")
    a = ap.parse_args()
    from oracle.leiden_ref import start_grid
    from sclens_b200 import Handle
    info_card = card()
    lines = []
    with Handle() as h:
        for spec in a.sizes.split(","):
            shape, T = spec.split(":")
            N, d = map(int, shape.split("x"))
            T = int(T)
            rng = np.random.default_rng(N)                   # the input of umap_bench.py
            C = rng.normal(0, 0.05, (20, d))
            X = (C[rng.integers(0, 20, N)] + rng.normal(0, 0.01, (N, d))).astype(np.float32)
            h.umap(X, 15, 2, n_epochs=0, init="random")
            g = h.umap_graph()
            grid = start_grid()
            h.leiden(None, grid[:2], 2)                          # warm-up (module load, pools)
            t0 = time.perf_counter()
            lab, ncl, mod, li = h.leiden(None, grid, T)
            t_batch = time.perf_counter() - t0
            t_leiden = li.t_move_ms + li.t_refine_ms + li.t_aggregate_ms + li.t_labels_ms
            t0 = time.perf_counter()
            found, (eg, em), ci = h.cluster(None, 2, 20, T)
            t_search = time.perf_counter() - t0
            rec = {"shape": f"{N}x{d}", "N": N, "d": d, "k": 15, "metric": "cosine", "graph_nnz": int(g.nnz),
                   "n_trials": T, "batch_resolutions": len(grid),
                   "batch_s_host_wall": t_batch, "batch_t_validate_ms": li.t_validate_ms, "batch_t_move_ms": li.t_move_ms,
                   "batch_t_refine_ms": li.t_refine_ms, "batch_t_aggregate_ms": li.t_aggregate_ms,
                   "batch_t_labels_ms": li.t_labels_ms, "batch_max_levels": li.max_levels,
                   "batch_max_iterations": li.max_iterations, "batch_capped_levels": li.capped_levels,
                   "batch_copy_levels": li.copy_levels,
                   "batch_copy_levels_per_s": li.copy_levels / (t_leiden / 1e3) if t_leiden > 0 else None,
                   "batch_cluster_counts_per_resolution": [int(np.median(r)) for r in ncl],
                   "search_s_host_wall": t_search, "search_rounds": ci.n_rounds, "search_evaluated": ci.n_evaluated,
                   "search_found": sorted(int(k) for k in found), "search_t_leiden_ms": ci.t_leiden_ms,
                   "search_t_ecs_ms": ci.t_ecs_ms, "search_t_total_ms": ci.t_total_ms,
                   "search_copy_levels": ci.copy_levels,
                   "ic": {int(k): float(v["ic"]) for k, v in found.items()}, **info_card}
            if N <= 68000 and not a.no_host:
                import networkx as nx
                G = nx.from_scipy_sparse_array(g.astype(np.float64))
                t0 = time.perf_counter()
                comms = nx.community.louvain_communities(G, weight="weight", resolution=1.0, seed=0)
                rec["host_cpu_networkx_louvain_one_trial_s"] = time.perf_counter() - t0
                rec["host_cpu_networkx_louvain_clusters"] = len(comms)
            else:
                rec["host_cpu_networkx_louvain_one_trial_s"] = "not measured"
            print(json.dumps(rec), flush=True)
            lines.append(rec)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
