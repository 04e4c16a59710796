"""Stage-by-stage check of the two-stage eigensolver on the GPU (scl_debug_two_stage) against numpy Float64, then timings of
the full solve per stage: python scripts/two_stage_check.py [sizes...] [--time N]"""
import ctypes as C
import json
import sys
import time

import numpy as np

sys.path.insert(0, ".")
from sclens_b200 import Handle  # noqa: E402
from sclens_b200._lib import ptr  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
sizes = [int(a) for a in args] or [256, 520, 1000, 2052]
time_n = 0
for a in sys.argv[1:]:
    if a.startswith("--time="):
        time_n = int(a.split("=")[1])
B, LDAB = 64, 128


def band_to_dense(AB, n):
    M = np.zeros((n, n))
    for dgl in range(LDAB):
        v = AB[: n - dgl, dgl].astype(np.float64) if dgl < n else None
        if v is None or dgl >= n:
            break
        M[np.arange(dgl, n), np.arange(0, n - dgl)] = v
    M = M + np.tril(M, -1).T
    return M


report = {}
with Handle() as h:
    for n in sizes:
        rng = np.random.default_rng(n)
        X = rng.standard_normal((n, n + 300))
        X -= X.mean(axis=0)
        G = np.ascontiguousarray((X @ X.T / X.shape[1]).astype(np.float32))
        G64 = G.astype(np.float64)
        wref = np.linalg.eigvalsh(G64)
        AB = np.zeros((n, LDAB), np.float32)
        d, e = np.zeros(n, np.float32), np.zeros(n - 1, np.float32)
        small = n <= 2100
        Q2 = np.zeros((n, n), np.float32) if small else None
        Q = np.zeros((n, n), np.float32) if small else None
        flags = (C.c_int32 * 2)()
        t0 = time.time()
        h._ck(h.lib.scl_debug_two_stage(h.h, n, ptr(G, C.c_float), ptr(AB, C.c_float), ptr(d, C.c_float), ptr(e, C.c_float),
                                        ptr(Q2, C.c_float) if small else None, ptr(Q, C.c_float) if small else None, flags))
        r = {"fail_flag": int(flags[0]), "npanels": int(flags[1]), "wall_s": time.time() - t0}
        Bd = band_to_dense(AB, n)
        ii, jj = np.indices((n, n))
        r["band_nonfinite"] = int((~np.isfinite(AB)).sum())
        r["band_outside_halfwidth_max"] = float(np.abs(AB[:, B + 1:]).max())
        wb = np.linalg.eigvalsh(Bd)
        r["stage1_eig_err"] = float(np.abs(wb - wref).max() / wref[-1])
        T = np.diag(d.astype(np.float64)) + np.diag(e.astype(np.float64), 1) + np.diag(e.astype(np.float64), -1)
        wt = np.linalg.eigvalsh(T)
        r["stage2_eig_err_vs_band"] = float(np.abs(wt - wb).max() / wref[-1])
        r["total_eig_err"] = float(np.abs(wt - wref).max() / wref[-1])
        if small:
            Q2m = Q2.T.astype(np.float64)   # column v of the transformation = row v of the buffer
            Qm = Q.T.astype(np.float64)
            r["q2_orth"] = float(np.abs(Q2m.T @ Q2m - np.eye(n)).max())
            r["q2_similarity_err"] = float(np.abs(Q2m.T @ Bd @ Q2m - T).max() / wref[-1])
            r["q_orth"] = float(np.abs(Qm.T @ Qm - np.eye(n)).max())
            r["q_similarity_err"] = float(np.abs(Qm.T @ G64 @ Qm - T).max() / wref[-1])
            Q1m = Qm @ Q2m.T
            r["q1_similarity_err"] = float(np.abs(Q1m.T @ G64 @ Q1m - Bd).max() / wref[-1])
        report[str(n)] = r
        print(n, json.dumps(r), flush=True)

    if time_n:
        n = time_n
        out = {}

        def bench(mode, il=0, iu=0):
            ms = C.c_double()
            h._ck(h.lib.scl_bench_syevd(h.h, n, mode, il, iu, C.byref(ms)))
            st = np.zeros(8)
            h.lib.scl_debug_last_solve(h.h, ptr(st, C.c_double))
            return ms.value, [round(float(x), 2) for x in st]

        for name, one_stage, mode, il, iu in (("one_stage_values_only", 1, 8, 0, 0), ("two_stage_values_only", 0, 8, 0, 0),
                                              ("two_stage_values_only_2", 0, 8, 0, 0),
                                              ("two_stage_smallest_half", 0, 7, 1, n // 2 + 65), ("two_stage_all_vectors", 0, 6, 0, 0),
                                              ("one_stage_smallest_half", 1, 7, 1, n // 2 + 65)):
            h._ck(h.lib.scl_debug_force_one_stage(one_stage))
            try:
                out[name] = bench(mode, il, iu)
            except Exception as ex:  # noqa: BLE001
                out[name] = str(ex)
            print(name, out[name], flush=True)
        h.lib.scl_debug_force_one_stage(0)
        report["timing_%d" % n] = out
open("gpurun_out/r2_two_stage_check.json", "w").write(json.dumps(report, indent=1))
