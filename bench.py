#!/usr/bin/env python
"""bench.py - sclens() throughput on synthetic data of the BASELINE.json shapes.

    python bench.py --gpus N --steps K --warmup W [--workload C|B|small|D|E] [--impl reference] [--dump-outputs DIR]

Workloads: C = 68k cells x 20k genes (BASELINE.json configs[2], the shape the metric is quoted on; default),
B = 10k x 20k (configs[1]), small = 2k x 3k (smoke), D = 500k x 25k (configs[3]: signal stage only - cell-sharded
Gram + NCCL reduce of the packed triangle + the two eigensolves), E = C with 100 perturbation replicates (configs[4]).

Exactly --steps passes are timed.  Warm-up runs --warmup passes but stops after the third once two consecutive passes
agree within 1 %; the line reports the warm-up passes run next to `warmup_requested`.

--dump-outputs DIR writes what the last timed pass computed - the arrays a caller reads back from the handle - as
DIR/<name>.npy (float32 / float64, at most 64 MB in all).  The synthetic inputs depend on the workload's seed only, so
two builds run with the same arguments can be compared output for output.

One "step" = one complete sclens() pass (signal detection + robustness test, n_perturb=20) over
the synthetic count matrix of the workload.  Our arm:
  value  cells/s with the CSC counts already resident in HBM (library stream CUDA events)
  e2e    cells/s through the public API sclens_b200.sclens(X_host, handle=h): pinned host -> device copy of
         the CSC, the whole path, device -> host read of every result; the rank's handle (library context) is
         reused, a cold call that creates its own handle is reported beside it (B / small workloads)
  roofline   the dominant own kernel, the tcgen05 Gram: algorithmic n(n+1)K FLOP per launch over its
             CUDA-event time, against MEASURED_PEAKS.json; the HBM-bound densify kernel beside it
  cpu_baseline   the oracle (reference device_="cpu" numerics) timed on the host cores on a bounded
             sample and scaled to one sclens() pass (what was sampled is spelled out)
`--impl reference` times that CPU implementation as the reference arm.
Under torchrun (N>1) every rank owns one GPU; ranks cooperate on ONE sclens() pass ("strong").
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N cells, M genes, seed)  -- BASELINE.json configs[1], configs[2], configs[3], configs[4]
    "B": (10000, 20000, 0),
    "C": (68000, 20000, 1),
    "small": (2000, 3000, 3),
    "D": (500000, 25000, 2),
    "E": (68000, 20000, 1),
}
T_START = time.perf_counter()
# search steps the reference arm assumes (it runs before any GPU pass exists): the count our own pass takes on the
# same synthetic matrix (deterministic per workload and seed; measured on B200, profiles/r1_bench_*.json)
NOMINAL_SEARCH_STEPS = {"B": 14, "C": 14, "small": 14, "D": 14, "E": 14}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------
# synthetic counts (same recipe as sclens_b200.synth.make_counts; Poisson draws on the GPU when there is one)
# --------------------------------------------------------------------------------------
def make_counts_fast(N, M, seed, device=None):
    from sclens_b200 import synth
    if device is None:
        return synth.make_counts(N, M, seed=seed)
    import torch
    rng = np.random.default_rng(seed)
    K = 8
    prof = synth._profiles(M, K, rng, 0.10, 1.0)
    types = rng.integers(0, K, size=N)
    ldepth = rng.normal(0.0, 0.35, size=N)
    sub = rng.choice(N, size=min(N, 512), replace=False)
    min_cells = 40

    def floored(D):
        pmin = -np.log1p(-min(0.5, min_cells / N)) / D
        p = np.maximum(prof, pmin)
        return p / p.sum(axis=1, keepdims=True)

    def zero_frac(D):
        lam = (D * np.exp(ldepth[sub]))[:, None] * floored(D)[types[sub]]
        return float(np.exp(-lam).mean())

    lo, hi = 1.0, 1e7
    for _ in range(60):
        mid = np.sqrt(lo * hi)
        if zero_frac(mid) > 0.92:
            lo = mid
        else:
            hi = mid
    D = float(np.sqrt(lo * hi))
    p = torch.tensor(floored(D), dtype=torch.float32, device=device)
    depth = torch.tensor(D * np.exp(ldepth), dtype=torch.float32, device=device)
    ttypes = torch.tensor(types, device=device)
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    rows, cols, vals = [], [], []
    block = 4096
    for s in range(0, N, block):
        e = min(N, s + block)
        lam = depth[s:e, None] * p[ttypes[s:e]]
        c = torch.poisson(lam, generator=gen)
        nz = torch.nonzero(c)
        rows.append((nz[:, 0] + s).to(torch.int32).cpu().numpy())
        cols.append(nz[:, 1].to(torch.int32).cpu().numpy())
        vals.append(c[nz[:, 0], nz[:, 1]].cpu().numpy().astype(np.float32))
    X = sp.coo_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(N, M),
                      dtype=np.float32).tocsc()
    X.sort_indices()
    return X


# --------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------
# CPU arm: the oracle's device_="cpu" numerics (the reference's CPU path restated), each distinct stage timed once
# --------------------------------------------------------------------------------------
def cpu_stages(X, frac=1):
    """Times each distinct stage of the reference's CPU path (normalise :677-696, Float64 Gram :345-359, LAPACK eigen
    with vectors :384, corr_mat + column maximum :742) ONCE with all host cores, at full size (frac=1) or on the first
    1/frac of the smaller side.  Returns the measured seconds and the shape they were measured on."""
    from oracle import sclens_oracle as orc
    N, M = X.shape
    nm = min(N, M)
    if frac > 1:
        ns = max(300, nm // frac)
        Xs = X[:ns, :] if N <= M else X[:, :ns]
        Xs = Xs[:, np.diff(Xs.tocsc().indptr) > 0] if N <= M else Xs[np.diff(Xs.tocsr().indptr) > 0, :]
        Xs = sp.csc_matrix(Xs)
    else:
        Xs = X
    t = {}
    t0 = time.perf_counter()
    dense, _ = orc.normalize_main(Xs)                                   # :677-696 (Float64, dense)
    t["normalise"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    Y = orc.wishart_matrix(dense, 1 if N <= M else 2, "cpu")            # :345-359 Float64 syrk
    t["gram_f64"] = time.perf_counter() - t0
    shape = tuple(dense.shape)
    del dense
    t0 = time.perf_counter()
    L, V = orc.get_eigen(Y, "cpu")                                      # :384 LAPACK, all eigenpairs
    t["eigen_vectors"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    _ = np.abs(V.T @ V[:, : V.shape[1] // 2 + 1]).max(axis=0)           # corr_mat + nanmaximum (:742)
    t["corr"] = time.perf_counter() - t0
    return t, shape, int(Y.shape[0])


def cpu_pass_seconds(t, shape, n_s, N, M, n_search, n_perturb):
    """One sclens() pass of the reference's CPU path from the stage times: every get_sigev / get_eigvec call is
    normalise + Gram + eigen-with-vectors (:529-532, :492-494) - 2 in get_sigev, 1 reference basis, n_search search
    steps, n_perturb replicates - plus one corr_mat per search step; a sub-size measurement is scaled by N*M, n^2*K, n^3."""
    nm = min(N, M)
    lin = (N * M) / (shape[0] * shape[1])
    cube = (nm / n_s) ** 3
    gram_scale = (nm / n_s) ** 2 * (max(N, M) / (shape[1] if N <= M else shape[0]))
    n_full = 2 + 1 + n_search + n_perturb
    return n_full * (t["normalise"] * lin + t["gram_f64"] * gram_scale + t["eigen_vectors"] * cube) + n_search * t["corr"] * cube, n_full


def cpu_sample(X, n_search, n_perturb, frac=4):
    """Bounded sample for the cpu_baseline entry of our own line: stages on 1/frac of the smaller side."""
    N, M = X.shape
    cores = os.cpu_count() or 1
    t, shape, n_s = cpu_stages(X, frac)
    total, n_full = cpu_pass_seconds(t, shape, n_s, N, M, n_search, n_perturb)
    sample = (f"oracle cpu-mode stages timed once on a {shape[0]}x{shape[1]} sub-matrix (1/{frac} of the smaller side) with "
              f"{cores} cores: normalise {t['normalise']:.2f}s, f64 Gram {t['gram_f64']:.2f}s, LAPACK eig n={n_s} "
              f"{t['eigen_vectors']:.2f}s, corr {t['corr']:.2f}s; scaled by N*M, n^2*K, n^3 and the pass's stage counts "
              f"({n_full} normalise+Gram+eig incl. {n_search} search steps and {n_perturb} perturbations)")
    return total, cores, sample


def reference_arm(X, workload, n_search, n_perturb, budget_s):
    """--impl reference: the CPU path's stages measured ONCE AT FULL SIZE when that fits the budget (a 1/4-size probe
    predicts it), otherwise on the largest 1/frac sample that does; never repeated per requested step."""
    N, M = X.shape
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    tp, shp, n_p = cpu_stages(X, 4)      # the probe: a quarter of the smaller side (LAPACK is well into its n^3 regime there)
    probe_s = time.perf_counter() - t0
    ratio = min(N, M) / n_p
    pred_full = (tp["normalise"] * (N * M) / (shp[0] * shp[1]) + tp["gram_f64"] * ratio ** 2 +
                 (tp["eigen_vectors"] + tp["corr"]) * ratio ** 3)
    frac = 1
    while frac < 4 and pred_full / (frac ** 3) > budget_s:
        frac *= 2
    try:      # the Float64 dense pipeline holds ~5 copies of the N x M matrix at its peak: stay inside the host's free memory
        import psutil
        avail = psutil.virtual_memory().available
        while frac < 4 and 6.0 * N * M * 8.0 / frac > 0.8 * avail:
            frac *= 2
    except Exception:
        pass
    if frac >= 4:
        t, shape, n_s, measured_s = tp, shp, n_p, probe_s
    else:
        t0 = time.perf_counter()
        t, shape, n_s = cpu_stages(X, frac)
        measured_s = time.perf_counter() - t0
    total, n_full = cpu_pass_seconds(t, shape, n_s, N, M, n_search, n_perturb)
    size = "FULL size" if frac == 1 else f"1/{frac} of the smaller side"
    sample = (f"reference CPU path (oracle cpu mode = device_=\"cpu\" numerics) stages measured once at {size} "
              f"({shape[0]}x{shape[1]} dense, eig n={n_s}) with {cores} cores in {measured_s:.0f}s wall: "
              + ", ".join(f"{k} {v:.2f}s" for k, v in t.items())
              + f"; one pass = {n_full} x (normalise + Gram + eigen) + {n_search} x corr"
              + ("" if frac == 1 else "; scaled to full size by N*M, n^2*K, n^3")
              + f"; search steps nominal={n_search}, n_perturb={n_perturb}; 1/4-size probe predicted {pred_full:.0f}s for the full-size stages")
    return total, cores, sample, {"stage_seconds": t, "measured_at": list(shape), "eig_n": n_s, "frac": frac,
                                  "measured_wall_s": measured_s, "probe_wall_s": probe_s}


# --------------------------------------------------------------------------------------
def make_counts_csc_gpu(N, M, seed, device, gene_block=64):
    """Same recipe, generated gene block by gene block on the GPU so the entries come out in CSC order (no COO -> CSC
    conversion of 1e9 entries on the host): workload D."""
    import torch
    from sclens_b200 import synth
    rng = np.random.default_rng(seed)
    K = 8
    prof = synth._profiles(M, K, rng, 0.10, 1.0)
    types = rng.integers(0, K, size=N)
    ldepth = rng.normal(0.0, 0.35, size=N)
    sub = rng.choice(N, size=min(N, 512), replace=False)
    min_cells = 40

    def floored(D):
        pmin = -np.log1p(-min(0.5, min_cells / N)) / D
        p = np.maximum(prof, pmin)
        return p / p.sum(axis=1, keepdims=True)

    def zero_frac(D):
        lam = (D * np.exp(ldepth[sub]))[:, None] * floored(D)[types[sub]]
        return float(np.exp(-lam).mean())

    lo, hi = 1.0, 1e7
    for _ in range(60):
        mid = np.sqrt(lo * hi)
        if zero_frac(mid) > 0.92:
            lo = mid
        else:
            hi = mid
    D = float(np.sqrt(lo * hi))
    pT = torch.tensor(floored(D).T.copy(), dtype=torch.float32, device=device)      # M x K
    depth = torch.tensor(D * np.exp(ldepth), dtype=torch.float32, device=device)
    ttypes = torch.tensor(types, device=device)
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    rows, vals, counts = [], [], []
    for g0 in range(0, M, gene_block):
        g1 = min(M, g0 + gene_block)
        lam = pT[g0:g1][:, ttypes] * depth[None, :]                                  # genes x cells
        c = torch.poisson(lam, generator=gen)
        nz = torch.nonzero(c)                                                        # sorted by (gene, cell): CSC order
        counts.append(torch.bincount(nz[:, 0], minlength=g1 - g0).cpu().numpy())
        rows.append(nz[:, 1].to(torch.int32).cpu().numpy())
        vals.append(c[nz[:, 0], nz[:, 1]].cpu().numpy().astype(np.float32))
    indptr = np.concatenate([[0], np.cumsum(np.concatenate(counts))]).astype(np.int64)
    X = sp.csc_matrix((np.concatenate(vals), np.concatenate(rows), indptr), shape=(N, M), dtype=np.float32)
    X.has_sorted_indices = True
    return X


DUMP_LIMIT_BYTES = 64 << 20


def pass_outputs(h, si, ri):
    """Everything a caller reads back from the handle after a pass (scl_get_*), by name, as float32 / float64 arrays:
    the signal stage, and the robustness stage when the pass ran one (ri is None otherwise)."""
    out = {"L": h.L(), "L_mp": h.L_mp()}
    for k in ("n_signal", "n_Lmp", "lambda_c", "b_plus", "b_minus", "ks_static", "pass_"):
        out[k] = np.float64(getattr(si, k))
    if si.n_signal > 0:
        out["signal_ev"] = h.signal_ev()
        out["signal_evec"] = h.signal_evec()
        out.update({f"rec_{k}": v for k, v in h.rec_vals().items()})
    if ri is not None:
        for k in ("n_search", "min_pc", "n_robust", "n_add", "p_sel", "p_th", "n_subspace_fallbacks"):
            out[k] = np.float64(getattr(ri, k))
        out["gene_basis"] = h.gene_basis()
        out["b_"], out["m_scores"], out["sd_scores"] = h.scores()
        out["sig_id"] = h.sig_id().astype(np.float64)
        out["search_p"], out["search_d"] = h.search_trace()
    return out


def dump_outputs(outdir, arrays, limit=DUMP_LIMIT_BYTES):
    """DIR/<name>.npy for every array.  Should the whole exceed `limit`, each array over an equal share of it keeps a
    fixed, seeded sample of its longest axis; the sampled positions go to DIR/<name>_index.npy."""
    os.makedirs(outdir, exist_ok=True)
    share = limit // len(arrays) - 256          # two .npy headers
    sample = sum(np.asarray(a).nbytes for a in arrays.values()) > limit - 128 * len(arrays)
    written = 0
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        if sample and a.nbytes > share:
            ax = int(np.argmax(a.shape))
            keep = max(1, share // (a.nbytes // a.shape[ax] + 8))          # sampled slices + their float64 positions
            idx = np.sort(np.random.default_rng(0).choice(a.shape[ax], size=keep, replace=False))
            a = np.take(a, idx, axis=ax)
            np.save(os.path.join(outdir, f"{name}_index.npy"), idx.astype(np.float64))
            written += idx.size * 8
        np.save(os.path.join(outdir, f"{name}.npy"), a)
        written += a.nbytes
    return written


_REAL_STDOUT = None


def emit(line: str):
    """the one JSON line, on the process's original stdout"""
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        print(line, flush=True)
    else:
        os.write(_REAL_STDOUT, (line + "\n").encode())


def main():
    # stdout carries ONE JSON line.  Native libraries write there too (NCCL prints its version banner to stdout at
    # NCCL_DEBUG=VERSION and =WARN), so file descriptor 1 points at stderr for the whole run and the line goes to the saved one.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2, help="timed passes")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # default = the configuration BASELINE.json's metric is quoted on (68k x 20k, fits one GPU)
    ap.add_argument("--workload", default=os.environ.get("SCLENS_BENCH_WORKLOAD") or "C", choices=sorted(WORKLOADS))
    ap.add_argument("--n-perturb", type=int, default=None)
    ap.add_argument("--gram-mode", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed pass to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU pass; the reference arm times stages only")
    if args.n_perturb is None:
        args.n_perturb = 100 if args.workload == "E" else 20
    signal_only = args.workload == "D"

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    N, M, seed = WORKLOADS[args.workload]
    what = ("signal stage only (normalise, cell-sharded Gram, packed-triangle reduce, data + null eigensolves, MP/TW fit)"
            if signal_only else "full MP/TW fit + sparsity search + stability")
    config = {"workload": f"{args.workload}: synthetic {N} cells x {M} genes, ~92% sparse, n_perturb={args.n_perturb}, {what}",
              "N": N, "M": M, "l2": "inputs exceed L2 (dense operand >= 400 MB)",
              "parallelism": f"one sclens() pass shared by {world} rank(s): cell-sharded Gram, eigensolves of the pass spread over ranks, replicates r mod {world}"}

    if args.impl == "reference":
        if rank != 0:
            return
        X = make_counts_fast(N, M, seed)
        ref_budget = float(os.environ.get("SCLENS_REF_BUDGET_S", "420"))
        total, cores, sample, detail = reference_arm(X, args.workload, NOMINAL_SEARCH_STEPS[args.workload], args.n_perturb, ref_budget)
        v = N / total
        emit(json.dumps({"impl": "reference", "metric": "sclens_cells_per_s", "value": v, "unit": "cells/s",
                          "n_gpus": args.gpus, "steps": 1, "steps_requested": args.steps, "warmup": 0,
                          "warmup_requested": args.warmup, "ms_per_step": total * 1e3,
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": config,
                          "note": "ms_per_step is one full sclens() pass of the CPU path assembled from stage times measured once "
                                  "(cpu_baseline.sample); the stages are not re-run per requested step",
                          "cpu_baseline": {"value": v, "unit": "cells/s", "cores": cores, "kind": "port", "sample": sample,
                                           **detail},
                          "e2e": {"value": v, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    from sclens_b200 import Handle, sclens
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    t0 = time.perf_counter()
    X = make_counts_csc_gpu(N, M, seed, dev) if args.workload == "D" else make_counts_fast(N, M, seed, device=dev)
    log(f"[rank {rank}] synthetic counts {X.shape} nnz={X.nnz} sparsity={1 - X.nnz / (N * M):.4f} in {time.perf_counter() - t0:.1f}s")

    h = Handle(device=local_rank, gram_mode=args.gram_mode, seed=seed)

    def fresh_uid():
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            import ctypes as C
            buf = (C.c_uint8 * 128)()
            assert h.lib.scl_nccl_unique_id(buf) == 0
            uid = torch.tensor(list(buf), dtype=torch.uint8, device=dev)
        dist.broadcast(uid, 0)
        return bytes(uid.cpu().tolist())

    if world > 1:
        h.comm_init(fresh_uid(), rank, world)
    h.set_counts(X)

    def one_pass():
        if signal_only:      # scl_run_pass with n_perturb = 0: the signal stage alone, shared by the ranks
            return h.run_pass(th=60.0, p_step=0.001, n_perturb=0)[0], None
        return h.run_pass(th=60.0, p_step=0.001, n_perturb=args.n_perturb)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def agree(x, op):
        """one value on every rank (max / min over ranks)"""
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    # ---- warm-up: at least min(3, requested) passes; beyond that only until two consecutive passes agree within 1 %
    warm_s = []
    for i in range(args.warmup):
        barrier()
        t0 = time.perf_counter()
        si, ri = one_pass()
        barrier()
        warm_s.append(agree(time.perf_counter() - t0, dist.ReduceOp.MAX if world > 1 else None))
        log(f"[rank {rank}] warmup {i}: {warm_s[-1]:.2f}s n_signal={si.n_signal}" +
            ("" if ri is None else f" n_search={ri.n_search} p_sel={ri.p_sel:.3f} n_robust={ri.n_robust}"))
        if len(warm_s) >= 3 and abs(warm_s[-1] - warm_s[-2]) <= 0.01 * warm_s[-1]:
            break
    warm_done = len(warm_s)
    steps = args.steps

    h.reset_profile()
    launches0 = h.profile().kernel_launches
    clocks = ClockSampler(local_rank)
    clocks.start()
    barrier()
    h.timer_start()
    for _ in range(steps):
        si, ri = one_pass()
    ms = h.timer_stop()
    barrier()
    clk = clocks.stop()
    prof = h.profile()
    launches = prof.kernel_launches - launches0
    ms = agree(ms, dist.ReduceOp.MAX if world > 1 else None)
    ms_per_step = ms / steps
    value = N / (ms_per_step / 1e3)
    if args.dump_outputs and rank == 0:      # every rank holds the same results of the shared pass
        nbytes = dump_outputs(args.dump_outputs, pass_outputs(h, si, ri))
        log(f"[rank 0] outputs of the last timed pass: {nbytes / 2 ** 20:.1f} MB in {args.dump_outputs}")

    # ---- e2e through the public API with host buffers (pinned), results read back
    e2e = None
    if args.e2e_steps > 0 and not signal_only:
        try:
            pinned = [torch.from_numpy(a).pin_memory() for a in (X.indptr.astype(np.uint32).view(np.int32),
                                                                 X.indices.astype(np.uint32).view(np.int32), X.data)]
            Xp = sp.csc_matrix((pinned[2].numpy(), pinned[1].numpy().view(np.uint32), pinned[0].numpy().view(np.uint32)),
                               shape=X.shape)
            h2d = sum(int(p.numel() * p.element_size()) for p in pinned)
            d2h = 0

            def call(handle):
                out = sclens(Xp, n_perturb=args.n_perturb, gram_mode=args.gram_mode, verbose=False, seed=seed,
                             device=local_rank, handle=handle)
                nbytes = sum(int(np.asarray(v).nbytes) for v in (out["L"], out["L_mp"], out["signal_evec"], out["signal_ev"],
                                                                 out["gene_basis"], out["robustness_scores"]["b_"],
                                                                 out["robustness_scores"]["m_scores"],
                                                                 out["robustness_scores"]["sd_scores"], out["sig_id"]))
                nbytes += sum(int(np.asarray(v).nbytes) for v in out["rec_vals"].values())
                return nbytes, dict(out["info"]["host_ms"])

            # one cold call (N = 1, small workloads only): the call creates and destroys its own handle - cuSOLVER state and
            # every device workspace are set up inside it.  Reported beside the headline, not as the headline.
            cold_s, cold_host_ms = None, None
            if world == 1 and args.workload in ("B", "small"):
                barrier()
                t0 = time.perf_counter()
                _, cold_host_ms = call(None)
                barrier()
                cold_s = time.perf_counter() - t0
            # the timed calls reuse the rank's handle (the library context: workspaces, cuSOLVER state, NCCL communicator),
            # as a user running sclens() on one matrix after another would; host buffers in, every result read back
            e2e_s = 0.0
            e2e_host_ms = {}
            for _ in range(args.e2e_steps):
                barrier()
                t0 = time.perf_counter()
                d2h, e2e_host_ms = call(h)
                barrier()
                e2e_s += time.perf_counter() - t0
            e2e_s = agree(e2e_s / args.e2e_steps, dist.ReduceOp.MAX if world > 1 else None)
            e2e = {"value": N / e2e_s, "unit": "cells/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                   "seconds_per_step": e2e_s, "steps": args.e2e_steps, "host_ms_last_call": e2e_host_ms,
                   "handle": "reused across calls (device workspaces, cuSOLVER state and the NCCL communicator persist)",
                   "cold_call_seconds": cold_s, "cold_call_host_ms": cold_host_ms}
        except Exception as exc:      # the device-timed headline above must survive a failure of this leg
            if world > 1:
                raise                  # ranks must stay in step: a one-sided failure cannot be patched over
            e2e = {"value": None, "unit": "cells/s", "error": f"{type(exc).__name__}: {exc}"[:300]}

    if rank != 0:
        h.close()
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "MEASURED_PEAKS.json (sustained bf16 / copy)" if peaks else "fallback of B200_PROFILING.md"
    # DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed `ncu --set full`
    # captures of the same kernels at this workload's shapes (profiles/r2_traffic.json, else r1; null for other workloads)
    traffic = {}
    for name in ("r1_traffic.json", "r2_traffic.json"):
        try:
            traffic.update(json.load(open(os.path.join(ROOT, "profiles", name))).get(args.workload, {}))
        except Exception:
            pass

    def rate(work, ms_, scale):
        return work / (ms_ * 1e-3) / scale if ms_ > 0 else 0.0

    gram_tf = rate(prof.gram_alg_flops, prof.gram_gemm_ms, 1e12)
    dens_gbs = rate(prof.densify_alg_bytes, prof.densify_ms, 1e9)
    sparse_gbs = rate(prof.sparse_alg_bytes, prof.sparse_ms, 1e9)
    stats_gbs = rate(prof.stats_alg_bytes, prof.stats_ms, 1e9)
    roofline = {"kernel": "k_gemm_umma (tcgen05 Gram, syrk schedule)", "bound": "tensor", "achieved": gram_tf,
                "peak": tf_peak, "unit": "TFLOP/s", "frac": gram_tf / tf_peak, "traffic": traffic.get("k_gemm_umma"),
                "peak_source": peak_src, "launches": int(prof.gram_gemm_launches),
                "avg_ms_per_launch": prof.gram_gemm_ms / max(1, prof.gram_gemm_launches),
                "alg_flops_per_launch": prof.gram_alg_flops / max(1, prof.gram_gemm_launches),
                "hbm_kernel": {"kernel": "k_densify_tma2 (normalised dense binary16 operand: background + sparse patches composed in shared memory, TMA bulk stores)",
                               "bound": "hbm", "achieved": dens_gbs, "peak": hbm_peak, "unit": "GB/s",
                               "frac": dens_gbs / hbm_peak, "launches": int(prof.densify_launches),
                               "alg_bytes_per_launch": prof.densify_alg_bytes / max(1, prof.densify_launches),
                               "traffic": traffic.get("k_densify")},
                "sparse": {"kernels": "null-matrix permutation + perturbation merge (k_merge_lines and helpers)", "bound": "hbm",
                           "achieved": sparse_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": sparse_gbs / hbm_peak,
                           "calls": int(prof.sparse_calls), "alg_bytes": "20 nnz per null permutation, 8 nnz + 12 n_add per merge (SURVEY 8d)",
                           "avg_ms_per_call": prof.sparse_ms / max(1, prof.sparse_calls)},
                "stats": {"kernels": "statistics line passes (k_row_sum, k_lines<...>, reductions)", "bound": "hbm",
                          "achieved": stats_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": stats_gbs / hbm_peak,
                          "calls": int(prof.stats_calls), "alg_bytes": "40 nnz per normalisation (4 nnz + 3 x 8 nnz + 12 nnz patch pass)",
                          "avg_ms_per_call": prof.stats_ms / max(1, prof.stats_calls)}}
    # the eigensolves: own two-stage solver (dense -> band -> tridiagonal -> Float64 tridiagonal stage -> Q2, Q1) since round 2;
    # cuSOLVER runs only when a solve falls back (counted).  Stage totals come from the solver's own CUDA events.
    eig = np.zeros(8)
    h.lib.scl_debug_eig_stage_totals(h.h, eig.ctypes.data_as(C.POINTER(C.c_double)))
    n_eig = min(N, M)
    q_blk = (n_eig - 3) // 64
    nblk = (q_blk + 1) * (q_blk + 2) // 2
    q2_exec = eig[6] / 16.0 * nblk * 300 * 4096.0        # 300 m16n8k16 MMAs per 16 vectors and reflector block
    q2_peak = 148 * 4 * 4096 / 8.0 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12   # one mma.sync per 8 cycles and sub-partition
    roofline["eigensolver"] = {
        "solver": "own two-stage reduction (sy2sb.cu, sb2st.cu, tridiag.cu, backtrans.cu); cuSOLVER only on fallback",
        "solves": int(eig[5]), "fallbacks_to_one_stage": int(eig[7]), "eigenvector_columns_back_transformed": int(eig[6]),
        "ms_by_stage": {"dense_to_band": eig[0], "band_to_tridiagonal": eig[1], "tridiagonal_eigenproblem_f64": eig[2],
                        "back_transformation_q2": eig[3], "back_transformation_q1": eig[4]},
        "q2_kernel": {"kernel": "k_q2_apply_h (register-stationary block reflectors, split binary16 on mma.sync m16n8k16)",
                      "bound": "tensor (warp-level path)", "achieved": rate(q2_exec, eig[3], 1e12), "peak": q2_peak,
                      "unit": "TFLOP/s executed", "frac": rate(q2_exec, eig[3], 1e12) / q2_peak if q2_peak else None,
                      "peak_source": "scripts/mma_rate.cu measured on B200: 8 cycles per mma.sync per sub-partition, at sm_max_mhz",
                      "alg_flops": 2.0 * n_eig * n_eig * eig[6],
                      "note": "executed = 3 MMAs per step (hi hi, lo hi, hi lo) x the compact-WY block form; algorithmic = 2 n^2 per vector"}}
    stage_ms = {"gram_gemm": prof.gram_gemm_ms, "other_gemm": prof.other_gemm_ms, "densify": prof.densify_ms,
                "stats": prof.stats_ms, "sparse": prof.sparse_ms, "eigensolves": prof.syevd_ms, "syevd_library": prof.syevd_ms,
                "syevd_library_note": "historical key: since round 2 these are the own eigensolver's kernels (see roofline.eigensolver)",
                "syevd_calls": int(prof.syevd_calls), "refine_f64": prof.refine_ms, "small": prof.small_ms,
                "nccl_collectives": prof.comm_ms, "nccl_payload_bytes": prof.comm_bytes, "total": ms}
    phase = {"signal_normalise_gram": si.t_gram_ms, "signal_syevd": si.t_syevd_ms, "null_matrix": si.t_null_ms,
             "mp_fit_host": si.t_fit_ms, "backproject": si.t_backproject_ms}
    result = {"n_signal": si.n_signal, "lambda_c": si.lambda_c}
    if ri is not None:
        phase.update({"noise_baseline_and_zero_candidates": ri.t_baseline_ms, "search_total": ri.t_search_ms,
                      "search_syevd": ri.t_search_syevd_ms, "perturbations": ri.t_perturb_ms,
                      "scores": ri.t_score_ms, "gene_basis": ri.t_outputs_ms})
        result.update({"n_search": ri.n_search, "p_sel": ri.p_sel, "n_robust": ri.n_robust,
                       "n_subspace_fallbacks": ri.n_subspace_fallbacks})
    line = {"metric": "sclens_cells_per_s", "value": value, "unit": "cells/s", "n_gpus": world, "steps": steps,
            "steps_requested": args.steps, "warmup": warm_done, "warmup_requested": args.warmup,
            "warmup_seconds": warm_s, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f16 operands / f32 accumulate (Gram), f32 eigensolver (split-f16 / three-term tf32 tensor-core products, f64 tridiagonal stage), f64 statistics",
            "data": "synthetic", "config": config, "clocks": clk, "gpu_launches": int(launches),
            "roofline": roofline, "stage_ms_over_timed_region": stage_ms, "phase_ms": phase, "phase_ms_last_step": phase,
            "gemm_tflops": {"other_gemm_2mnk": rate(prof.other_gemm_flops, prof.other_gemm_ms, 1e12)},
            "result": result, "wall_s_at_line": None}
    if ri is not None and ri.t_perturb_ms > 0:
        line["perturbation_replicates_per_s"] = args.n_perturb / (ri.t_perturb_ms * 1e-3)
    if e2e is not None:
        line["e2e"] = e2e
    if world == 1 and not args.no_cpu_baseline and not signal_only:
        try:
            total, cores, sample = cpu_sample(X, ri.n_search, args.n_perturb)
            line["cpu_baseline"] = {"value": N / total, "unit": "cells/s", "cores": cores, "kind": "port", "sample": sample,
                                    "seconds_per_pass_estimate": total}
        except Exception as exc:          # e.g. host memory: report it, keep the line
            line["cpu_baseline"] = {"value": None, "unit": "cells/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"failed: {type(exc).__name__}: {exc}"[:300]}
    line["wall_s_at_line"] = time.perf_counter() - T_START
    emit(json.dumps(line))
    h.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
