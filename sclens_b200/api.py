"""Host-side mirror of the reference interface for the hot path:

    scLENS.sclens(inp_df; device_="gpu", th=60, p_step=0.001, n_perturb=20, centering="mean")
    (/root/reference/src/scLENS.jl:649) -> Dict with the keys of :826-830.

Everything numeric happens behind the C ABI (libsclens_b200.so); this module only converts
the DataFrame to CSC (df2sparr, :90-120), calls the library and assembles the result
dictionary.  The Julia binding a maintainer would add does exactly the same through
``ccall`` (see INTEGRATION.md and julia/sclens_b200.jl).
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import numpy as np
import scipy.sparse as sp

try:   # DataFrames in, DataFrames out (as the reference); imported once here, not inside a call
    import pandas as pd
except ImportError:  # pragma: no cover
    pd = None

from . import _lib
from ._lib import Config, Profile, RobustInfo, SclError, SignalInfo, UmapInfo, UmapParams, as_f32, as_u32, ptr


def df2sparr(inp_df):
    """df2sparr (:90-120): DataFrame (col 0 = 'cell', then genes) -> canonical CSC Float32 with
    UInt32 indices, plus cell and gene ids.  scipy sparse / ndarray inputs are accepted too."""
    if pd is not None and isinstance(inp_df, pd.DataFrame):
        cell_id = inp_df.iloc[:, 0].astype(str).to_numpy()
        genes = inp_df.columns[1:]
        body = inp_df.iloc[:, 1:]
        if all(isinstance(t, pd.SparseDtype) for t in body.dtypes):
            X = sp.csc_matrix(body.sparse.to_coo(), dtype=np.float32)
        else:
            X = sp.csc_matrix(body.to_numpy(dtype=np.float32))
        gene_id = np.asarray(genes, dtype=object)
    else:
        X = inp_df if (sp.isspmatrix_csc(inp_df) and inp_df.dtype == np.float32) else sp.csc_matrix(inp_df, dtype=np.float32)
        cell_id = np.array([f"c{i}" for i in range(X.shape[0])], dtype=object)
        gene_id = np.array([f"g{j}" for j in range(X.shape[1])], dtype=object)
    # canonical CSC with strictly positive stored values is what the C ABI takes; an input that already is
    # canonical (one O(nnz) check) is passed through without a copy
    if not X.has_canonical_format:
        X = X.copy()
        X.sum_duplicates()
    if X.nnz and float(X.data.min()) <= 0.0:
        X = X.copy()
        X.eliminate_zeros()
    return X, cell_id, gene_id


def speculative_search_merge(d2_in_step_order, p_th, p_step=0.001, tank_n=5):
    """Stop rule of the sparsity search (:748-760) applied in step order to second-smallest values that
    ranks evaluated speculatively (step s used p_ = 0.999 - s*p_step).  Returns (n_steps, p_selected)
    once the rule fires, else None - identical to running the loop sequentially.  Mirrors the C++ logic
    of run_robustness for the multi-rank search; pure host code."""
    p_ = 0.999
    for step in range(len(d2_in_step_order)):
        last = d2_in_step_order[max(0, step + 1 - tank_n): step + 1]
        if (sum(x < p_th for x in last) > tank_n - 1) or p_ < 0.9:
            return step + 1, p_ + (tank_n - 1) * p_step
        p_ -= p_step
    return None


class Handle:
    """Owns one scl_handle (all device state of one sclens() call)."""

    def __init__(self, device: int = 0, gram_mode: int = _lib.SCL_GRAM_FP16, cta_group: int = 0, verbose: bool = False,
                 seed: int = 0, exact_perturb: bool = False, subspace_extra: int = 0, subspace_degree: int = 0,
                 gram_chunk_kb: int = 0, gram_tc_diag: int = 0, no_refine: bool = False, centering: str = "mean"):
        self.lib = _lib.load()
        cfg = Config(device=device, gram_mode=gram_mode, cta_group=cta_group, verbose=int(verbose), seed=seed,
                     subspace_extra=subspace_extra, subspace_degree=subspace_degree, exact_perturb=int(exact_perturb),
                     gram_chunk_kb=int(gram_chunk_kb), gram_tc_diag=int(gram_tc_diag), no_refine=int(no_refine),
                     centering=1 if centering == "median" else 0)
        self.centering = "median" if centering == "median" else "mean"
        self.h = C.c_void_p()
        rc = self.lib.scl_create(C.byref(self.h), C.byref(cfg))
        if rc != 0:
            raise SclError(rc, (self.lib.scl_last_error(None) or b"").decode())
        self.sinfo: Optional[SignalInfo] = None
        self.rinfo: Optional[RobustInfo] = None
        self.N = self.M = 0
        self.world, self.rank = 1, 0

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.scl_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise SclError(rc, (self.lib.scl_last_error(self.h) or b"").decode())

    # ---- inputs / draws
    def set_counts(self, X: sp.csc_matrix):
        X = sp.csc_matrix(X, dtype=np.float32)
        X.sort_indices()
        self.N, self.M = X.shape
        colptr, rowval, val = as_u32(X.indptr), as_u32(X.indices), as_f32(X.data)
        self._ck(self.lib.scl_set_counts_csc(self.h, self.N, self.M, X.nnz, ptr(colptr, C.c_uint32),
                                             ptr(rowval, C.c_uint32), ptr(val, C.c_float), 0))

    def set_zero_candidates(self, z1, z2):
        z1, z2 = as_u32(z1), as_u32(z2)
        self._ck(self.lib.scl_set_zero_candidates(self.h, len(z1), ptr(z1, C.c_uint32), ptr(z2, C.c_uint32), 0))

    def set_null_draws(self, perm, rows):
        perm, rows = as_u32(perm), as_u32(rows)
        self._ck(self.lib.scl_set_null_draws(self.h, len(perm), ptr(perm, C.c_uint32), ptr(rows, C.c_uint32), 0))

    def set_noise_baseline(self, p_th: float):
        self._ck(self.lib.scl_set_noise_baseline(self.h, float(p_th)))

    def push_search_sample(self, s):
        s = as_u32(s)
        self._ck(self.lib.scl_push_search_sample(self.h, len(s), ptr(s, C.c_uint32), 0))

    def push_perturb_sample(self, s):
        s = as_u32(s)
        self._ck(self.lib.scl_push_perturb_sample(self.h, len(s), ptr(s, C.c_uint32), 0))

    def comm_init(self, uid: bytes, rank: int, world: int):
        """Join the NCCL communicator of a cooperative pass.  A handle that already is rank `rank` of `world` keeps its
        communicator (the library ignores the new id), so sclens(handle=h, comm=...) can be called again and again."""
        buf = (C.c_uint8 * 128).from_buffer_copy(uid)
        self._ck(self.lib.scl_comm_init(self.h, buf, rank, world))
        self.world, self.rank = world, rank

    def profile(self) -> Profile:
        p = Profile()
        self._ck(self.lib.scl_get_profile(self.h, C.byref(p)))
        return p

    def timer_start(self):
        self._ck(self.lib.scl_timer_start(self.h))

    def timer_stop(self) -> float:
        ms = C.c_double()
        self._ck(self.lib.scl_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def reset_profile(self):
        self._ck(self.lib.scl_reset_profile(self.h))

    # ---- the path
    def run_signal(self) -> SignalInfo:
        info = SignalInfo()
        self._ck(self.lib.scl_run_signal(self.h, C.byref(info)))
        self.sinfo = info
        return info

    def run_robustness(self, th=60.0, p_step=0.001, n_perturb=20) -> RobustInfo:
        info = RobustInfo()
        self._ck(self.lib.scl_run_robustness(self.h, float(th), float(p_step), int(n_perturb), C.byref(info)))
        self.rinfo = info
        return info

    def run_pass(self, th=60.0, p_step=0.001, n_perturb=20):
        """Both stages in one call (scl_run_pass): on several ranks the eigensolves of the pass are dealt to the ranks.
        Returns (SignalInfo, RobustInfo); RobustInfo is None when there is no signal (:780-784)."""
        si, ri = SignalInfo(), RobustInfo()
        self._ck(self.lib.scl_run_pass(self.h, float(th), float(p_step), int(n_perturb), C.byref(si), C.byref(ri)))
        self.sinfo = si
        self.rinfo = ri if (si.n_signal > 0 and n_perturb > 0) else None
        return si, self.rinfo

    # ---- results
    def _getf(self, fn, n, dtype=np.float32, ctype=C.c_float):
        out = np.empty(n, dtype=dtype)
        self._ck(fn(self.h, ptr(out, ctype)))
        return out

    def L(self):
        return self._getf(self.lib.scl_get_L, self.sinfo.nm)

    def L_mp(self):
        return self._getf(self.lib.scl_get_Lmp, self.sinfo.n_Lmp)

    def signal_ev(self):
        return self._getf(self.lib.scl_get_signal_ev, self.sinfo.n_signal)

    def signal_evec(self):
        """N x n_signal (unit columns)."""
        k = self.sinfo.n_signal
        out = np.empty((k, self.N), dtype=np.float32)
        if k:
            self._ck(self.lib.scl_get_signal_evec(self.h, ptr(out, C.c_float)))
        return out.T

    def gene_basis(self):
        """n_signal x M."""
        k = self.sinfo.n_signal
        out = np.empty((self.M, k), dtype=np.float32)
        self._ck(self.lib.scl_get_gene_basis(self.h, ptr(out, C.c_float)))
        return out.T

    def rec_vals(self):
        N, M = self.N, self.M
        tgc, l2 = np.empty(N), np.empty(N)
        mean, sd, cent = np.empty(M), np.empty(M), np.empty(M)
        self._ck(self.lib.scl_get_rec_vals(self.h, ptr(tgc, C.c_double), ptr(mean, C.c_double), ptr(sd, C.c_double),
                                           ptr(l2, C.c_double), ptr(cent, C.c_double)))
        return {"TGC": tgc, "mat2_mean": mean.reshape(1, M), "mat2_std": sd.reshape(1, M), "norm_tgc": l2,
                "cent_": cent.reshape(1, M)}

    def scores(self):
        k, P = self.sinfo.n_signal, self.rinfo.n_perturb
        npairs = P * (P - 1) // 2
        b = np.empty((npairs, k), dtype=np.float32)
        m, sd = np.empty(k), np.empty(k)
        self._ck(self.lib.scl_get_scores(self.h, ptr(b, C.c_float), ptr(m, C.c_double), ptr(sd, C.c_double)))
        return b.T, m, sd

    def sig_id(self):
        out = np.empty(self.rinfo.n_robust, dtype=np.int32)
        if len(out):
            self._ck(self.lib.scl_get_sig_id(self.h, ptr(out, C.c_int32)))
        return out

    def null_csc(self) -> sp.csc_matrix:
        nnz = C.c_int64()
        self._ck(self.lib.scl_get_null_csc(self.h, C.byref(nnz), None, None, None))
        colptr = np.empty(self.M + 1, np.uint32)
        rowval = np.empty(max(1, nnz.value), np.uint32)
        val = np.empty(max(1, nnz.value), np.float32)
        self._ck(self.lib.scl_get_null_csc(self.h, C.byref(nnz), ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32),
                                           ptr(val, C.c_float)))
        return sp.csc_matrix((val[:nnz.value], rowval[:nnz.value].astype(np.int64), colptr.astype(np.int64)),
                             shape=(self.N, self.M))

    def search_trace(self):
        n = self.rinfo.n_search
        p, d = np.empty(n), np.empty(n)
        self._ck(self.lib.scl_get_search_trace(self.h, ptr(p, C.c_double), ptr(d, C.c_double)))
        return p, d

    def perturbed_evec(self, r):
        mp = self.rinfo.min_pc
        V = np.empty((mp, self.N), dtype=np.float32)
        L = np.empty(mp, dtype=np.float32)
        self._ck(self.lib.scl_get_perturbed_evec(self.h, r, ptr(V, C.c_float), ptr(L, C.c_float)))
        return V.T, L

    # ---- apply_umap stages (scl_op_knn / scl_op_umap)
    def knn(self, X, k=15, metric="cosine"):
        """Exact kNN of the rows of X (N x d): (idx, dist), both N x k, self excluded, ascending (distance, index)."""
        Xc = _umap_matrix(X)
        N, d = Xc.shape[1], Xc.shape[0]
        k, m = _umap_k(k, N), _umap_metric(metric)
        idx, dist = np.empty((N, k), np.int32), np.empty((N, k), np.float32)
        self._ck(self.lib.scl_op_knn(self.h, N, d, ptr(Xc, C.c_float), k, m, ptr(idx, C.c_int32), ptr(dist, C.c_float)))
        return idx, dist

    def umap(self, X, k=15, nc=2, md=0.1, metric="cosine", *, n_epochs=300, seed=0, init="spectral", init_embedding=None,
             spread=1.0, learning_rate=1.0, repulsion_strength=1.0, neg_sample_rate=5, local_connectivity=1.0,
             spectral_maxiter=100):
        """UMAP_ of apply_umap! on the rows of X (N x d): returns (embedding N x nc, UmapInfo).  ``init_embedding``
        (N x nc) replaces the computed start.  The kNN and the fuzzy graph stay on the handle (umap_graph, umap_knn)."""
        Xc = _umap_matrix(X)
        N, d = Xc.shape[1], Xc.shape[0]
        p = _umap_params(N, k, nc, md, metric, n_epochs, seed, init, spread, learning_rate, repulsion_strength,
                         neg_sample_rate, local_connectivity, spectral_maxiter)
        ie = None
        if init_embedding is not None:
            ie = np.ascontiguousarray(np.asarray(init_embedding, dtype=np.float32).T)    # N x nc column-major
            if ie.shape != (p.n_components, N) or not np.isfinite(ie).all():
                raise ValueError("init_embedding must be a finite N x nc array")
        out = np.empty((p.n_components, N), np.float32)
        info = UmapInfo()
        self._ck(self.lib.scl_op_umap(self.h, N, d, ptr(Xc, C.c_float), C.byref(p), ptr(ie, C.c_float), ptr(out, C.c_float),
                                      C.byref(info)))
        self.umap_N, self.umap_k = N, p.n_neighbors
        return out.T.copy(), info

    def umap_graph(self) -> sp.csr_matrix:
        nnz = C.c_int64()
        self._ck(self.lib.scl_get_umap_graph(self.h, C.byref(nnz), None, None, None))
        N = self.umap_N
        rp, ci, v = np.empty(N + 1, np.uint32), np.empty(max(1, nnz.value), np.uint32), np.empty(max(1, nnz.value), np.float32)
        self._ck(self.lib.scl_get_umap_graph(self.h, C.byref(nnz), ptr(rp, C.c_uint32), ptr(ci, C.c_uint32), ptr(v, C.c_float)))
        n = nnz.value
        return sp.csr_matrix((v[:n], ci[:n].astype(np.int64), rp.astype(np.int64)), shape=(N, N))

    def umap_knn(self):
        N, k = self.umap_N, self.umap_k
        idx, dist = np.empty((N, k), np.int32), np.empty((N, k), np.float32)
        self._ck(self.lib.scl_get_umap_knn(self.h, ptr(idx, C.c_int32), ptr(dist, C.c_float)))
        return idx, dist


_UMAP_METRICS = {"euclidean": 0, "cosine": 1}
_UMAP_INITS = {"spectral": 0, "random": 1}


def _umap_matrix(X):
    """N x d host matrix -> C-order d x N Float32 (== N x d column-major), checked finite."""
    if pd is not None and isinstance(X, pd.DataFrame):
        X = X.iloc[:, 1:].to_numpy() if X.shape[1] and X.columns[0] == "cell" else X.to_numpy()
    X = np.asarray(X, dtype=np.float32)
    if X.ndim != 2 or X.shape[0] < 2 or X.shape[1] < 1 or X.shape[1] > 1024:
        raise ValueError("need an N x d matrix with N >= 2 and 1 <= d <= 1024")
    if not np.isfinite(X).all():
        raise ValueError("the input has non-finite entries")
    return np.ascontiguousarray(X.T)


def _umap_k(k, N):
    k = int(k)
    if not (1 <= k <= 64) or k >= N:
        raise ValueError(f"n_neighbors must satisfy 1 <= k <= 64 and k < N (k = {k}, N = {N})")
    return k


def _umap_metric(metric):
    m = getattr(metric, "lower", lambda: None)()
    if m not in _UMAP_METRICS:
        raise ValueError(f"metric must be one of {sorted(_UMAP_METRICS)}, got {metric!r}")
    return _UMAP_METRICS[m]


def _umap_params(N, k, nc, md, metric, n_epochs, seed, init, spread, learning_rate, repulsion_strength, neg_sample_rate,
                 local_connectivity, spectral_maxiter):
    k = _umap_k(k, N)
    if not (1 <= int(nc) <= 16):
        raise ValueError("nc must be in [1, 16]")
    if init not in _UMAP_INITS:
        raise ValueError(f"init must be one of {sorted(_UMAP_INITS)}, got {init!r}")
    if int(n_epochs) < 0 or int(neg_sample_rate) < 0 or int(spectral_maxiter) < 0:
        raise ValueError("n_epochs, neg_sample_rate and spectral_maxiter must be >= 0")
    vals = dict(min_dist=float(md), spread=float(spread), learning_rate=float(learning_rate),
                repulsion_strength=float(repulsion_strength), local_connectivity=float(local_connectivity))
    if not all(math.isfinite(v) for v in vals.values()) or vals["min_dist"] < 0 or vals["spread"] <= 0 \
            or vals["learning_rate"] <= 0 or vals["repulsion_strength"] < 0 or not (0 <= vals["local_connectivity"] <= k):
        raise ValueError(f"bad UMAP parameters {vals}")
    return UmapParams(n_neighbors=k, n_components=int(nc), n_epochs=int(n_epochs), metric=_umap_metric(metric),
                      init=_UMAP_INITS[init], neg_sample_rate=int(neg_sample_rate), spectral_maxiter=int(spectral_maxiter),
                      seed=int(seed) & (2 ** 64 - 1), **vals)


def sclens(inp_df, device_="gpu", th=60, p_step=0.001, n_perturb=20, centering="mean", *, draws=None, seed=0,
           gram_mode=_lib.SCL_GRAM_FP16, exact_perturb=False, verbose=True, device=0, return_handle=False, comm=None, handle=None):
    """Drop-in for scLENS.sclens (:649-832).  Returns the reference's result dictionary with
    string keys (":pca" -> "pca", ...; "λ" is also available as "lambda").  ``sig_id`` is
    0-based here (the Julia shim adds 1).  ``draws`` optionally injects the random draws
    (an object with the fields of oracle Draws) for parity runs.  ``comm=(nccl_unique_id_bytes, rank, world)``
    makes this call one rank of a cooperative multi-GPU pass (one process per GPU; every rank passes the same
    counts and receives the same results).  ``handle`` reuses an existing Handle (its device workspaces, cuSOLVER
    state and, if initialised, its NCCL communicator) instead of creating one; the caller keeps ownership."""
    if device_ != "gpu":
        raise ValueError('sclens_b200 implements device_="gpu" only (no CPU fallback exists)')
    if centering not in ("mean", "median"):                             # :655-657
        print("Warning: The specified centering method is not supported in the current algorithm. scLENS will automatically "
              "use mean centering.")
        centering = "mean"
    if handle is not None and handle.centering != centering:
        raise ValueError(f"the handle was created for centering={handle.centering!r}")
    if verbose:
        print("Extracting matrices")                                    # :661
    import time as _time
    _t = [_time.perf_counter()]

    def _lap():
        _t.append(_time.perf_counter())
        return 1e3 * (_t[-1] - _t[-2])

    host_ms = {}
    X, cell_id, gene_id = df2sparr(inp_df)
    host_ms["df2sparr"] = _lap()
    N, M = X.shape
    own = handle is None
    h = Handle(device=device, gram_mode=gram_mode, verbose=verbose, seed=seed, exact_perturb=exact_perturb,
               centering=centering) if own else handle
    host_ms["create_handle"] = _lap()
    try:
        if comm is not None:
            h.comm_init(*comm)
        h.set_counts(X)
        host_ms["upload_counts_and_csr_mirror"] = _lap()
        if draws is not None:
            if getattr(draws, "z_idx1", None) is not None:
                h.set_zero_candidates(draws.z_idx1, draws.z_idx2)
            if getattr(draws, "null_perm", None) is not None:
                h.set_null_draws(draws.null_perm, draws.null_rows)
            if getattr(draws, "p_th", None) is not None:
                h.set_noise_baseline(draws.p_th)
            for s in getattr(draws, "search_sple", []) or []:
                h.push_search_sample(s)
            for s in getattr(draws, "perturb_sple", []) or []:
                h.push_perturb_sample(s)
        if verbose:
            print("Extracting Signals...")                              # :702
        _lap()
        cooperative = h.world > 1
        if cooperative:
            # one pass shared by the ranks: the eigensolves of both stages are dealt out together (scl_run_pass)
            si, ri = h.run_pass(th=th, p_step=p_step, n_perturb=n_perturb)
            host_ms["run_pass"] = _lap()
        else:
            si = h.run_signal()
            host_ms["run_signal"] = _lap()
        L, L_mp = h.L(), h.L_mp()
        results = {"L": L, "L_mp": L_mp, "λ": si.lambda_c, "lambda": si.lambda_c, "cell_id": cell_id}
        if si.n_signal == 0:                                            # :780-784
            if verbose:
                print("warning: There is no signal")
            return (results, h) if return_handle else results
        if verbose:
            print("Calculating noise baseline...")                      # :707
            print("Calculating sparsity level for the perturbation...")  # :716
        if not cooperative:
            _lap()
            ri = h.run_robustness(th=th, p_step=p_step, n_perturb=n_perturb)
            host_ms["run_robustness"] = _lap()
        nV, nL = h.signal_evec(), h.signal_ev()
        b_, m_scores, sd_scores = h.scores()
        sig_id = h.sig_id()
        if verbose:
            print("Reconstructing reduced data...")                     # :809
        sq = np.sqrt(nL.astype(np.float32))
        Xout0 = nV * sq[None, :]                                        # :810
        Xout1 = nV[:, sig_id] * sq[sig_id][None, :]                     # :811

        def frame(mat):
            if pd is None:
                return mat
            df = pd.DataFrame(mat, columns=[f"x{i + 1}" for i in range(mat.shape[1])])
            df.insert(0, "cell", cell_id)
            return df

        results.update({
            "pca": frame(Xout0), "pca_n1": frame(Xout1), "sig_id": sig_id,
            "robustness_scores": {"b_": b_, "rob_score": m_scores, "m_scores": m_scores, "sd_scores": sd_scores},
            "signal_evec": nV, "signal_ev": nL, "gene_id": gene_id, "gene_basis": h.gene_basis(),
            "pass": bool(si.pass_), "rec_vals": h.rec_vals() if centering == "mean" else {},   # mean path only (:676-695)
            "info": {"host_ms": host_ms, "p_sel": ri.p_sel, "n_search": ri.n_search, "p_th": ri.p_th, "min_pc": ri.min_pc,
                     "n_add": ri.n_add, "n_subspace_fallbacks": ri.n_subspace_fallbacks, "ks_static": si.ks_static, "b_plus": si.b_plus, "b_minus": si.b_minus,
                     "timings_ms": {"gram": si.t_gram_ms, "syevd_signal": si.t_syevd_ms, "null": si.t_null_ms,
                                    "fit": si.t_fit_ms, "backproject": si.t_backproject_ms,
                                    "baseline": ri.t_baseline_ms, "search": ri.t_search_ms,
                                    "search_syevd": ri.t_search_syevd_ms, "perturb": ri.t_perturb_ms,
                                    "score": ri.t_score_ms, "outputs": ri.t_outputs_ms}},
        })
        host_ms["read_results"] = _lap()
        return (results, h) if return_handle else results
    finally:
        if own and not return_handle:
            h.close()


def qc_indices_device(X, gene_name, min_tp_c=0, min_tp_g=0, max_tp_c=np.inf, max_tp_g=np.inf, min_genes_per_cell=200,
                      max_genes_per_cell=0, min_cells_per_gene=15, mito_percent=5.0, ribo_percent=0.0, *, device=0, handle=None):
    """The filters of scLENS.preprocess (:183-225) on the device (``scl_op_preprocess``): returns ``(fc_idx, gene_idx,
    filtered CSC)`` - kept cells (ascending), kept genes in output order (stable sort by Float32 mean) and the filtered
    matrix - or None when nothing survives.  The filtered matrix stays on the handle as its counts, so ``sclens(...,
    handle=h)`` can follow without another upload.  Only the regular expressions over the gene names run on the host."""
    import re
    X = sp.csc_matrix(X, dtype=np.float32)
    if not X.has_canonical_format:
        X.sum_duplicates()
    X.eliminate_zeros()
    X.sort_indices()
    N, M = X.shape
    flags = np.zeros(M, np.uint8)
    for j, g in enumerate(gene_name):
        g = str(g)
        flags[j] = (1 if re.match(r"^mt-.", g, flags=re.I) else 0) | (2 if re.match(r"^RP[SL].", g, flags=re.I) else 0)   # :196-197
    qp = _lib.QcParams(min_tp_c=float(min_tp_c), min_tp_g=float(min_tp_g), max_tp_c=float(max_tp_c), max_tp_g=float(max_tp_g),
                       min_genes_per_cell=int(min_genes_per_cell), max_genes_per_cell=int(max_genes_per_cell),
                       min_cells_per_gene=int(min_cells_per_gene), mito_percent=float(mito_percent), ribo_percent=float(ribo_percent))
    own = handle is None
    h = Handle(device=device) if own else handle
    try:
        colptr, rowval, val = as_u32(X.indptr), as_u32(X.indices), as_f32(X.data)
        nc, ng, nnz = C.c_int32(), C.c_int32(), C.c_int64()
        fc, gi = np.empty(N, np.int32), np.empty(M, np.int32)
        h._ck(h.lib.scl_op_preprocess(h.h, N, M, X.nnz, ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32), ptr(val, C.c_float), 0,
                                      flags.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(qp), C.byref(nc), C.byref(ng),
                                      C.byref(nnz), ptr(fc, C.c_int32), ptr(gi, C.c_int32)))
        if nc.value == 0 or ng.value == 0:
            return None
        h.N, h.M = nc.value, ng.value
        oc, orow, oval = np.empty(ng.value + 1, np.uint32), np.empty(max(1, nnz.value), np.uint32), np.empty(max(1, nnz.value), np.float32)
        h._ck(h.lib.scl_get_counts_csc(h.h, ptr(oc, C.c_uint32), ptr(orow, C.c_uint32), ptr(oval, C.c_float)))
        out = sp.csc_matrix((oval[:nnz.value], orow[:nnz.value].astype(np.int64), oc.astype(np.int64)), shape=(nc.value, ng.value))
        return fc[:nc.value].copy(), gi[:ng.value].copy(), out
    finally:
        if own:
            h.close()


def preprocess(tmp_df, min_tp_c=0, min_tp_g=0, max_tp_c=np.inf, max_tp_g=np.inf, min_genes_per_cell=200, max_genes_per_cell=0,
               min_cells_per_gene=15, mito_percent=5.0, ribo_percent=0.0, *, verbose=True, device=0, handle=None):
    """Drop-in for scLENS.preprocess (:160-236) with the filters on the device: DataFrame (col 0 'cell', then genes) ->
    filtered DataFrame with genes sorted by mean expression, or None ("There is no high quality cells and genes")."""
    cell_name = tmp_df.iloc[:, 0].to_numpy()
    gene_name = np.asarray(tmp_df.columns[1:], dtype=object)
    body = tmp_df.iloc[:, 1:]
    if all(isinstance(t, pd.SparseDtype) for t in body.dtypes):
        X = sp.csc_matrix(body.sparse.to_coo(), dtype=np.float32)
    else:
        X = sp.csc_matrix(body.to_numpy(dtype=np.float32))
    X.eliminate_zeros()
    if verbose:
        print("Inp_spec")                                                                  # :168-169
        print(f"data size: {tmp_df.shape}, sparsity: {1 - X.nnz / (X.shape[0] * X.shape[1])}")
    res = qc_indices_device(X, gene_name, min_tp_c, min_tp_g, max_tp_c, max_tp_g, min_genes_per_cell, max_genes_per_cell,
                            min_cells_per_gene, mito_percent, ribo_percent, device=device, handle=handle)
    if res is None:
        if verbose:
            print("There is no high quality cells and genes")                              # :232
        return None
    fc_idx, gene_idx, out = res
    o_df = pd.DataFrame.sparse.from_spmatrix(out, columns=gene_name[gene_idx])
    o_df.insert(0, "cell", cell_name[fc_idx])
    if verbose:
        print(f"After filtering>> data size: {o_df.shape}, sparsity: {1 - out.nnz / (out.shape[0] * out.shape[1])}")   # :229
    return o_df


def get_denoised_df(inp_obj, device_="gpu", *, device=0, handle=None, dtype=np.float64):
    """Drop-in for scLENS.get_denoised_df (:889-931): the denoised count matrix rebuilt from the robust signals of a
    result dictionary of :func:`sclens` (keys ``gene_basis``, ``sig_id``, ``pca_n1``, ``rec_vals``, ``gene_id``,
    ``cell_id``).  One fused device kernel behind ``scl_op_denoise``; returns a DataFrame (cell, genes...) like the
    reference, Float64 by default (the reference's element type) or Float32."""
    if device_ != "gpu":
        raise ValueError('sclens_b200 implements device_="gpu" only (no CPU fallback exists)')
    sig_id = np.asarray(inp_obj["sig_id"], dtype=np.int64)
    if sig_id.size == 0:
        raise ValueError("no robust signal (sig_id is empty): nothing to reconstruct")
    gene_basis = np.asarray(inp_obj["gene_basis"], dtype=np.float32)
    g_mat = np.ascontiguousarray(gene_basis[sig_id, :].T)                      # r x M column-major == C order of M x r
    pca_n1 = inp_obj["pca_n1"]
    if pd is not None and isinstance(pca_n1, pd.DataFrame):
        pca_n1 = pca_n1.iloc[:, 1:].to_numpy()
    A = np.ascontiguousarray(np.asarray(pca_n1, dtype=np.float32).T)            # N x r column-major == C order of r x N
    r, N = A.shape
    M = g_mat.shape[0]
    if g_mat.shape[1] != r:
        raise ValueError("pca_n1 and gene_basis[sig_id, :] disagree on the number of robust signals")
    rec = inp_obj["rec_vals"]
    vec = {k: np.ascontiguousarray(np.asarray(rec[k], dtype=np.float64).ravel())
           for k in ("TGC", "mat2_mean", "mat2_std", "norm_tgc", "cent_")}
    if len(vec["TGC"]) != N or len(vec["norm_tgc"]) != N or any(len(vec[k]) != M for k in ("mat2_mean", "mat2_std", "cent_")):
        raise ValueError("rec_vals do not match the shapes of pca_n1 / gene_basis")
    dtype = np.dtype(dtype)
    if dtype not in (np.dtype(np.float64), np.dtype(np.float32)):
        raise ValueError("dtype must be float64 or float32")
    out = np.empty((M, N), dtype=dtype)                                         # N x M column-major
    own = handle is None
    h = Handle(device=device) if own else handle
    try:
        h._ck(h.lib.scl_op_denoise(h.h, N, M, r, ptr(A, C.c_float), ptr(g_mat, C.c_float), ptr(vec["TGC"], C.c_double),
                                   ptr(vec["mat2_mean"], C.c_double), ptr(vec["mat2_std"], C.c_double),
                                   ptr(vec["norm_tgc"], C.c_double), ptr(vec["cent_"], C.c_double),
                                   int(dtype == np.dtype(np.float32)), out.ctypes.data_as(C.c_void_p)))
    finally:
        if own:
            h.close()
    if pd is None:
        return out.T
    odf = pd.DataFrame(out.T, columns=[str(g) for g in inp_obj["gene_id"]])
    odf.insert(0, "cell", np.asarray(inp_obj["cell_id"]))
    return odf


def apply_umap(res, k=15, nc=2, md=0.1, metric="cosine", *, n_epochs=300, seed=0, init="spectral", device=0, handle=None,
               spread=1.0, learning_rate=1.0, repulsion_strength=1.0, neg_sample_rate=5, local_connectivity=1.0,
               spectral_maxiter=100):
    """Drop-in for scLENS.apply_umap! (:863-873): UMAP of the robust signals on the device.  Reads ``res["pca_n1"]``
    when it exists and has at least one column, otherwise ``res["pca"]`` (N x r, DataFrame with a leading "cell" column
    or array).  Stores ``res["umap"]`` (N x nc, rows in ``cell_id`` order) and ``res["umap_obj"]`` = {"graph": the
    symmetric fuzzy graph as scipy CSR, "knns", "dists": N x k (0-based), "a", "b", "info"} and returns ``res``.
    Exact kNN (no NN-descent) and a synchronous, deterministic epoch: the same seed gives the same embedding."""
    def signals(key):
        m = res.get(key)
        if pd is not None and isinstance(m, pd.DataFrame) and "cell" in m.columns:
            m = m.drop(columns="cell")
        return m if m is not None and np.ndim(m) == 2 and np.shape(m)[1] >= 1 else None

    src = signals("pca_n1")
    if src is None:
        src = signals("pca")
    if src is None:
        raise ValueError("the result has neither a non-empty 'pca_n1' nor a 'pca' entry")
    X = _umap_matrix(src)
    N = X.shape[1]
    _umap_params(N, k, nc, md, metric, n_epochs, seed, init, spread, learning_rate, repulsion_strength, neg_sample_rate,
                 local_connectivity, spectral_maxiter)    # every argument checked before a device is touched
    own = handle is None
    h = Handle(device=device) if own else handle
    try:
        emb, info = h.umap(X.T, k, nc, md, metric, n_epochs=n_epochs, seed=seed, init=init, spread=spread,
                           learning_rate=learning_rate, repulsion_strength=repulsion_strength,
                           neg_sample_rate=neg_sample_rate, local_connectivity=local_connectivity,
                           spectral_maxiter=spectral_maxiter)
        graph = h.umap_graph()
        knns, dists = h.umap_knn()
    finally:
        if own:
            h.close()
    res["umap"] = emb
    res["umap_obj"] = {"graph": graph, "knns": knns, "dists": dists, "a": info.a, "b": info.b,
                       "info": {"graph_nnz": info.graph_nnz, "spectral_iters": info.spectral_iters,
                                "init_fallback": info.init_fallback,
                                "timings_ms": {"knn": info.t_knn_ms, "graph": info.t_graph_ms, "init": info.t_init_ms,
                                               "layout": info.t_layout_ms}}}
    return res
