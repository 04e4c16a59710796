"""-m gpu tests of the two stages that carry the 1e-4 contract of the eigenvalues (DESIGN.md section 2), each on its own:

- the Float64 Rayleigh-Ritz refinement (refine.cu, through scl_debug_refine) against its numpy restatement
  (oracle/refine_ref.py) to one FP32 ulp, against a Kato-Temple bound on matrices with a designed spectrum, and on clusters;
- the Gram bias calibration (pipeline.cu, through scl_debug_gram_calibrated) against a restatement of its sample pairs and
  fit, bit for bit where it copies or scales, and against the exact Gram matrix;
- the tridiagonal stage's exit for spectra with more than 2048 clustered eigenvalues."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from sclens_b200 import Handle
from sclens_b200._lib import ptr

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import refine_ref as rr  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def h():
    with Handle() as hh:
        yield hh


# ---- refinement -------------------------------------------------------------------------------------------------------

def designed(n, lam, seed):
    """G64 = Q diag(lam) Q' (Q from the QR of a seeded Gaussian), its FP32 rounding G and the exact eigenvectors as rows."""
    Q = np.linalg.qr(np.random.default_rng(seed).standard_normal((n, n)))[0]
    G64 = (Q * lam) @ Q.T
    G64 = (G64 + G64.T) / 2
    return G64, np.ascontiguousarray(G64.astype(np.float32)), Q.T.copy()


def rotate_rows(V, idx, seed):
    R = np.linalg.qr(np.random.default_rng(seed).standard_normal((len(idx), len(idx))))[0]
    V = V.copy()
    V[idx] = R @ V[idx]
    return V


def dev_refine(h, G, V):
    n = G.shape[0]
    G = np.ascontiguousarray(G, np.float32)
    V = np.ascontiguousarray(V, np.float32)
    L, st = np.empty(n, np.float32), np.zeros(2, np.int32)
    h._ck(h.lib.scl_debug_refine(h.h, n, ptr(G, C.c_float), ptr(V, C.c_float), ptr(L, C.c_float), ptr(st, C.c_int32)))
    return L, [int(st[0]), int(st[1])]


def tri_solve(h, G, v0, v1):
    n = G.shape[0]
    L, V, out = np.empty(n, np.float32), np.empty((max(1, v1 - v0), n), np.float32), np.zeros(6)
    h._ck(h.lib.scl_op_syevd_tri(h.h, n, ptr(G, C.c_float), v0, v1, ptr(L, C.c_float), ptr(V, C.c_float), ptr(out, C.c_double)))
    return L, V[: v1 - v0], out


def assert_parity(L, st, G, V):
    """Device against the restatement: one FP32 ulp per value, the same clusters."""
    want, _, _, st_want = rr.refine(G.astype(np.float32), np.asarray(V, np.float32), return_parts=True)
    ulp = np.spacing(np.abs(want))
    assert np.all(np.abs(L.astype(np.float64) - want) <= ulp), np.max(np.abs(L.astype(np.float64) - want) / ulp)
    assert st == st_want, (st, st_want)


def spectrum_with_pair(n, seed):
    lam = np.sort(np.random.default_rng(seed).uniform(0.5, 3.0, n))
    if n >= 2:
        k = n // 2 - 1 if n > 2 else 0
        lam[k + 1] = lam[k] + 4e-5
        lam = np.sort(lam)
    return lam


@pytest.mark.parametrize("n", [2, 127, 128, 129, 130, 1001, 2531])
def test_refine_matches_restatement(h, n):
    """Shapes around the 128 x 128 tile (a partial tile, n % 4 != 0 takes the scalar loads), n = 2, and a production-like
    order.  Synthetic vectors: exact eigenvectors with 1e-4 noise and one close pair rotated into each other (a cluster);
    solver vectors: the own eigensolver's FP32 eigenvectors of a Wishart matrix."""
    lam = spectrum_with_pair(n, n)
    _, G, V = designed(n, lam, n + 1)
    V = V + 1e-4 / np.sqrt(n) * np.random.default_rng(n + 2).standard_normal(V.shape)   # |noise| ~ 1e-4 per vector
    k = int(np.argmin(np.diff(lam))) if n > 2 else 0
    t = np.deg2rad(43.0)
    V[[k, k + 1]] = np.array([[np.cos(t), np.sin(t)], [-np.sin(t), np.cos(t)]]) @ V[[k, k + 1]]
    V = V.astype(np.float32)
    L, st = dev_refine(h, G, V)
    assert_parity(L, st, G, V)
    assert st[0] >= 1
    if n >= 127:
        rng = np.random.default_rng(n + 3)
        A = rng.standard_normal((n, n + 300))
        W = np.ascontiguousarray((A @ A.T / A.shape[1]).astype(np.float32))
        _, Vs, out = tri_solve(h, W, 0, n)
        assert out[5] == 0
        L, st = dev_refine(h, W, Vs)
        assert_parity(L, st, W, Vs)


@pytest.mark.parametrize("n", [1001, 2531])
def test_refine_kato_temple_bound(h, n):
    """Every singleton's refined value lies within the Kato-Temple bound r^2 / delta of the designed eigenvalue (r: the
    Float64 residual of its vector, delta: the distance to the rest of the designed spectrum less |G - G64|_2), plus
    |G - G64|_2 (the FP32 matrix is not exactly the designed one), plus 2 FP32 ulps.  The bound is not fitted to the
    device: the solver's raw FP32 eigenvalues break it."""
    lam = np.concatenate([np.linspace(0.2, 2.4, n - 5), [3.0, 4.5, 6.0, 9.0, 14.0]])    # bulk + spikes, all gaps known
    G64, G, _ = designed(n, lam, 7 * n)
    E = G.astype(np.float64) - G64
    e2 = np.linalg.norm(E, 2)
    assert e2 < 1e-7 * lam[-1]
    Lraw, V, out = tri_solve(h, G, 0, n)
    assert out[5] == 0
    L, st = dev_refine(h, G, V)
    assert_parity(L, st, G, V)
    _, vals, cl, _ = rr.refine(G, V, return_parts=True)
    pos = np.argsort(np.argsort(vals, kind="stable"), kind="stable")   # sorted position of the value of vector i
    Gd = G.astype(np.float64)
    Vd = V.astype(np.float64)
    vv = np.einsum("ij,ij->i", Vd, Vd)
    GV = Vd @ Gd
    rho = np.einsum("ij,ij->i", GV, Vd) / vv
    r = np.linalg.norm(GV - rho[:, None] * Vd, axis=1) / np.sqrt(vv)
    singles = np.array([i for i, j in cl if i == j])
    assert len(singles) > 0.9 * n
    j = np.searchsorted(lam, rho[singles])
    j = np.clip(j, 1, n - 1)
    j = np.where(np.abs(lam[j - 1] - rho[singles]) < np.abs(lam[j] - rho[singles]), j - 1, j)   # nearest designed value
    others = np.abs(lam[None, :] - rho[singles][:, None])
    others[np.arange(len(singles)), j] = np.inf
    delta = others.min(axis=1) - e2
    assert np.all(delta > 0)
    bound = r[singles] ** 2 / delta + e2 + 2 * np.spacing(np.float32(lam[j])).astype(np.float64)
    got = L[pos[singles]].astype(np.float64)
    err = np.abs(got - lam[j])
    assert np.all(err <= bound), (np.max(err / bound), singles[np.argmax(err / bound)])
    raw_err = np.abs(Lraw[singles].astype(np.float64) - lam[j])
    assert np.any(raw_err > bound), "the raw solver values meet the bound: the test has no teeth"


def close_tol(e2, lam):
    return e2 + 2 * np.spacing(np.float32(np.max(np.abs(lam)))).astype(np.float64)


def test_refine_rotated_pair(h):
    """DESIGN's case: two eigenvalues 4e-5 apart whose vectors are rotated by 43 degrees into each other.  The Rayleigh
    quotients are off by sin^2(43) x 4e-5; the 2 x 2 Ritz values recover both."""
    n, k = 600, 300
    lam = np.linspace(0.5, 3.0, n)
    lam[k + 1] = lam[k] + 4e-5
    G64, G, V = designed(n, lam, 11)
    t = np.deg2rad(43.0)
    V[[k, k + 1]] = np.array([[np.cos(t), np.sin(t)], [-np.sin(t), np.cos(t)]]) @ V[[k, k + 1]]
    V = V.astype(np.float32)
    L, st = dev_refine(h, G, V)
    assert_parity(L, st, G, V)
    assert st == [1, 2]
    tol = close_tol(np.linalg.norm(G.astype(np.float64) - G64, 2), lam)
    assert np.all(np.abs(L.astype(np.float64) - lam) <= tol), np.max(np.abs(L - lam))
    assert abs(rr.band(G, V)[k, 0] - lam[k]) > 10 * tol       # what a singleton would have returned
    # the scale of a vector does not matter: rows times 2 and times 1/2 give the same bits
    s = np.where(np.arange(n) % 2 == 0, 2.0, 0.5).astype(np.float32)
    L2, st2 = dev_refine(h, G, V * s[:, None])
    np.testing.assert_array_equal(L2, L)
    assert st2 == st


@pytest.mark.parametrize("run,want", [(20, [1, 20]), (150, [2, 96])])
def test_refine_runs_of_near_equal_eigenvalues(h, run, want):
    """A run of near-equal eigenvalues (1e-6 apart) with an arbitrary orthonormal basis of their span: one chain longer than
    the band (20), or a run the 96-member cap splits in two (150).  Every refined value of the run stays within its spread,
    the others are the designed values, and each block keeps the trace of its Rayleigh quotients."""
    n, k = 700, 200
    lam = np.linspace(0.5, 3.0, n)
    lam[k: k + run] = lam[k] + 1e-6 * np.arange(run)
    lam = np.sort(lam)
    G64, G, V = designed(n, lam, 13 + run)
    V = rotate_rows(V, np.arange(k, k + run), 17).astype(np.float32)
    L, st = dev_refine(h, G, V)
    assert_parity(L, st, G, V)
    assert st == want
    tol = close_tol(np.linalg.norm(G.astype(np.float64) - G64, 2), lam)
    Ld = L.astype(np.float64)
    assert np.all(Ld[k: k + run] >= lam[k] - tol) and np.all(Ld[k: k + run] <= lam[k + run - 1] + tol)
    rest = np.setdiff1d(np.arange(n), np.arange(k, k + run))
    assert np.all(np.abs(Ld[rest] - lam[rest]) <= tol)
    assert abs(Ld[k: k + run].sum() - lam[k: k + run].sum()) <= run * tol


# ---- Gram bias calibration --------------------------------------------------------------------------------------------

def calib_pairs(S, rows):
    """calib_pair of pipeline.cu in numpy uint64 arithmetic."""
    with np.errstate(over="ignore"):
        x = (np.arange(S, dtype=np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        x ^= x >> np.uint64(29)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(32)
    i = ((x & np.uint64(0xFFFFFFFF)) % np.uint64(rows)).astype(np.int64)
    j = ((x >> np.uint64(32)) % np.uint64(rows - 1)).astype(np.int64)
    j = np.where(j >= i, j + 1, j)
    return i, j


def gram_operand(rows, K, seed, orthogonal=False):
    """Rows with a common positive component (off-diagonal sums of one sign, as in normalised expression data): the case
    whose truncation bias the calibration measures.  orthogonal: disjoint supports, every exact off-diagonal entry 0."""
    rng = np.random.default_rng(seed)
    if orthogonal:
        A = np.zeros((rows, K), np.float32)
        w = K // rows
        for r in range(rows):
            A[r, r * w:(r + 1) * w] = rng.standard_normal(w) + 1.0
    else:
        A = (rng.standard_normal((rows, K)) * 0.5 + np.abs(rng.standard_normal(K))[None, :]).astype(np.float32)
    hi = A.astype(np.float16)
    lo = (A - hi.astype(np.float32)).astype(np.float16)
    ld = (K + 7) // 8 * 8
    pad = lambda x: np.ascontiguousarray(np.pad(x, ((0, 0), (0, ld - K)))).view(np.uint16)   # noqa: E731
    return A, hi, lo, pad(hi), pad(lo), ld


def dev_gram_calibrated(h, rows, K, ld, hi_p, lo_p, scale, diag):
    G, f = np.empty((rows, rows), np.float32), np.zeros(1)
    h._ck(h.lib.scl_debug_gram_calibrated(h.h, rows, K, ld, ptr(hi_p, C.c_uint16), ptr(lo_p, C.c_uint16) if lo_p is not None else None,
                                          scale, ptr(diag, C.c_double), ptr(G, C.c_float), ptr(f, C.c_double)))
    return G, float(f[0])


def dev_gram(h, rows, K, ld, hi_p, lo_p, scale):
    G = np.empty((rows, rows), np.float32)
    h._ck(h.lib.scl_op_gram(h.h, rows, K, ld, ptr(hi_p, C.c_uint16), ptr(lo_p, C.c_uint16) if lo_p is not None else None,
                            scale, ptr(G, C.c_float)))
    return G


def exact_terms(hi, lo, split):
    """The products the tensor core forms, summed exactly enough (Float64 on the device): hi hi' (+ hi lo' + lo hi')."""
    import torch
    H = torch.from_numpy(hi.astype(np.float64)).cuda()
    X = H @ H.T
    if split:
        Lo = torch.from_numpy(lo.astype(np.float64)).cuda()
        X += H @ Lo.T + Lo @ H.T
    out = X.cpu().numpy()
    del H, X
    torch.cuda.empty_cache()
    return out


@pytest.mark.parametrize("K", [4000, 68000])
@pytest.mark.parametrize("split", [False, True])
def test_gram_calibration(h, K, split):
    """The factor against the restated samples and fit (1e-9), the diagonal and the off-diagonal bit for bit, and DESIGN's
    'one common factor' claim: after dividing by the factor, the least-squares slope of (G - exact) on exact over every
    off-diagonal pair is zero within the sampling noise of the 2048-sample fit.  K = 68 000 accumulates many promoted
    chunks."""
    rows = 320
    A, hi, lo, hi_p, lo_p, ld = gram_operand(rows, K, K + int(split))
    lo_p = lo_p if split else None
    scale = np.float32(1.0 / K)
    diag = np.einsum("ij,ij->i", A.astype(np.float64), A.astype(np.float64))
    G, f = dev_gram_calibrated(h, rows, K, ld, hi_p, lo_p, float(scale), diag)
    # restated samples and fit, on the device's own off-diagonal values
    S = 2048
    i, j = calib_pairs(S, rows)
    ex_all = exact_terms(hi, lo, split)
    e = ex_all[i, j]
    t = G[i, j].astype(np.float64) * (1.0 / np.float64(scale))
    sxx, sxy = np.sum(e * e), np.sum((t - e) * e)
    f_ref = 1.0 + sxy / sxx if sxx > 0 else 1.0
    if not (0.999 < f_ref < 1.001):
        f_ref = 1.0
    assert abs(f - f_ref) < 1e-9, (f, f_ref)
    assert abs(f - 1.0) > 1e-8, f              # there is a bias to calibrate
    # diagonal: float32(float32(diag * scale) * f), bit for bit
    d_want = (np.float32(diag * np.float64(scale)).astype(np.float64) * f).astype(np.float32)
    np.testing.assert_array_equal(np.diag(G), d_want)
    # off-diagonal: the syrk of scl_op_gram, bit for bit
    G0 = dev_gram(h, rows, K, ld, hi_p, lo_p, float(scale))
    off = ~np.eye(rows, dtype=bool)
    np.testing.assert_array_equal(G[off], G0[off])
    # one common factor: the slope over all pairs after dividing by f, against the standard error of the sample slope
    b = sxy / sxx
    u = (t - e) - b * e
    se = np.sqrt(np.sum(u * u * e * e)) / sxx
    iu = np.triu_indices(rows, 1)
    ea = ex_all[iu]
    ya = G[iu].astype(np.float64) / (f * np.float64(scale)) - ea
    slope = np.sum(ya * ea) / np.sum(ea * ea)
    assert abs(slope) < 5 * se, (slope, se, f - 1)
    assert abs(f - 1.0) > 20 * se                # and the factor itself is far outside that noise


@pytest.mark.parametrize("split", [False, True])
def test_gram_calibration_orthogonal_rows_give_one(h, split):
    """Rows with disjoint supports: every exact off-diagonal entry (and every sample) is 0, so the fit has nothing to measure
    and the guard returns exactly 1; the diagonal is then the exact one."""
    rows, K = 128, 4096
    A, hi, lo, hi_p, lo_p, ld = gram_operand(rows, K, 3, orthogonal=True)
    diag = np.einsum("ij,ij->i", A.astype(np.float64), A.astype(np.float64))
    scale = np.float32(1.0 / K)
    G, f = dev_gram_calibrated(h, rows, K, ld, hi_p, lo_p if split else None, float(scale), diag)
    assert f == 1.0
    np.testing.assert_array_equal(np.diag(G), np.float32(diag * np.float64(scale)))
    assert np.all(G[~np.eye(rows, dtype=bool)] == 0)


# ---- tridiagonal stage: spectra with more than 2048 clustered eigenvalues ----------------------------------------------

@pytest.mark.parametrize("n_equal", [2049, 2048])
def test_tridiagonal_cluster_limit(h, n_equal):
    """A diagonal matrix of order 2100 stays exactly tridiagonal (e = 0), so equal values reach the tridiagonal stage as one
    cluster.  More than 2048 clustered vectors: the stage declines and the solve falls back to cusolverDnSsyevd, counted;
    exactly 2048: the own cluster pass handles them.  The one-stage path is forced: no stage-1 panel of a diagonal matrix can
    be factored, so the two-stage path would fall back to it anyway after a tridiagonal stage of its own."""
    n = 2100
    rng = np.random.default_rng(n_equal)
    vals = np.concatenate([np.full(n_equal, 1.5), rng.uniform(0.2, 1.0, n - n_equal)])
    vals = vals[rng.permutation(n)].astype(np.float32)
    D = np.ascontiguousarray(np.diag(vals))
    st0, st = np.zeros(8), np.zeros(8)
    try:
        h._ck(h.lib.scl_debug_force_one_stage(1))
        h._ck(h.lib.scl_debug_last_solve(h.h, ptr(st0, C.c_double)))
        L, V, out = tri_solve(h, D, 0, n)
        h._ck(h.lib.scl_debug_last_solve(h.h, ptr(st, C.c_double)))
    finally:
        h.lib.scl_debug_force_one_stage(0)
    if n_equal > 2048:
        assert out[5] == 1 and st[7] == st0[7] + 1, (out, st0, st)
    else:
        assert out[5] == 0 and st[7] == st0[7] and out[3] == 1 and out[4] == 2048, (out, st0, st)
    np.testing.assert_allclose(L, np.sort(vals), rtol=1e-6, atol=1e-7)
    Vc = V.T.astype(np.float64)
    assert np.max(np.abs(D.astype(np.float64) @ Vc - Vc * L[None, :])) < 1e-5
    assert np.max(np.abs(Vc.T @ Vc - np.eye(n))) < 1e-5
