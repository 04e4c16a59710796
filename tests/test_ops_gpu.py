"""-m gpu parity tests of the function-level operators, called through the C ABI and checked
against the CPU oracle (oracle/sclens_oracle.py) on the same seeded inputs."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import sclens_oracle as orc
from sclens_b200 import Handle, _lib
from sclens_b200._lib import ptr
from sclens_b200.synth import make_counts

pytestmark = pytest.mark.gpu


def f16_split(a):
    hi = a.astype(np.float16)
    lo = (a - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def pad_rows(a, ld):
    out = np.zeros((a.shape[0], ld), dtype=a.dtype)
    out[:, :a.shape[1]] = a
    return out


@pytest.fixture(scope="module")
def h():
    with Handle() as hh:
        yield hh


@pytest.fixture(scope="module")
def h1():
    with Handle(cta_group=1) as hh:
        yield hh


def run_gemm(hh, A, B, split, colmajor=False, alpha=1.0):
    m, K = A.shape
    n = B.shape[0]
    ld = (K + 7) // 8 * 8
    a_hi, a_lo = f16_split(A)
    b_hi, b_lo = f16_split(B)
    a_hi, a_lo, b_hi, b_lo = [np.ascontiguousarray(pad_rows(x, ld)).view(np.uint16) for x in (a_hi, a_lo, b_hi, b_lo)]
    Cm = np.empty((n, m) if colmajor else (m, n), dtype=np.float32)
    rc = hh.lib.scl_op_gemm_tn(hh.h, m, n, K, ld, ld, ptr(a_hi, C.c_uint16), ptr(a_lo, C.c_uint16) if split else None,
                               ptr(b_hi, C.c_uint16), ptr(b_lo, C.c_uint16) if split else None, alpha, int(colmajor),
                               ptr(Cm, C.c_float))
    hh._ck(rc)
    return Cm.T if colmajor else Cm


@pytest.mark.parametrize("shape", [(128, 256, 64), (300, 200, 1000), (1000, 37, 4100), (257, 513, 72), (64, 16, 8)])
@pytest.mark.parametrize("cg", [2, 1])
def test_gemm_tn_fp16(h, h1, shape, cg):
    hh = h if cg == 2 else h1
    m, n, K = shape
    rng = np.random.default_rng(m * 7 + n)
    A = rng.standard_normal((m, K)).astype(np.float32)
    B = rng.standard_normal((n, K)).astype(np.float32)
    ref = A.astype(np.float16).astype(np.float64) @ B.astype(np.float16).astype(np.float64).T
    got = run_gemm(hh, A, B, split=False)
    scale = np.max(np.abs(ref))
    # exact binary16 products, FP32 tensor-core accumulation (truncating) in chunks of <= 2048 terms
    assert np.max(np.abs(got - ref)) / scale < 2e-5
    got_t = run_gemm(hh, A, B, split=False, colmajor=True, alpha=0.5)
    assert np.max(np.abs(got_t - 0.5 * ref)) / scale < 2e-5


@pytest.mark.parametrize("cg", [2, 1])
def test_gemm_tn_split_is_fp32_accurate(h, h1, cg):
    hh = h if cg == 2 else h1
    rng = np.random.default_rng(5)
    m, n, K = 384, 96, 3000
    A = rng.standard_normal((m, K)).astype(np.float32)
    B = rng.standard_normal((n, K)).astype(np.float32)
    ref = A.astype(np.float64) @ B.astype(np.float64).T
    got = run_gemm(hh, A, B, split=True)
    err = np.max(np.abs(got - ref)) / np.max(np.abs(ref))
    assert err < 1e-5, err


@pytest.mark.parametrize("rows,K", [(256, 512), (700, 1300), (1030, 333), (90, 4000)])
@pytest.mark.parametrize("cg", [2, 1])
@pytest.mark.parametrize("split", [False, True])
def test_gram_syrk(h, h1, rows, K, cg, split):
    hh = h if cg == 2 else h1
    rng = np.random.default_rng(rows + K)
    A = rng.standard_normal((rows, K)).astype(np.float32)
    ld = (K + 7) // 8 * 8
    hi, lo = f16_split(A)
    hi_p = np.ascontiguousarray(pad_rows(hi, ld)).view(np.uint16)
    lo_p = np.ascontiguousarray(pad_rows(lo, ld)).view(np.uint16)
    G = np.empty((rows, rows), dtype=np.float32)
    hh._ck(hh.lib.scl_op_gram(hh.h, rows, K, ld, ptr(hi_p, C.c_uint16), ptr(lo_p, C.c_uint16) if split else None,
                              1.0 / K, ptr(G, C.c_float)))
    src = A.astype(np.float64) if split else hi.astype(np.float64)
    ref = src @ src.T / K
    # bound: tensor-core truncation bias on a same-sign sum, <= 256 MMAs per accumulation chunk x ~8e-8 (DESIGN.md);
    # the pipeline replaces the diagonal (the only such sum) by exact Float64 sums of squares
    assert np.max(np.abs(G - ref)) / np.max(np.abs(ref)) < 3e-5
    assert np.array_equal(G, G.T)       # mirrored store: exactly symmetric


def normalize_dev(h, X, layout, with_lo=True):
    """scl_op_normalize: (hi, lo or None) as [lines][ld] uint16, and the statistics."""
    N, M = X.shape
    lines, length = (M, N) if layout == 0 else (N, M)
    ld = (length + 7) // 8 * 8
    hi = np.empty((lines, ld), dtype=np.uint16)
    lo = np.empty((lines, ld), dtype=np.uint16) if with_lo else None
    st = dict(tgc=np.empty(N), l2=np.empty(N), mean=np.empty(M), sd=np.empty(M), cent=np.empty(M))
    colptr, rowval, val = _lib.as_u32(X.indptr), _lib.as_u32(X.indices), _lib.as_f32(X.data)
    h._ck(h.lib.scl_op_normalize(h.h, N, M, X.nnz, ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32),
                                 ptr(val, C.c_float), layout, ld, ptr(hi, C.c_uint16), ptr(lo, C.c_uint16),
                                 ptr(st["tgc"], C.c_double), ptr(st["mean"], C.c_double), ptr(st["sd"], C.c_double),
                                 ptr(st["l2"], C.c_double), ptr(st["cent"], C.c_double)))
    return hi, lo, st, length


def assert_normalize_oracle(ref, rec, layout, hi, lo, st, length):
    np.testing.assert_array_equal(st["tgc"], rec["TGC"])
    np.testing.assert_allclose(st["mean"], rec["mat2_mean"].ravel(), rtol=1e-12)
    np.testing.assert_allclose(st["sd"], rec["mat2_std"].ravel(), rtol=1e-11)
    np.testing.assert_allclose(st["l2"], rec["norm_tgc"], rtol=1e-11)
    np.testing.assert_allclose(st["cent"], rec["cent_"].ravel(), rtol=1e-9, atol=1e-15)
    want = ref.T if layout == 0 else ref
    got_hi = hi.view(np.float16)[:, :length].astype(np.float64)
    # hi alone is the correctly rounded binary16 value (up to float32 background arithmetic)
    assert np.max(np.abs(got_hi - want) / (np.abs(want) + 1e-3)) < 6e-4
    assert not hi.view(np.float16)[:, length:].any()
    if lo is not None:
        got = got_hi + lo.view(np.float16)[:, :length].astype(np.float64)
        # hi + lo reproduces the Float32 rounding of the Float64 reference value
        assert np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want))) < 4e-7


# (2301, 4700) spans several writer strips and has gene lines above the CTA-per-line threshold of the statistics
# passes; (260, 20000) has cell lines above it
NORM_SHAPES = [(500, 800), (900, 400), (2301, 4700), (260, 20000)]


@pytest.mark.parametrize("N,M", NORM_SHAPES)
@pytest.mark.parametrize("layout", [0, 1])
def test_normalize_matches_oracle(h, N, M, layout):
    X = make_counts(N, M, seed=11, K=4, de_prob=0.3, lfc_sd=1.5)
    ref, rec = orc.normalize_main(X)
    hi, lo, st, length = normalize_dev(h, X, layout)
    assert_normalize_oracle(ref, rec, layout, hi, lo, st, length)


@pytest.fixture
def norm_tuning(h):
    """Restores the default launch choices of the normalisation kernels (statistics variant 4, whole-CTA lines above
    4096 entries, automatic writer) after the test."""
    yield lambda variant, heavy, writer: h._ck(h.lib.scl_debug_set_tuning(variant, heavy, writer))
    h._ck(h.lib.scl_debug_set_tuning(4, 4096, -1))


@pytest.mark.parametrize("N,M", NORM_SHAPES)
@pytest.mark.parametrize("layout", [0, 1])
def test_normalize_every_writer_and_statistics_variant(h, norm_tuning, N, M, layout):
    """The hi-only output (the single-pass Gram operand: writer -1 picks the staged TMA-store writer 2 without lo) meets the
    oracle; every dense writer gives the hi bytes of the hi+lo call, with or without lo, and a zero pad; every launch
    variant of the statistics passes, and whole-CTA lines from 64 entries on, meet the oracle."""
    X = make_counts(N, M, seed=11, K=4, de_prob=0.3, lfc_sd=1.5)
    ref, rec = orc.normalize_main(X)
    norm_tuning(4, 4096, -1)
    hi0, lo0, st, length = normalize_dev(h, X, layout)
    hi, _, st1, _ = normalize_dev(h, X, layout, with_lo=False)
    assert_normalize_oracle(ref, rec, layout, hi, None, st1, length)
    for writer in (-1, 0, 1, 2, 3):
        norm_tuning(-1, 0, writer)
        hi, _, _, _ = normalize_dev(h, X, layout, with_lo=False)
        np.testing.assert_array_equal(hi, hi0, err_msg=f"writer {writer}, hi only")
        hi, lo, _, _ = normalize_dev(h, X, layout)
        np.testing.assert_array_equal(hi, hi0, err_msg=f"writer {writer}, hi + lo")
        np.testing.assert_array_equal(lo, lo0, err_msg=f"writer {writer}, lo")
    norm_tuning(-1, 0, -1)
    for variant, heavy in [(v, 4096) for v in range(9)] + [(4, 64), (8, 64)]:
        norm_tuning(variant, heavy, -2)
        hi, lo, st1, _ = normalize_dev(h, X, layout)
        assert_normalize_oracle(ref, rec, layout, hi, lo, st1, length)
        if variant < 8 and heavy == 4096:   # the line passes differ in launch shape only: the same Float64 sums
            for k in st:
                np.testing.assert_array_equal(st1[k], st[k], err_msg=f"statistics variant {variant}: {k}")


def csc_arrays(X):
    return _lib.as_u32(X.indptr), _lib.as_u32(X.indices), _lib.as_f32(X.data)


@pytest.mark.parametrize("N,M", [(300, 500), (9000, 60), (70, 9000)])
@pytest.mark.parametrize("binarise", [0, 1])
def test_perturb_merge_bit_exact(h, N, M, binarise):
    X = make_counts(N, M, seed=3, K=3)
    rng = np.random.default_rng(4)
    z1, z2 = orc.draw_zero_candidates(X, rng)
    sple = rng.choice(len(z1), size=len(z1) // 3, replace=False)
    want = orc.perturbed_matrix(X, z1, z2, sple, bool(binarise))
    colptr, rowval, val = csc_arrays(X)
    ar, ac = _lib.as_u32(z1[sple]), _lib.as_u32(z2[sple])
    nnz_out = X.nnz + len(sple)
    oc, orow, ov = np.empty(M + 1, np.uint32), np.empty(nnz_out, np.uint32), np.empty(nnz_out, np.float32)
    h._ck(h.lib.scl_op_perturb_merge(h.h, N, M, X.nnz, ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32),
                                     ptr(val, C.c_float), len(sple), ptr(ar, C.c_uint32), ptr(ac, C.c_uint32),
                                     binarise, ptr(oc, C.c_uint32), ptr(orow, C.c_uint32), ptr(ov, C.c_float)))
    np.testing.assert_array_equal(oc, want.indptr)
    np.testing.assert_array_equal(orow, want.indices)
    np.testing.assert_array_equal(ov, want.data)


def test_perturb_merge_general_semantics(h):
    """sparse(I,J,V) semantics for additions that hit stored entries or each other (cannot happen for draws from
    the zero candidates, but the operator must still sum them like Julia's sparse(), src/scLENS.jl:735/:774),
    and the degenerate cases: no additions at all, additions only in empty lines."""
    N, M = 400, 300
    X = make_counts(N, M, seed=9, K=3)
    colptr, rowval, val = csc_arrays(X)
    coo = X.tocoo()
    rng = np.random.default_rng(10)
    hit = rng.choice(X.nnz, size=50, replace=False)
    zr, zc = orc.draw_zero_candidates(X, rng)
    ar = np.concatenate([coo.row[hit], zr[:200], zr[:20]])          # 50 on stored entries, 20 duplicated zeros
    ac = np.concatenate([coo.col[hit], zc[:200], zc[:20]])
    for binarise, (rows_, cols_) in [(0, (ar, ac)), (1, (ar, ac)), (0, (ar[:0], ac[:0]))]:
        base = X.copy()
        if binarise:
            base.data[:] = 1.0
        want = sp.csc_matrix(base + sp.coo_matrix((np.ones(len(rows_), np.float32), (rows_, cols_)), shape=(N, M)))
        want.sort_indices()
        n_out = X.nnz + len(rows_)
        oc, orow, ov = np.empty(M + 1, np.uint32), np.zeros(n_out, np.uint32), np.zeros(n_out, np.float32)
        a1, a2 = _lib.as_u32(rows_), _lib.as_u32(cols_)
        h._ck(h.lib.scl_op_perturb_merge(h.h, N, M, X.nnz, ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32),
                                         ptr(val, C.c_float), len(rows_), ptr(a1, C.c_uint32) if len(rows_) else None,
                                         ptr(a2, C.c_uint32) if len(rows_) else None, binarise, ptr(oc, C.c_uint32),
                                         ptr(orow, C.c_uint32), ptr(ov, C.c_float)))
        np.testing.assert_array_equal(oc, want.indptr)
        np.testing.assert_array_equal(orow[:want.nnz], want.indices)
        np.testing.assert_array_equal(ov[:want.nnz], want.data)


@pytest.mark.parametrize("N,M", [(300, 500), (9000, 60)])
@pytest.mark.parametrize("aligned", [True, False])
def test_permute_null_bit_exact(h, N, M, aligned):
    X = make_counts(N, M, seed=5, K=3)
    rng = np.random.default_rng(6)
    order = None if aligned else rng.permutation(M)   # emulates Julia's Dict order (duplicates summed)
    perm, rows = orc.draw_null(X, rng, order)
    if not aligned:
        rows[-1] = N - 1                              # keep the reference's implied shape == (N, M)
    want = orc.build_null(X, perm, rows)
    colptr, rowval, val = csc_arrays(X)
    nnz = C.c_int64()
    oc, orow, ov = np.empty(M + 1, np.uint32), np.empty(X.nnz, np.uint32), np.empty(X.nnz, np.float32)
    h._ck(h.lib.scl_op_permute_null(h.h, N, M, X.nnz, ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32),
                                    ptr(val, C.c_float), ptr(perm, C.c_uint32), ptr(rows, C.c_uint32), C.byref(nnz),
                                    ptr(oc, C.c_uint32), ptr(orow, C.c_uint32), ptr(ov, C.c_float)))
    assert nnz.value == want.nnz
    if not aligned:
        assert want.nnz < X.nnz                       # duplicates really were merged
    np.testing.assert_array_equal(oc[:want.shape[1] + 1], want.indptr)
    np.testing.assert_array_equal(orow[:want.nnz], want.indices)
    np.testing.assert_array_equal(ov[:want.nnz], want.data)


def test_device_null_draw_properties(h):
    """Device-drawn null matrix: same per-gene counts, same value multiset, rows distinct."""
    N, M = 2000, 300
    X = make_counts(N, M, seed=8, K=3)
    colptr, rowval, val = csc_arrays(X)
    nnz = C.c_int64()
    oc, orow, ov = np.empty(M + 1, np.uint32), np.empty(X.nnz, np.uint32), np.empty(X.nnz, np.float32)
    h._ck(h.lib.scl_op_permute_null(h.h, N, M, X.nnz, ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32),
                                    ptr(val, C.c_float), None, None, C.byref(nnz), ptr(oc, C.c_uint32),
                                    ptr(orow, C.c_uint32), ptr(ov, C.c_float)))
    assert nnz.value == X.nnz
    np.testing.assert_array_equal(oc, X.indptr)
    np.testing.assert_array_equal(np.sort(ov), np.sort(X.data))
    for j in range(M):
        seg = orow[oc[j]:oc[j + 1]]
        assert np.all(np.diff(seg.astype(np.int64)) > 0) and (len(seg) == 0 or seg[-1] < N)
    assert not np.array_equal(orow, X.indices)


def test_syevd_and_mp_fit(h):
    rng = np.random.default_rng(2)
    n = 600
    A = rng.standard_normal((n, 900)).astype(np.float32)
    G = (A @ A.T / 900).astype(np.float32)
    L, V, ms = np.empty(n, np.float32), np.empty((n, n), np.float32), C.c_double()
    h._ck(h.lib.scl_op_syevd(h.h, n, ptr(G, C.c_float), ptr(L, C.c_float), ptr(V, C.c_float), C.byref(ms)))
    Lref = np.linalg.eigvalsh(G.astype(np.float64))
    np.testing.assert_allclose(L, Lref, rtol=2e-5, atol=2e-6)
    Vc = V.T  # column-major eigenvectors
    assert np.max(np.abs(G.astype(np.float64) @ Vc - Vc * L[None, :])) < 5e-5
    # mp fit against the oracle
    B = rng.standard_normal((n, 900)).astype(np.float32)
    Lr = np.linalg.eigvalsh((B @ B.T / 900).astype(np.float64)).astype(np.float32)
    Lsig = L.copy()
    Lsig[-3:] *= 1.6
    out = np.empty(8)
    assert h.lib.scl_op_mp_fit(ptr(Lsig, C.c_float), n, ptr(Lr[:-1].copy(), C.c_float), n - 1, ptr(out, C.c_double)) == 0
    L_mp, b_plus, b_min, it = orc.mp_calculation(Lsig.astype(np.float64), Lr[:-1].astype(np.float64))
    lam = orc.tw(Lsig.astype(np.float64), L_mp)[0]
    assert abs(out[0] - lam) < 1e-12 * lam and abs(out[1] - b_plus) < 1e-12 and abs(out[2] - b_min) < 1e-12
    assert int(out[4]) == len(L_mp) and int(out[5]) == it and int(out[7]) == int((Lsig > lam).sum())
    chk = orc.mp_check(L_mp)
    assert abs(out[3] - chk["ks_static"]) < 1e-9 and bool(out[6]) == chk["pass"]


def _tri_solve(h, G, v0, v1):
    n = G.shape[0]
    L, V, out = np.empty(n, np.float32), np.empty((max(1, v1 - v0), n), np.float32), np.zeros(6)
    h._ck(h.lib.scl_op_syevd_tri(h.h, n, ptr(G, C.c_float), v0, v1, ptr(L, C.c_float), ptr(V, C.c_float), ptr(out, C.c_double)))
    return L, V[: v1 - v0].T, out


@pytest.mark.parametrize("case", ["wishart", "centred", "wide_range_of_scales"])
def test_syevd_tri_matches_float64(h, case):
    """Own tridiagonal stage (Ssytrd -> Float64 multisection + twisted factorisation -> Sormtr) against numpy's Float64
    eigh of the same FP32 matrix: same tolerances as the library solve above, all vectors / an index range / values only."""
    rng = np.random.default_rng(5)
    n = 640
    A = rng.standard_normal((n, 900))
    if case == "centred":
        A -= A.mean(axis=0)                       # one exactly-null direction (column-centred N <= M matrix)
    if case == "wide_range_of_scales":
        A *= np.exp(rng.normal(0, 2.0, size=(n, 1)))   # graded rows: eigenvalues over ~6 decades
    G = (A @ A.T / 900).astype(np.float32)
    Lref, Vref = np.linalg.eigh(G.astype(np.float64))
    scale = float(Lref[-1])
    L, V, out = _tri_solve(h, G, 0, n)
    assert out[5] == 0, "fell back to the library solver"
    np.testing.assert_allclose(L, Lref, rtol=2e-5, atol=2e-6 * scale)
    G64 = G.astype(np.float64)
    assert np.max(np.abs(G64 @ V - V * L[None, :])) < 5e-5 * max(1.0, scale)
    assert np.max(np.abs(V.T.astype(np.float64) @ V - np.eye(n))) < 5e-5
    # index range (what a sparsity-search step asks for) and values only give the same numbers
    v0, v1 = 3, n // 2 + 40
    L2, V2, _ = _tri_solve(h, G, v0, v1)
    np.testing.assert_array_equal(L2, L)
    assert np.max(np.abs(np.abs(np.sum(V2 * V[:, v0:v1], axis=0)) - 1.0)) < 1e-5
    L3, _, _ = _tri_solve(h, G, 0, 0)
    np.testing.assert_array_equal(L3, L)


@pytest.mark.parametrize("n", [300, 1000, 2531])
def test_own_tridiagonalisation_matches_float64(h, n):
    """The one-stage path, forced at every order (scl_debug_force_one_stage): sytrd.cu (persistent cooperative Householder
    tridiagonalisation, lower triangle only), the own tridiagonal stage and Sormtr - eigenvalues, residuals, orthogonality -
    against numpy's Float64 eigh, same tolerances as the library path; shapes that are not multiples of the 32-column panel or
    the 128 x 128 update tile."""
    rng = np.random.default_rng(n)
    A = rng.standard_normal((n, n + 300))
    A -= A.mean(axis=0)
    G = (A @ A.T / A.shape[1]).astype(np.float32)
    Lref = np.linalg.eigvalsh(G.astype(np.float64))
    st = np.zeros(8)
    try:
        h._ck(h.lib.scl_debug_force_one_stage(1))
        L, V, out = _tri_solve(h, G, 0, n)
        h._ck(h.lib.scl_debug_last_solve(h.h, ptr(st, C.c_double)))
    finally:
        h.lib.scl_debug_force_one_stage(0)
    assert out[5] == 0, "fell back to the library solver"
    assert st[5] == 0, ("the two-stage path produced the result", st)
    np.testing.assert_allclose(L, Lref, rtol=2e-5, atol=3e-6 * float(Lref[-1]))
    G64 = G.astype(np.float64)
    assert np.max(np.abs(G64 @ V - V * L[None, :])) < 5e-5 * max(1.0, float(Lref[-1]))
    assert np.max(np.abs(V.T.astype(np.float64) @ V - np.eye(n))) < 5e-5


def test_syevd_tri_exact_multiplicities(h):
    """Every eigenvalue exactly double (two identical diagonal blocks) plus a block of exact zeros: twisted factorisation alone
    would return parallel vectors; the cluster pass (inverse iteration + Gram-Schmidt inside the cluster) must give an
    orthonormal basis of every eigenspace."""
    rng = np.random.default_rng(6)
    nb = 150
    A = rng.standard_normal((nb, 300))
    B = (A @ A.T / 300).astype(np.float32)
    n = 2 * nb + 20
    G = np.zeros((n, n), np.float32)
    G[:nb, :nb] = B
    G[nb:2 * nb, nb:2 * nb] = B
    perm = rng.permutation(n)
    G = np.ascontiguousarray(G[np.ix_(perm, perm)])
    L, V, out = _tri_solve(h, G, 0, n)
    assert out[5] == 0, out
    Lref = np.linalg.eigvalsh(G.astype(np.float64))
    np.testing.assert_allclose(L, Lref, rtol=2e-5, atol=5e-6)
    assert np.max(np.abs(G.astype(np.float64) @ V - V * L[None, :])) < 5e-5
    assert np.max(np.abs(V.T.astype(np.float64) @ V - np.eye(n))) < 5e-5
    # a diagonal matrix stays exactly tridiagonal (e = 0) with exactly repeated eigenvalues: this is the case that reaches
    # the cluster pass (the FP32 tridiagonalisation above splits the pairs by ~1e-7, far above the 1e-9 |T| cluster gap)
    vals = np.repeat(rng.uniform(0.5, 3.0, size=60), 3).astype(np.float32)
    vals = np.concatenate([vals, np.zeros(7, np.float32)])
    vals = vals[rng.permutation(len(vals))]
    D = np.diag(vals).astype(np.float32)
    L, V, out = _tri_solve(h, D, 0, len(vals))
    assert out[5] == 0 and out[3] == 61 and out[4] == len(vals), out
    np.testing.assert_allclose(L, np.sort(vals), rtol=1e-6, atol=1e-7)
    assert np.max(np.abs(D.astype(np.float64) @ V - V * L[None, :])) < 1e-5
    assert np.max(np.abs(V.T.astype(np.float64) @ V - np.eye(len(vals)))) < 1e-5


@pytest.mark.parametrize("shape", [(301, 420), (400, 250)])
def test_normalize_median_centering_matches_oracle(shape):
    """centering="median" (:653-654): the dense operand against the oracle's Float32 restatement, with genes expressed in
    most cells (non-zero medians, both parities of N) and the usual sparse genes (median = an implicit zero)."""
    N, M = shape
    X = make_counts(N, M, seed=5, K=3, de_prob=0.3, lfc_sd=1.5).tolil()
    rng = np.random.default_rng(0)
    for j in range(8):
        col = rng.poisson(4.0 if j < 6 else 0.7, size=(N, 1)).astype(np.float32)   # j >= 6: close to half the cells
        X[:, j] = col
    X = sp.csc_matrix(X, dtype=np.float32)
    X.eliminate_zeros()
    X.sort_indices()
    want = orc.logn_scale_pre_scale_median(X).astype(np.float64)
    with Handle(centering="median") as hh:
        for layout in (0, 1):
            lines, length = (M, N) if layout == 0 else (N, M)
            ld = (length + 7) // 8 * 8
            hi = np.empty((lines, ld), np.uint16)
            lo = np.empty((lines, ld), np.uint16)
            colptr, rowval, val = _lib.as_u32(X.indptr), _lib.as_u32(X.indices), _lib.as_f32(X.data)
            hh._ck(hh.lib.scl_op_normalize(hh.h, N, M, X.nnz, ptr(colptr, C.c_uint32), ptr(rowval, C.c_uint32),
                                           ptr(val, C.c_float), layout, ld, ptr(hi, C.c_uint16), ptr(lo, C.c_uint16),
                                           None, None, None, None, None))
            got = hi.view(np.float16).astype(np.float64) + lo.view(np.float16).astype(np.float64)
            got = got[:, :length].T if layout == 0 else got[:, :length]
            np.testing.assert_allclose(got, want, rtol=3e-4, atol=3e-5)       # the oracle itself is Float32 here


class _QueuedDraws:
    """Stands in for numpy's Generator inside the oracle: hands out arrays that were drawn elsewhere, in call order."""

    def __init__(self, *arrays):
        self.q = list(arrays)

    def integers(self, lo, hi, size=None, dtype=np.int64):
        a = self.q.pop(0)
        assert len(a) == size and a.min() >= lo and a.max() < hi
        return a.astype(dtype)


@pytest.mark.parametrize("shape,seed", [((300, 500), 11), ((700, 260), 12), ((64, 40), 13)])
def test_device_zero_candidates_follow_the_reference_recipe(shape, seed):
    """Production draw of z_idx1 / z_idx2 (:668-673) on the device: fed the same uniform draws (restated on the host from the
    library's counter-based generator), the oracle's setdiff / first-occurrence step must give the same two vectors, bit for bit."""
    N, M = shape
    X = make_counts(N, M, seed=seed, K=3, de_prob=0.3, lfc_sd=1.5) if N >= 200 else \
        sp.random(N, M, density=0.3, random_state=seed, format="csc", dtype=np.float32)
    X = sp.csc_matrix(X, dtype=np.float32)
    X.data[:] = np.maximum(1.0, np.round(X.data * 5))
    X.sort_indices()
    with Handle(seed=seed) as hh:
        hh.set_counts(X)
        n = C.c_int64()
        hh._ck(hh.lib.scl_op_draw_zero_candidates(hh.h, 1000 + seed, C.byref(n), None, None))
        z1, z2 = np.empty(max(1, X.nnz), np.uint32), np.empty(max(1, X.nnz), np.uint32)
        n2 = C.c_int64()
        hh._ck(hh.lib.scl_op_draw_zero_candidates(hh.h, 1000 + seed, C.byref(n2), ptr(z1, C.c_uint32), ptr(z2, C.c_uint32)))
        assert n2.value == n.value                    # deterministic for a given seed
        z1, z2 = z1[: n.value], z2[: n.value]
        rows, cols = np.empty(X.nnz, np.uint32), np.empty(X.nnz, np.uint32)
        assert hh.lib.scl_op_zero_candidate_draws(1000 + seed, X.nnz, N, M, ptr(rows, C.c_uint32), ptr(cols, C.c_uint32)) == 0
        want1, want2 = orc.draw_zero_candidates(X, _QueuedDraws(rows, cols))
        np.testing.assert_array_equal(z1, np.asarray(want1, np.uint32))
        np.testing.assert_array_equal(z2, np.asarray(want2, np.uint32))
        # properties that do not depend on the generator: inside the grid, distinct, disjoint from the stored entries,
        # and as many as nnz uniform draws leave: NM(1 - exp(-nnz/NM)) distinct positions, a fraction (1 - density) of them zeros
        key = z2.astype(np.int64) * N + z1
        assert z1.max() < N and z2.max() < M and len(np.unique(key)) == len(key)
        nzr, nzc = X.nonzero()
        assert not np.isin(key, nzc.astype(np.int64) * N + nzr).any()
        grid = N * M
        expect = grid * (1 - np.exp(-X.nnz / grid)) * (1 - X.nnz / grid)
        assert abs(n.value - expect) < 6 * np.sqrt(expect) + 3
        # the draws themselves are uniform on the grid: chi-square of the row and column marginals (large shapes only)
        if N >= 200:
            for v, k in ((rows, N), (cols, M)):
                cnt = np.bincount(v, minlength=k)
                chi2 = ((cnt - len(v) / k) ** 2 / (len(v) / k)).sum()
                assert abs(chi2 - (k - 1)) < 6 * np.sqrt(2 * (k - 1)), (chi2, k)
        # sample(1:n_cand, n_take, replace=false) (:731, :772): distinct members of the pool; n_take = n_cand is a permutation
        for n_take in (n.value // 3, n.value):
            r, c = np.empty(max(1, n_take), np.uint32), np.empty(max(1, n_take), np.uint32)
            hh._ck(hh.lib.scl_op_draw_subset(hh.h, n_take, 77, ptr(r, C.c_uint32), ptr(c, C.c_uint32)))
            k2 = c[:n_take].astype(np.int64) * N + r[:n_take]
            assert len(np.unique(k2)) == n_take and np.isin(k2, key).all()
        r2, c2 = np.empty(n.value, np.uint32), np.empty(n.value, np.uint32)
        hh._ck(hh.lib.scl_op_draw_subset(hh.h, n.value // 3, 78, ptr(r2, C.c_uint32), ptr(c2, C.c_uint32)))
        assert not np.array_equal(r2[: n.value // 3], r[: n.value // 3])     # another seed, another sample


def test_device_noise_baseline_matches_the_oracle_expectation(h):
    """p_th (:709-712) from the device generator against the oracle's draw_noise_baseline: both estimate
    E max_{nm} |N(0, 1/nm)| from 5000 replicates, so they agree within a few standard errors of that mean."""
    for nm in (450, 2000):
        ref = np.array([np.max(np.abs(np.random.default_rng(s).normal(0, np.sqrt(1 / nm), size=nm))) for s in range(4000)])
        se = ref.std(ddof=1) / np.sqrt(5000)
        want = orc.draw_noise_baseline(nm, np.random.default_rng(5), n_rep=5000)
        got = []
        for seed in (1, 2, 3):
            p = C.c_double()
            h._ck(h.lib.scl_op_noise_baseline(h.h, nm, 5000, seed, C.byref(p)))
            got.append(p.value)
            assert abs(p.value - ref.mean()) < 5 * se * np.sqrt(1 + 5000 / 4000), (nm, p.value, ref.mean(), se)
            assert abs(p.value - want) < 7 * se
        assert len(set(got)) == 3          # seeds matter


def test_corr_colabsmax(h):
    rng = np.random.default_rng(9)
    n, nv, nw = 700, 650, 331
    V = np.linalg.qr(rng.standard_normal((n, nv)))[0].T.astype(np.float32).copy()
    W = np.linalg.qr(rng.standard_normal((n, nw)))[0].T.astype(np.float32).copy()
    d = np.empty(nw, np.float32)
    h._ck(h.lib.scl_op_corr_colabsmax(h.h, n, nv, nw, ptr(V, C.c_float), ptr(W, C.c_float), ptr(d, C.c_float)))
    ref = np.max(np.abs(V.astype(np.float64) @ W.astype(np.float64).T), axis=0)
    np.testing.assert_allclose(d, ref, rtol=0, atol=3e-6)


def test_topk_subspace(h):
    rng = np.random.default_rng(12)
    n, K = 1500, 2500
    A = rng.standard_normal((n, K))
    U = np.linalg.qr(rng.standard_normal((n, 6)))[0]
    A += U @ (np.array([9, 6, 4, 3, 2.2, 1.9])[:, None] * rng.standard_normal((6, K)))
    G = (A @ A.T / K).astype(np.float32)
    k = 9
    L, V, it = np.empty(k, np.float32), np.empty((k, n), np.float32), C.c_int32()
    h._ck(h.lib.scl_op_topk_subspace(h.h, n, ptr(G, C.c_float), k, ptr(L, C.c_float), ptr(V, C.c_float), C.byref(it)))
    Lr, Vr = np.linalg.eigh(G.astype(np.float64))
    Lr, Vr = Lr[::-1][:k], Vr[:, ::-1][:, :k]
    np.testing.assert_allclose(L, Lr, rtol=2e-5)
    cosines = np.abs(np.sum(V.T.astype(np.float64) * Vr, axis=0))
    gaps = np.minimum(np.abs(np.diff(np.concatenate([[np.inf], Lr]))), np.abs(np.diff(np.concatenate([Lr, [np.linalg.eigvalsh(G.astype(np.float64))[-k - 1]]]))))
    ang = np.arccos(np.clip(cosines, 0, 1))
    assert np.all(ang < 2e-4 * Lr / gaps + 1e-3), (ang, gaps)


def test_scores_match_oracle(h):
    rng = np.random.default_rng(13)
    N, k, min_pc, P = 900, 4, 6, 7
    nV = np.linalg.qr(rng.standard_normal((N, k)))[0]
    sets = []
    for r in range(P):
        noise = np.concatenate([np.full(k // 2, 0.15), np.full(k - k // 2, 1.2)])
        base = np.concatenate([nV + noise[None, :] * rng.standard_normal((N, k)) / np.sqrt(N) * 3,
                               rng.standard_normal((N, min_pc - k))], axis=1)
        Q = np.linalg.qr(base)[0][:, rng.permutation(min_pc)]
        sets.append(Q)
    rob, sig = orc.robustness_scores(nV, sets, 60)
    nV32 = np.ascontiguousarray(nV.T, dtype=np.float32)
    sets32 = np.ascontiguousarray(np.stack([s.T for s in sets]), dtype=np.float32)
    npairs = P * (P - 1) // 2
    b = np.empty((npairs, k), np.float32)
    m, sd = np.empty(k), np.empty(k)
    sid, nrob = np.empty(k, np.int32), C.c_int32()
    h._ck(h.lib.scl_op_scores(h.h, N, k, min_pc, P, ptr(nV32, C.c_float), ptr(sets32, C.c_float), 60.0,
                              ptr(b, C.c_float), ptr(m, C.c_double), ptr(sd, C.c_double), ptr(sid, C.c_int32),
                              C.byref(nrob)))
    np.testing.assert_allclose(b.T, rob["b_"], atol=5e-6)
    np.testing.assert_allclose(m, rob["m_scores"], atol=5e-6)
    np.testing.assert_allclose(sd, rob["sd_scores"], atol=5e-6)
    np.testing.assert_array_equal(sid[:nrob.value], sig)


@pytest.mark.parametrize("n,case", [(300, "wishart"), (1000, "centred"), (1203, "centred"), (2531, "wishart"),
                                    (1536, "wide_range_of_scales")])
def test_two_stage_solver_matches_float64(h, n, case):
    """Two-stage reduction (sy2sb.cu dense -> band, sb2st.cu band -> tridiagonal by bulge chasing, backtrans.cu), the path of
    every order >= 256: eigenvalues, residuals and orthogonality against numpy's Float64 eigh of the same FP32 matrix, with the
    tolerances of the one-stage path; orders that are not multiples of the 64-column panel, the 128 x 128 update tile or 4
    (padded copy); all vectors / an index range / values only agree.  Stage 1 multiplies in split binary16 when
    n / 8192 <= |G|_F <= 1024 and in three-term TF32 otherwise: the graded rows of "wide_range_of_scales" take TF32, the
    other cases split binary16."""
    rng = np.random.default_rng(n)
    A = rng.standard_normal((n, n + 300))
    if case == "centred":
        A -= A.mean(axis=0)
    if case == "wide_range_of_scales":
        A *= np.exp(rng.normal(0, 1.5, size=(n, 1)))
    G = (A @ A.T / A.shape[1]).astype(np.float32)
    fro = np.linalg.norm(G.astype(np.float64))
    assert (n / 8192 <= fro <= 1024) == (case != "wide_range_of_scales"), fro
    Lref = np.linalg.eigvalsh(G.astype(np.float64))
    scale = float(Lref[-1])
    st, st0 = np.zeros(8), np.zeros(8)
    h.lib.scl_debug_last_solve(h.h, ptr(st0, C.c_double))   # fallback counters are cumulative per handle
    L, V, out = _tri_solve(h, G, 0, n)
    h._ck(h.lib.scl_debug_last_solve(h.h, ptr(st, C.c_double)))
    v0, v1 = 3, n // 2 + 40
    L2, V2, _ = _tri_solve(h, G, v0, v1)
    L3, _, _ = _tri_solve(h, G, 0, 0)
    assert out[5] == 0 and st[5] == 1 and st[6] == st0[6], ("the two-stage path did not produce the result", out, st, st0)
    np.testing.assert_allclose(L, Lref, rtol=2e-5, atol=3e-6 * scale)
    G64 = G.astype(np.float64)
    assert np.max(np.abs(G64 @ V - V * L[None, :])) < 5e-5 * max(1.0, scale)
    assert np.max(np.abs(V.T.astype(np.float64) @ V - np.eye(n))) < 5e-5
    np.testing.assert_array_equal(L2, L)
    assert np.max(np.abs(np.abs(np.sum(V2 * V[:, v0:v1], axis=0)) - 1.0)) < 1e-5
    np.testing.assert_array_equal(L3, L)


@pytest.mark.parametrize("v0,v1", [(100, 110), (0, 1), (650, 700)])
def test_two_stage_few_vectors(h, v0, v1):
    """An index range of a few eigenvectors (one 16-vector tile of the stage-2 kernel, the panel-by-panel stage-1
    back-transformation instead of the block reflectors) gives the vectors of the full solve."""
    n = 700
    rng = np.random.default_rng(3)
    A = rng.standard_normal((n, n + 200))
    G = (A @ A.T / A.shape[1]).astype(np.float32)
    L, V, out = _tri_solve(h, G, 0, n)
    L2, V2, out2 = _tri_solve(h, G, v0, v1)
    assert out[5] == 0 and out2[5] == 0
    np.testing.assert_array_equal(L2, L)
    assert np.max(np.abs(np.abs(np.sum(V2 * V[:, v0:v1], axis=0)) - 1.0)) < 1e-5


def test_two_stage_solver_rank_deficient_panels_fall_back(h):
    """A block-diagonal matrix with an exactly zero block has panels that CholeskyQR cannot factor: the solve must notice
    (panel flag), take the one-stage path on the kept copy, say so in the counters, and still be right."""
    rng = np.random.default_rng(11)
    nb = 300
    A = rng.standard_normal((nb, 500))
    Bm = (A @ A.T / 500).astype(np.float32)
    n = 2 * nb + 40
    G = np.zeros((n, n), np.float32)
    G[:nb, :nb] = Bm
    G[nb:2 * nb, nb:2 * nb] = Bm
    st = np.zeros(8)
    L, V, out = _tri_solve(h, G, 0, n)
    h._ck(h.lib.scl_debug_last_solve(h.h, ptr(st, C.c_double)))
    Lref = np.linalg.eigvalsh(G.astype(np.float64))
    np.testing.assert_allclose(L, Lref, rtol=2e-5, atol=5e-6)
    assert np.max(np.abs(G.astype(np.float64) @ V - V * L[None, :])) < 5e-5
    assert np.max(np.abs(V.T.astype(np.float64) @ V - np.eye(n))) < 5e-5
    assert st[6] >= 1 or st[5] == 1, st


@pytest.mark.parametrize("n", [256, 520, 1000])
def test_two_stage_reduction_stage_by_stage(h, n):
    """scl_debug_two_stage: the band matrix after stage 1 and the tridiagonal matrix after stage 2 keep the spectrum; the
    stage-2 transformation applied to the identity is orthogonal and maps band to tridiagonal; Q = Q1 Q2 maps the input to
    the tridiagonal matrix."""
    rng = np.random.default_rng(n)
    X = rng.standard_normal((n, n + 300))
    X -= X.mean(axis=0)
    G = np.ascontiguousarray((X @ X.T / X.shape[1]).astype(np.float32))
    G64 = G.astype(np.float64)
    wref = np.linalg.eigvalsh(G64)
    AB = np.zeros((n, 128), np.float32)
    d, e = np.zeros(n, np.float32), np.zeros(n - 1, np.float32)
    Q2, Q = np.zeros((n, n), np.float32), np.zeros((n, n), np.float32)
    flags = (C.c_int32 * 2)()
    h._ck(h.lib.scl_debug_two_stage(h.h, n, ptr(G, C.c_float), ptr(AB, C.c_float), ptr(d, C.c_float), ptr(e, C.c_float),
                                    ptr(Q2, C.c_float), ptr(Q, C.c_float), flags))
    assert flags[0] == 0
    Bd = np.zeros((n, n))
    for dg in range(65):
        Bd[np.arange(dg, n), np.arange(0, n - dg)] = AB[: n - dg, dg]
    Bd = Bd + np.tril(Bd, -1).T
    assert np.abs(AB[:, 65:]).max() == 0.0
    tol = 2e-6 * wref[-1]
    assert np.abs(np.linalg.eigvalsh(Bd) - wref).max() < tol
    T = np.diag(d.astype(np.float64)) + np.diag(e.astype(np.float64), 1) + np.diag(e.astype(np.float64), -1)
    assert np.abs(np.linalg.eigvalsh(T) - wref).max() < tol
    Q2m, Qm = Q2.T.astype(np.float64), Q.T.astype(np.float64)
    assert np.abs(Q2m.T @ Q2m - np.eye(n)).max() < 1e-5 and np.abs(Qm.T @ Qm - np.eye(n)).max() < 1e-5
    assert np.abs(Q2m.T @ Bd @ Q2m - T).max() < 5e-6 * wref[-1]
    assert np.abs(Qm.T @ G64 @ Qm - T).max() < 5e-6 * wref[-1]
