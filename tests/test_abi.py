"""CPU tests of the C-ABI boundary: the library loads, exports every symbol the header declares,
binds with the signatures the Python mirror uses, and fails loudly without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "sclens_b200.h")).read()
    return sorted(set(re.findall(r"SCL_API\s+[\w\s\*]+?\b(scl_\w+)\s*\(", txt)))


def test_header_and_binding_agree(lib_built):
    from sclens_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 40
    assert sorted(_lib.SIGNATURES) == syms
    lib = C.CDLL(lib_built)
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/sclens_b200.h but not exported"


def test_no_torch_types_in_the_abi():
    txt = open(os.path.join(ROOT, "include", "sclens_b200.h")).read()
    assert "torch" not in txt.lower() and "at::" not in txt and "std::" not in txt
    assert 'extern "C"' in txt


def test_struct_layouts_match_header(lib_built, tmp_path):
    """sizeof of every struct as gcc sees the header == the ctypes mirror (plain C, no C++ needed)."""
    import subprocess
    from sclens_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "sclens_b200.h"\nint main(void){printf("%zu %zu %zu %zu\\n",'
                   'sizeof(scl_config),sizeof(scl_signal_info),sizeof(scl_robust_info),sizeof(scl_profile));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert sizes == [C.sizeof(_lib.Config), C.sizeof(_lib.SignalInfo), C.sizeof(_lib.RobustInfo), C.sizeof(_lib.Profile)]


def test_fails_loudly_without_gpu(lib_built):
    """In a process that sees no device (none there, or hidden by CUDA_VISIBLE_DEVICES)."""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, pytest\n"
            "from sclens_b200 import Handle, SclError, sclens\n"
            "with pytest.raises(SclError) as e:\n"
            "    Handle()\n"
            "assert e.value.code == -4 and 'no CPU fallback' in str(e.value)\n"
            "with pytest.raises(ValueError):\n"
            "    sclens(np.eye(4), device_='cpu')\n" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                         text=True)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: no product source imports it, and importing the package does
    not pull it in."""
    import subprocess
    import sys
    pkg = os.path.join(ROOT, "sclens_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f"{f} imports the oracle"
    code = "import sys; sys.path.insert(0, %r); import sclens_b200, sclens_b200.preprocess, sclens_b200.synth; " \
           "assert not [m for m in sys.modules if m.split('.')[0] == 'oracle']" % ROOT
    subprocess.check_call([sys.executable, "-c", code])


def test_host_only_entry_points(lib_built):
    """scl_op_mp_fit and the work-partition helpers are pure host code: callable without a GPU."""
    from oracle import sclens_oracle as orc
    from sclens_b200 import _lib
    from sclens_b200._lib import ptr
    lib = _lib.load()
    rng = np.random.default_rng(0)
    n, K = 300, 700
    L = np.linalg.eigvalsh(np.cov(rng.standard_normal((n, K)), bias=True)).astype(np.float32)
    Lr = np.linalg.eigvalsh(np.cov(rng.standard_normal((n, K)), bias=True)).astype(np.float32)
    L[-3:] = [3.5, 4.5, 7.0]
    out = np.empty(8)
    Lr1 = np.ascontiguousarray(Lr[:-1])
    assert lib.scl_op_mp_fit(ptr(L, C.c_float), n, ptr(Lr1, C.c_float), n - 1, ptr(out, C.c_double)) == 0
    L_mp, b_plus, b_min, it = orc.mp_calculation(L.astype(np.float64), Lr1.astype(np.float64))
    lam = orc.tw(L.astype(np.float64), L_mp)[0]
    assert abs(out[0] - lam) < 1e-12 * lam and abs(out[1] - b_plus) < 1e-12 and abs(out[2] - b_min) < 1e-12
    assert int(out[4]) == len(L_mp) and int(out[5]) == it and int(out[7]) == 3
    chk = orc.mp_check(L_mp)
    assert abs(out[3] - chk["ks_static"]) < 1e-9 and bool(out[6]) == chk["pass"]
    # degenerate input -> error code, not a crash
    assert lib.scl_op_mp_fit(ptr(L, C.c_float), 1, ptr(Lr1, C.c_float), 1, ptr(out, C.c_double)) < 0
    ids = np.empty(32, np.int32)
    cnt = C.c_int32()
    seen = []
    for r in range(3):
        assert lib.scl_plan_replicates(20, 3, r, ptr(ids, C.c_int32), C.byref(cnt)) == 0
        seen += ids[:cnt.value].tolist()
    assert sorted(seen) == list(range(20))
    step = C.c_int32()
    assert lib.scl_plan_search_wave(2, 8, 5, C.byref(step)) == 0 and step.value == 21
    assert lib.scl_plan_replicates(20, 0, 0, None, C.byref(cnt)) < 0


def test_julia_shim_is_in_step_with_the_header():
    """julia/sclens_b200.jl cannot be executed here (no Julia in the image): check statically that every symbol it
    ccalls is declared in the header and that its struct mirrors list the same fields, in order, as the ctypes
    mirrors (which test_struct_layouts_match_header ties to the header)."""
    from sclens_b200 import _lib
    src = open(os.path.join(ROOT, "julia", "sclens_b200.jl")).read()
    called = set(re.findall(r"\(:(scl_\w+),\s*LIB\)", src))
    assert called and called <= set(header_symbols()), called - set(header_symbols())
    for name, mirror in (("SclConfig", _lib.Config), ("SclSignalInfo", _lib.SignalInfo), ("SclRobustInfo", _lib.RobustInfo)):
        body = src[src.index(f"struct {name}"):]
        body = body[:body.index("\nend")]
        fields = re.findall(r"(\w+)::", body)
        want = [f[0].rstrip("_") for f in mirror._fields_]
        assert fields == want, (name, fields, want)
    # positional constructor call has one argument per field
    ctor = re.search(r"SclConfig\(([^\n]*)\)\n", src[src.index("default_config"):]).group(1)
    depth, nargs = 0, 1
    for ch in ctor:
        depth += ch in "([{"
        depth -= ch in ")]}"
        nargs += ch == "," and depth == 0
    assert nargs == len(_lib.Config._fields_)


def _oracle_score_tail(b_, th):
    """Tail of oracle.robustness_scores (:797-806) on a given similarity table."""
    import math
    q1 = np.quantile(b_, 0.25, axis=1)
    q3 = np.quantile(b_, 0.75, axis=1)
    iqr = q3 - q1
    m, sd = np.zeros(b_.shape[0]), np.zeros(b_.shape[0])
    for s in range(b_.shape[0]):
        row = b_[s]
        f = row[(q1[s] - 1.5 * iqr[s] <= row) & (row <= q3[s] + 1.5 * iqr[s])]
        m[s] = np.median(f)
        sd[s] = np.std(f, ddof=1) if len(f) > 1 else np.nan
    return m, sd, np.nonzero(m > math.cos(math.radians(th)))[0]


@pytest.mark.parametrize("k,n_pairs,seed", [(7, 190, 0), (3, 1, 1), (5, 3, 2), (12, 45, 3), (1, 6, 4)])
def test_score_tail_matches_oracle(lib_built, k, n_pairs, seed):
    """scl_op_scores_from_pairs (Tukey fence, median, corrected std, robust set) is pure host code: compare with the
    oracle's restatement of :797-806, including one pair only (n_perturb = 2), outliers and tied values."""
    from sclens_b200 import _lib
    from sclens_b200._lib import ptr
    lib = _lib.load()
    rng = np.random.default_rng(seed)
    b = rng.uniform(0.3, 1.0, size=(k, n_pairs)).astype(np.float32)
    if n_pairs > 4:
        b[0, :2] = 0.01                       # outliers below the fence
        b[-1, :] = np.float32(0.75)           # all tied: iqr = 0, everything kept
        b[k // 2, ::2] = b[k // 2, 1]         # many ties
    bf = np.asfortranarray(b)                 # k x n_pairs column-major
    m, sd = np.empty(k), np.empty(k)
    sig = np.empty(k, np.int32)
    nrob = C.c_int32()
    for th in (60.0, 30.0, 75.0):
        assert lib.scl_op_scores_from_pairs(ptr(bf, C.c_float), k, n_pairs, th, ptr(m, C.c_double), ptr(sd, C.c_double),
                                            ptr(sig, C.c_int32), C.byref(nrob)) == 0
        wm, wsd, wsig = _oracle_score_tail(b.astype(np.float64), th)
        np.testing.assert_allclose(m, wm, rtol=1e-12)
        np.testing.assert_allclose(sd, wsd, rtol=1e-9, atol=1e-15, equal_nan=True)
        assert sig[:nrob.value].tolist() == wsig.tolist()
    assert lib.scl_op_scores_from_pairs(ptr(bf, C.c_float), 0, n_pairs, 60.0, None, None, None, C.byref(nrob)) < 0


def test_df2sparr_host_mirror():
    """df2sparr (:90-120) on the host: DataFrame with the cell column first and dense or pandas-sparse gene columns,
    scipy matrices and ndarrays all become the same canonical Float32 CSC (sorted, duplicates summed, stored zeros
    dropped) with the ids the result dictionary carries."""
    import pandas as pd
    import scipy.sparse as sp
    from sclens_b200 import df2sparr
    rng = np.random.default_rng(0)
    dense = rng.poisson(0.3, size=(40, 17)).astype(np.float32)
    dense[:, 5] = 0                                    # an all-zero gene stays a (empty) column
    genes = [f"G{j}" for j in range(17)]
    cells = [f"cell{i}" for i in range(40)]
    df = pd.DataFrame(dense, columns=genes)
    df.insert(0, "cell", cells)
    X, cid, gid = df2sparr(df)
    assert sp.isspmatrix_csc(X) and X.dtype == np.float32 and X.shape == (40, 17)
    assert X.has_canonical_format and (X.data > 0).all()
    np.testing.assert_array_equal(X.toarray(), dense)
    assert cid.tolist() == cells and list(gid) == genes
    sdf = pd.DataFrame({g: pd.arrays.SparseArray(dense[:, j], fill_value=0) for j, g in enumerate(genes)})
    sdf.insert(0, "cell", cells)
    Xs, _, _ = df2sparr(sdf)
    assert (Xs != X).nnz == 0 and np.array_equal(Xs.indptr, X.indptr) and np.array_equal(Xs.indices, X.indices)
    # COO input with duplicates and an explicit zero: summed / dropped like sparse(I, J, V) followed by dropzeros
    coo = sp.coo_matrix((np.array([1, 2, 0, 3], np.float32), (np.array([0, 0, 1, 2]), np.array([1, 1, 0, 3]))), shape=(4, 5))
    Xc, cid2, gid2 = df2sparr(coo)
    assert Xc.nnz == 2 and Xc[0, 1] == 3 and Xc[2, 3] == 3 and cid2[0] == "c0" and gid2[4] == "g4"
    Xn, _, _ = df2sparr(dense)
    assert (Xn != X).nnz == 0


def test_get_denoised_df_validates_before_touching_the_device(lib_built):
    """get_denoised_df (:889-931 mirror): shape / dtype / device_ errors are raised on the host; a well-formed call
    without a GPU fails loudly at handle creation (no CPU fallback)."""
    import torch
    from sclens_b200 import SclError, get_denoised_df
    N, M, k = 12, 9, 4
    rng = np.random.default_rng(0)
    res = {"gene_basis": rng.standard_normal((k, M)).astype(np.float32), "sig_id": np.array([0, 2]),
           "pca_n1": rng.standard_normal((N, 2)).astype(np.float32), "cell_id": np.arange(N), "gene_id": np.arange(M),
           "rec_vals": {"TGC": np.ones(N), "mat2_mean": np.zeros((1, M)), "mat2_std": np.ones((1, M)),
                        "norm_tgc": np.ones(N), "cent_": np.zeros((1, M))}}
    with pytest.raises(ValueError):
        get_denoised_df(res, device_="cpu")
    with pytest.raises(ValueError):
        get_denoised_df(dict(res, sig_id=np.array([], dtype=np.int64)))
    with pytest.raises(ValueError):
        get_denoised_df(dict(res, pca_n1=res["pca_n1"][:, :1]))
    with pytest.raises(ValueError):
        get_denoised_df(dict(res, rec_vals=dict(res["rec_vals"], TGC=np.ones(N + 1))))
    with pytest.raises(ValueError):
        get_denoised_df(res, dtype=np.float16)
    if not torch.cuda.is_available():
        with pytest.raises(SclError) as e:
            get_denoised_df(res)
        assert e.value.code == -4
