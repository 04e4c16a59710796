"""Oracle pin: consumes a fixture written by julia/export_fixture.jl (the unmodified reference run with a seeded RNG:
draws bundle + result Dict) and checks the oracle - and, with a GPU, the CUDA path - against it.

No run of the Julia reference has been recorded yet, so no such fixture is committed: the Julia-side tests SKIP until one
is committed as tests/golden/julia_fixture/ (they read nothing outside the repository).  The reader and the comparison
are exercised on every run by a fixture in the same format written from the oracle itself (which proves the plumbing, not the oracle)."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import sclens_oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "golden", "julia_fixture")
JULIA_TYPES = {"UInt32": np.uint32, "Int64": np.int64, "Float64": np.float64, "Float32": np.float32, "Int32": np.int32}


def read_fixture(path):
    """manifest.txt lines `name JuliaType d1xd2`; NAME.bin raw little-endian, column-major."""
    out = {}
    for ln in open(os.path.join(path, "manifest.txt")):
        name, jt, shape = ln.split()
        dims = tuple(int(d) for d in shape.split("x"))
        a = np.fromfile(os.path.join(path, name + ".bin"), dtype=JULIA_TYPES[jt])
        out[name] = a.reshape(dims, order="F") if len(dims) > 1 else a
    return out


def write_fixture(path, arrays):
    inv = {np.dtype(v): k for k, v in JULIA_TYPES.items()}
    os.makedirs(path, exist_ok=True)
    with open(os.path.join(path, "manifest.txt"), "w") as mf:
        for name, a in arrays.items():
            a = np.atleast_1d(np.asarray(a))
            np.asfortranarray(a).ravel(order="F").tofile(os.path.join(path, name + ".bin"))
            mf.write(f"{name} {inv[a.dtype]} {'x'.join(str(d) for d in a.shape)}\n")


def bundle(fx):
    """Fixture (1-based, Julia) -> counts and oracle Draws (0-based)."""
    N, M = (int(v) for v in fx["shape"])
    X = sp.csc_matrix((fx["X_nzval"], fx["X_rowval"].astype(np.int64) - 1, fx["X_colptr"].astype(np.int64) - 1), shape=(N, M))
    d = orc.Draws()
    d.z_idx1, d.z_idx2 = fx["z_idx1"].astype(np.int64) - 1, fx["z_idx2"].astype(np.int64) - 1
    d.null_perm, d.null_rows = fx["null_perm"].astype(np.int64) - 1, fx["null_rows"].astype(np.int64) - 1
    d.p_th = float(fx["p_th"][0])
    d.search_sple = [(fx[f"search_sple_{s}"] - 1).astype(np.uint32) for s in range(1, int(fx["n_search"][0]) + 1)]
    n_pert = sum(1 for k in fx if k.startswith("perturb_sple_"))
    d.perturb_sple = [(fx[f"perturb_sple_{r}"] - 1).astype(np.uint32) for r in range(1, n_pert + 1)]
    return X, d, n_pert


def compare(fx, res, info, eig_tol, vec_tol, score_tol):
    """Result of a run with the fixture's draws against the reference's outputs: the hot-path parity contract."""
    assert abs(float(fx["p_th"][0]) - float(fx["p_th"][1])) < 1e-12, "the harness replay fell out of step with the run"
    k = len(fx["signal_ev"])
    assert len(res["signal_ev"]) == k                                          # signal count: exact
    L, Lj = np.asarray(res["L"], np.float64), fx["L"]
    big = Lj >= float(info["b_min"])
    assert np.max(np.abs(L[big] - Lj[big]) / Lj[big]) < eig_tol                # eigenvalues: 1e-4 relative
    assert abs(float(res["lambda"]) - float(fx["lambda_c"][0])) / float(fx["lambda_c"][0]) < eig_tol
    assert abs(len(res["L_mp"]) - len(fx["L_mp"])) <= 1
    c = np.abs(np.sum(np.asarray(res["signal_evec"], np.float64) * fx["signal_evec"], axis=0))
    assert np.arccos(np.clip(c, 0, 1)).max() < vec_tol                         # signal eigenvectors up to sign
    assert info["n_search"] == int(fx["n_search"][0]) and abs(info["p_sel"] - float(fx["p_sel"][0])) < 1e-12
    np.testing.assert_array_equal(np.asarray(res["sig_id"]) + 1, fx["sig_id"])   # Julia is 1-based
    np.testing.assert_allclose(res["robustness_scores"]["m_scores"], fx["m_scores"], atol=score_tol)
    for key in ("TGC", "mat2_mean", "mat2_std", "norm_tgc", "cent_"):
        np.testing.assert_allclose(np.ravel(res["rec_vals"][key]), fx["rec_" + key], rtol=1e-9, atol=1e-14)


def test_fixture_format_round_trip(tmp_path):
    """Write a fixture in export_fixture.jl's format from an oracle run, read it back, replay it through the oracle."""
    from sclens_b200.synth import make_counts
    X = make_counts(260, 420, seed=8, K=4, de_prob=0.3, lfc_sd=1.5)
    res, draws, info = orc.sclens(X, rng=np.random.default_rng(1), mode="gpu-ref", n_perturb=4, n_baseline=100)
    arrays = {"shape": np.array(X.shape, np.int64), "X_colptr": X.indptr.astype(np.uint32) + 1, "X_rowval": X.indices.astype(np.uint32) + 1,
              "X_nzval": X.data.astype(np.float32), "z_idx1": draws.z_idx1.astype(np.uint32) + 1, "z_idx2": draws.z_idx2.astype(np.uint32) + 1,
              "null_perm": draws.null_perm.astype(np.uint32) + 1, "null_rows": draws.null_rows.astype(np.uint32) + 1,
              "p_th": np.array([draws.p_th, draws.p_th]), "n_search": np.array([info["n_search"]], np.int64),
              "p_sel": np.array([info["p_sel"]]), "L": np.asarray(res["L"], np.float64), "L_mp": np.asarray(res["L_mp"], np.float64),
              "lambda_c": np.array([float(res["lambda"])]), "signal_ev": np.asarray(res["signal_ev"], np.float64),
              "signal_evec": np.asarray(res["signal_evec"], np.float64), "sig_id": np.asarray(res["sig_id"], np.int64) + 1,
              "m_scores": np.asarray(res["robustness_scores"]["m_scores"], np.float64)}
    for s, a in enumerate(draws.search_sple):
        arrays[f"search_sple_{s + 1}"] = a.astype(np.uint32) + 1
    for r, a in enumerate(draws.perturb_sple):
        arrays[f"perturb_sple_{r + 1}"] = a.astype(np.uint32) + 1
    for key in ("TGC", "mat2_mean", "mat2_std", "norm_tgc", "cent_"):
        arrays["rec_" + key] = np.ravel(res["rec_vals"][key]).astype(np.float64)
    write_fixture(str(tmp_path), arrays)
    fx = read_fixture(str(tmp_path))
    assert fx["signal_evec"].shape == np.asarray(res["signal_evec"]).shape      # column-major round trip
    X2, d2, n_pert = bundle(fx)
    assert (X2 != X).nnz == 0 and n_pert == 4
    res2, _, info2 = orc.sclens(X2, draws=d2, mode="gpu-ref", n_perturb=n_pert)
    compare(fx, res2, info2, 1e-6, 1e-3, 1e-6)      # same code, same draws: only Float32 storage of the vectors differs


@pytest.mark.skipif(not os.path.exists(os.path.join(FIXTURE, "manifest.txt")),
                    reason="no fixture from julia/export_fixture.jl (no Julia in the build image): oracle parity stays unpinned")
def test_oracle_matches_the_julia_reference():
    fx = read_fixture(FIXTURE)
    X, d, n_pert = bundle(fx)
    res, _, info = orc.sclens(X, draws=d, mode="gpu-ref", n_perturb=n_pert)
    compare(fx, res, info, 1e-4, 5e-3, 2e-2)


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(os.path.join(FIXTURE, "manifest.txt")),
                    reason="no fixture from julia/export_fixture.jl (no Julia in the build image)")
def test_cuda_path_matches_the_julia_reference():
    from sclens_b200 import SCL_GRAM_FP16X3, sclens
    fx = read_fixture(FIXTURE)
    X, d, n_pert = bundle(fx)
    out = sclens(X, draws=d, n_perturb=n_pert, gram_mode=SCL_GRAM_FP16X3, exact_perturb=True, verbose=False)
    info = {"b_min": out["info"]["b_minus"], "n_search": out["info"]["n_search"], "p_sel": out["info"]["p_sel"]}
    compare(fx, out, info, 1e-4, 5e-3, 2e-2)
