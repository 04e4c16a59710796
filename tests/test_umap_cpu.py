"""CPU tests of apply_umap! (:863-873): the oracle's restatement of UMAP.jl's pieces, the host-side a/b fit of the library,
the ABI mirrors of the new structs, argument checks before any device is touched, and the evidence that the synchronous
epoch of the device layout costs no quality against UMAP.jl's edge-by-edge order."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import umap_ref as U

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def mixture(n_per, centers, d, seed, sd=1.0):
    rng = np.random.default_rng(seed)
    X = np.vstack([rng.normal(0, sd, (n_per, d)) + c for c in centers])
    return X, np.repeat(np.arange(len(centers)), n_per)


def test_oracle_fit_ab_at_default_min_dist():
    a, b = U.fit_ab(0.1)
    assert abs(a - 1.57694) < 1e-4 and abs(b - 0.89506) < 1e-4


def test_library_fit_ab_matches_oracle(lib_built):
    from sclens_b200 import _lib
    lib = _lib.load()
    for md, spread in ((0.0, 1.0), (0.05, 1.0), (0.1, 1.0), (0.25, 1.0), (0.5, 1.0), (0.8, 1.0), (0.1, 2.0)):
        a, b = C.c_double(), C.c_double()
        assert lib.scl_umap_fit_ab(md, spread, C.byref(a), C.byref(b)) == 0
        wa, wb = U.fit_ab(md, spread)
        assert abs(a.value - wa) < 1e-6 and abs(b.value - wb) < 1e-6, (md, spread, a.value, wa, b.value, wb)
    assert lib.scl_umap_fit_ab(0.1, 0.0, C.byref(a), C.byref(b)) < 0


def test_sigma_bisection_meets_log2k():
    X, _ = mixture(100, [np.zeros(6), np.full(6, 5.0)], 6, seed=1)
    for k in (5, 15, 30):
        idx, dist = U.knn(X, k, "euclidean")
        rho, sigma = U.smooth_knn_dists(dist, k)
        psum = np.exp(-np.maximum(dist - rho[:, None], 0) / sigma[:, None]).sum(1)
        np.testing.assert_allclose(psum, np.log2(k), atol=1e-5)
        assert (rho > 0).all() and np.allclose(rho, dist[:, 0])


def test_fuzzy_union_symmetric_in_unit_interval():
    X, _ = mixture(80, [np.zeros(4), np.full(4, 3.0), np.full(4, -3.0)], 4, seed=2)
    idx, dist = U.knn(X, 15, "cosine")
    g = U.graph_from_knn(idx, dist, 15)
    assert abs(g - g.T).max() == 0
    assert g.data.min() > 0 and g.data.max() <= 1.0
    assert g.diagonal().max() == 0 and g.has_sorted_indices


def test_struct_layouts_and_julia_mirrors(lib_built, tmp_path):
    from sclens_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "sclens_b200.h"\nint main(void){printf("%zu %zu\\n",'
                   'sizeof(scl_umap_params),sizeof(scl_umap_info));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert sizes == [C.sizeof(_lib.UmapParams), C.sizeof(_lib.UmapInfo)]
    jl = open(os.path.join(ROOT, "julia", "sclens_b200.jl")).read()
    for name, mirror in (("SclUmapParams", _lib.UmapParams), ("SclUmapInfo", _lib.UmapInfo)):
        body = jl[jl.index(f"struct {name}"):]
        body = body[:body.index("\nend")]
        assert re.findall(r"(\w+)::", body) == [f[0] for f in mirror._fields_], name


def test_apply_umap_validates_before_touching_the_device(lib_built):
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import numpy as np, pytest\n"
            "from sclens_b200 import SclError, apply_umap\n"
            "X = np.random.default_rng(0).standard_normal((50, 4)).astype(np.float32)\n"
            "res = {'pca_n1': X}\n"
            "for kw in (dict(k=0), dict(k=65), dict(k=50), dict(nc=0), dict(metric='manhattan'), dict(init='pca'),\n"
            "           dict(md=-1.0), dict(n_epochs=-1)):\n"
            "    with pytest.raises(ValueError):\n"
            "        apply_umap(dict(res), **kw)\n"
            "bad = X.copy(); bad[3, 1] = np.nan\n"
            "with pytest.raises(ValueError):\n"
            "    apply_umap({'pca_n1': bad})\n"
            "with pytest.raises(ValueError):\n"
            "    apply_umap({})\n"
            "with pytest.raises(SclError) as e:\n"
            "    apply_umap(res)\n"
            "assert e.value.code == -4\n" % ROOT)
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                         text=True)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]


def test_synchronous_epoch_costs_no_quality():
    """Deviation 2 (DESIGN.md): on a 3-cluster Gaussian mixture of 600 points, trustworthiness (k = 15) of the
    synchronous layout is at least that of UMAP.jl's edge-by-edge order minus 0.02, from the same spectral start."""
    from sklearn.manifold import trustworthiness
    X, _ = mixture(200, [np.zeros(5), np.full(5, 6.0), np.r_[np.full(3, 12.0), 0, 0]], 5, seed=0)
    idx, dist = U.knn(X, 15, "euclidean")
    g = U.graph_from_knn(idx, dist, 15)
    _, V = U.spectral_vectors(g, 2)
    P0 = V * (10.0 / V.max())
    a, b = U.fit_ab(0.1)
    t_sync = trustworthiness(X, U.layout_sync(g, P0, 200, a, b, seed=0), n_neighbors=15)
    t_seq = trustworthiness(X, U.layout_sequential(g, P0, 200, a, b, seed=0), n_neighbors=15)
    assert t_sync >= t_seq - 0.02, (t_sync, t_seq)


def test_draws_are_a_pure_function_of_their_counters():
    k1, k2 = U.stream_key(7, 1, 3), U.stream_key(7, 1, 4)
    u = U.draw_unit(k1, np.arange(1000), 0)
    assert (u >= 0).all() and (u < 1).all() and abs(u.mean() - 0.5) < 0.05
    assert not np.array_equal(u, U.draw_unit(k2, np.arange(1000), 0))
    np.testing.assert_array_equal(u, U.draw_unit(k1, np.arange(1000), 0))
    j = U.draw_index(k1, np.arange(5000), 3, 17)
    assert j.min() == 0 and j.max() == 16
