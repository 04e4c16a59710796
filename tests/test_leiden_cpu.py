"""CPU checks of the clustering pieces: the ECS closed form, IC, the search's planning step (host code behind the C ABI
against oracle/leiden_ref.py) and the layouts of the new ABI structs."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import leiden_ref as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_ecs_closed_form_matches_definition(seed):
    rng = np.random.default_rng(seed)
    a, b = rng.integers(0, 4, 60), rng.integers(0, 7, 60)
    assert abs(L.ecs_pair(a, b) - L.ecs_brute(a, b)) < 1e-12
    assert abs(L.ecs_pair(a, a) - 1.0) < 1e-15


def test_ecs_hand_computed():
    # A = {0,1},{2}; B = {0},{1,2}: cell 0: 1 - (|1/2 - 1| + 1/2)/2 = 1/2; cell 1: 1 - (1/2 + 0 + 1/2)/2 = 1/2;
    # cell 2: 1 - (1/2 + |1 - 1/2|)/2 = 1/2.
    assert abs(L.ecs_pair([0, 0, 1], [0, 1, 1]) - 0.5) < 1e-15
    # one cluster against singletons: cell i: 1 - (|1/3 - 1| + 2 * 1/3)/2 = 1/3
    assert abs(L.ecs_pair([0, 0, 0], [0, 1, 2]) - 1 / 3) < 1e-15


def test_ic_of_identical_and_renamed_labelings():
    rng = np.random.default_rng(3)
    a = rng.integers(0, 5, 100)
    renamed = (a + 3) % 5
    assert L.ic(L.ecs_matrix([a, a, renamed, a])) == pytest.approx(1.0, abs=1e-15)
    b = rng.integers(0, 5, 100)
    assert L.ic(L.ecs_matrix([a, b])) > 1.0


def test_weight_shift():
    assert L.weight_shift(1.0, 2_000_000) == 32
    assert L.weight_shift(1000.0, 10 ** 9) == 61 - 30 - 10


def _plan_lib(lib, gam, modes, k_min, k_max, **kw):
    from sclens_b200._lib import ClusterParams
    p = ClusterParams(k_min=k_min, k_max=k_max, n_trials=2, max_rounds=12, n_grid=16, max_widen=kw.get("max_widen", 4),
                      max_iterations=10, max_sweeps=64, gamma_lo=0.01, gamma_hi=10.0, theta=0.01, seed=0)
    g = np.asarray(gam, np.float64)
    m = np.asarray(modes, np.int32)
    out = np.empty(k_max - k_min + 3)
    n = C.c_int32()
    rc = lib.scl_cluster_plan(len(g), g.ctypes.data_as(C.POINTER(C.c_double)), m.ctypes.data_as(C.POINTER(C.c_int32)),
                              C.byref(p), out.ctypes.data_as(C.POINTER(C.c_double)), C.byref(n))
    assert rc == 0
    return list(out[:n.value])


@pytest.mark.parametrize("table", [
    lambda g: int(np.clip(np.floor(2 + 6 * np.log10(g / 0.01)), 1, 40)),            # monotone, every k reachable
    lambda g: int(np.clip(np.floor(30 * g), 3, 60)),                                  # at least three components
    lambda g: 12 if 0.3 < g < 0.4 else int(np.clip(np.floor(4 * np.log10(g / 0.001)), 1, 30)),   # a bump
])
def test_search_plan_matches_oracle(lib_built, table):
    from sclens_b200 import _lib
    lib = _lib.load()
    eg, em = L.search(table)
    lo, hi = 0.01 * 1e-4, 10.0 * 1e4
    # replay every step through the host planner
    grid = L.start_grid()
    n = len(grid)
    while n < len(eg):
        want = L.plan(eg[:n], em[:n], 2, 20, lo, hi)
        got = _plan_lib(lib, eg[:n], em[:n], 2, 20)
        np.testing.assert_allclose(got, want, rtol=1e-15)
        n += len(want)
    assert _plan_lib(lib, eg, em, 2, 20) == [] or len(eg) >= 16 + 12


def test_search_brackets_every_reachable_count():
    eg, em = L.search(lambda g: int(np.clip(np.floor(2 + 6 * np.log10(g / 0.01)), 1, 40)))
    assert set(range(2, 21)) <= set(em)
    eg, em = L.search(lambda g: int(np.clip(np.floor(30 * g), 3, 60)))
    assert 2 not in em and min(eg) < 0.01   # not reachable: widened to the limit, reported missing


def test_struct_layouts_of_the_clustering_abi(lib_built, tmp_path):
    from sclens_b200 import _lib
    src = tmp_path / "s.c"
    exe = tmp_path / "s"
    src.write_text('#include <stdio.h>\n#include "sclens_b200.h"\nint main(void){printf("%zu %zu %zu %zu\\n",'
                   'sizeof(scl_leiden_params),sizeof(scl_leiden_info),sizeof(scl_cluster_params),sizeof(scl_cluster_info));'
                   'return 0;}\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert sizes == [C.sizeof(_lib.LeidenParams), C.sizeof(_lib.LeidenInfo), C.sizeof(_lib.ClusterParams),
                     C.sizeof(_lib.ClusterInfo)]


def test_clustering_checks_arguments_before_the_device():
    import scipy.sparse as sp
    from sclens_b200 import clustering
    g = sp.identity(5, format="csr")
    with pytest.raises(ValueError):
        clustering({"umap_obj": {"graph": g}}, k_min=3, k_max=2)
    with pytest.raises(ValueError):
        clustering({"umap_obj": {"graph": g}}, k_max=9)
    with pytest.raises(ValueError):
        clustering({"umap_obj": {"graph": g}}, n_trials=1)
    with pytest.raises(ValueError):
        clustering({}, k_max=3)


@pytest.mark.parametrize("gamma", [0.5, 1.0, 2.0])
def test_oracle_leiden_connected_and_as_good_as_louvain(gamma):
    import networkx as nx
    from scipy.sparse.csgraph import connected_components
    from oracle import umap_ref as U
    rng = np.random.default_rng(21)
    C = rng.normal(0, 3.0, (6, 5))
    X = np.vstack([rng.normal(0, 1, (40, 5)) + c for c in C])
    idx, dist = U.knn(X, 15, "euclidean")
    g = U.graph_from_knn(idx, dist, 15)
    G = nx.from_scipy_sparse_array(g)
    q_lou = nx.community.modularity(G, nx.community.louvain_communities(G, weight="weight", resolution=gamma, seed=0),
                                    weight="weight", resolution=gamma)
    for trial in range(2):
        st = {}
        lab = L.leiden(g, gamma, seed=1, trial=trial, stats=st)
        assert st["max_levels"] >= 2
        k = lab.max() + 1
        assert (np.diff(np.bincount(lab)) <= 0).all()
        for c in range(k):
            m = np.nonzero(lab == c)[0]
            assert connected_components(g[m][:, m], directed=False)[0] == 1
        q = nx.community.modularity(G, [set(np.nonzero(lab == c)[0]) for c in range(k)], weight="weight",
                                    resolution=gamma)
        assert q >= q_lou - 0.01, (q, q_lou)
