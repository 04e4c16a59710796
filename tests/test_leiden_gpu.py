"""-m gpu checks of the device clustering (scl_op_leiden / scl_op_label_ecs / scl_op_cluster): determinism, batch
invariance, modularity and connectivity of the result, quality against networkx Louvain, long rows, graph validation,
ECS / IC against the oracle and the end-to-end clustering() call."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

from oracle import leiden_ref as L
from sclens_b200 import Handle, SclError, apply_umap, clustering, sclens
from sclens_b200.synth import make_counts

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def h():
    with Handle() as hh:
        yield hh


def mixture(n_per, n_clusters, d, seed, sep=8.0):
    rng = np.random.default_rng(seed)
    C = rng.normal(0, sep, (n_clusters, d))
    X = np.vstack([rng.normal(0, 1, (n_per, d)) + c for c in C]).astype(np.float32)
    return X, np.repeat(np.arange(n_clusters), n_per)


def umap_graph(h, X, k=15):
    h.umap(X, k, 2, metric="euclidean", n_epochs=0, init="random")
    return h.umap_graph()


def nx_graph(g):
    import networkx as nx
    return nx.from_scipy_sparse_array(sp.csr_matrix(g, dtype=np.float64))


def test_deterministic_and_seeded(h):
    X, _ = mixture(300, 5, 6, seed=1)
    g = umap_graph(h, X)
    a = h.leiden(g, [0.5, 1.0, 2.0], 4, seed=3)[0]
    b = h.leiden(g, [0.5, 1.0, 2.0], 4, seed=3)[0]
    c = h.leiden(g, [0.5, 1.0, 2.0], 4, seed=4)[0]
    assert a.tobytes() == b.tobytes()
    assert a.tobytes() != c.tobytes()


def test_batch_invariance(h):
    X, _ = mixture(250, 6, 5, seed=2)
    g = umap_graph(h, X)
    gam = [0.3, 1.0, 3.0]
    lab = h.leiden(g, gam, 3, seed=7)[0]
    for r, gm in enumerate(gam):
        alone = h.leiden(g, [gm], 3, seed=7)[0][0]
        np.testing.assert_array_equal(alone, lab[r])
        first = h.leiden(g, [gm], 1, seed=7)[0][0, 0]
        np.testing.assert_array_equal(first, lab[r, 0])


def test_handle_graph_equals_passed_graph(h):
    X, _ = mixture(200, 4, 5, seed=3)
    g = umap_graph(h, X)
    a = h.leiden(None, [1.0], 3, seed=1)
    b = h.leiden(g, [1.0], 3, seed=1)
    assert a[0].tobytes() == b[0].tobytes() and a[2].tobytes() == b[2].tobytes()


@pytest.mark.parametrize("gamma", [0.2, 1.0, 2.5])
def test_modularity_connectivity_quality(h, gamma):
    import networkx as nx
    X, _ = mixture(300, 8, 6, seed=4, sep=4.0)
    g = umap_graph(h, X).astype(np.float64)
    lab, ncl, mod, info = h.leiden(g, [gamma], 4, seed=2)
    G = nx_graph(g)
    lou = nx.community.louvain_communities(G, weight="weight", resolution=gamma, seed=0)
    q_lou = nx.community.modularity(G, lou, weight="weight", resolution=gamma)
    for t in range(4):
        l = lab[0, t]
        assert ncl[0, t] == l.max() + 1 and set(np.unique(l)) == set(range(ncl[0, t]))
        sizes = np.bincount(l)
        assert (np.diff(sizes) <= 0).all()
        comms = [set(np.nonzero(l == c)[0]) for c in range(ncl[0, t])]
        q = nx.community.modularity(G, comms, weight="weight", resolution=gamma)
        assert abs(mod[0, t] - q) <= 1e-9, (mod[0, t], q)
        assert q >= q_lou - 0.01, (q, q_lou)
        for c in range(ncl[0, t]):
            idx = np.nonzero(l == c)[0]
            assert connected_components(g[idx][:, idx], directed=False)[0] == 1


def oracle_graph(n_per=50, n_clusters=6, sep=2.0, seed=11):
    from oracle import umap_ref as U
    rng = np.random.default_rng(seed)
    C = rng.normal(0, sep, (n_clusters, 5))
    X = np.vstack([rng.normal(0, 1, (n_per, 5)) + c for c in C])
    idx, dist = U.knn(X, 15, "euclidean")
    return U.graph_from_knn(idx, dist, 15), X.astype(np.float32)


@pytest.mark.parametrize("source", ["oracle_graph", "device_graph"])
def test_labels_match_oracle_bit_for_bit(h, source):
    """Every label of every trial equals the oracle's step-for-step restatement (oracle/leiden_ref.leiden): same hashes,
    integer weights, gain expression and tie rules, across levels and iteration restarts.  The refinement's Gumbel draws
    go through the device's and numpy's double log, which may differ by an ulp: a choice could differ only when two
    perturbed scores lie within ~1e-16 of each other."""
    g, X = oracle_graph()
    if source == "device_graph":
        g = umap_graph(h, X).astype(np.float64)
    gam = [0.5, 1.0, 2.0]
    lab, ncl, _, info = h.leiden(g, gam, 4, seed=5)
    levels, iters = [], []
    for r, gm in enumerate(gam):
        for t in range(4):
            st = {}
            want = L.leiden(g, gm, seed=5, trial=t, stats=st)
            np.testing.assert_array_equal(lab[r, t], want, err_msg=f"gamma {gm} trial {t}")
            levels.append(st["max_levels"])
            iters.append(st["iterations"])
    assert info.weight_shift == 32 and info.max_levels == max(levels) and info.max_iterations == max(iters)
    assert max(levels) >= 2
    assert max(iters) >= 3      # the second iteration's restart changed labels, and the device followed it


def test_star_and_complete_graphs(h):
    n = 3000                                   # hub row of 2999 entries: the global-memory table
    star = sp.coo_matrix((np.ones(n - 1), (np.zeros(n - 1, int), np.arange(1, n))), shape=(n, n))
    star = (star + star.T).tocsr()
    lab, ncl, mod, _ = h.leiden(star, [1.0], 2, seed=0)
    assert (ncl >= 1).all() and np.isfinite(mod).all()
    for t in range(2):
        l = lab[0, t]
        for c in range(ncl[0, t]):
            idx = np.nonzero(l == c)[0]
            assert connected_components(star[idx][:, idx], directed=False)[0] == 1
    m = 700                                     # every row long
    full = sp.csr_matrix(np.ones((m, m)) - np.eye(m))
    lab, ncl, mod, _ = h.leiden(full, [1.0, 0.5], 2, seed=0)
    assert (ncl == 1).all()
    np.testing.assert_allclose(mod[1], 0.5, atol=1e-12)   # 1 - 0.5 * 1


def test_invalid_graphs_are_errors(h):
    g = sp.csr_matrix(np.array([[0, 1.0, 0], [1.0, 0, 2.0], [0, 2.0, 0]]))
    bad_sym = g.copy()
    bad_sym.data[0] = 3.0
    with pytest.raises(SclError) as e:
        h.leiden(bad_sym, [1.0], 1)
    assert e.value.code == -7
    bad_val = g.copy()
    bad_val.data[:] = np.nan
    with pytest.raises(SclError):
        h.leiden(bad_val, [1.0], 1)
    N, nnz, rp, ci, v = 3, g.nnz, g.indptr.astype(np.uint32), g.indices.astype(np.uint32), g.data.astype(np.float64)
    import ctypes as C
    from sclens_b200._lib import LeidenInfo, LeidenParams, ptr
    p = LeidenParams(n_trials=1, max_iterations=1, max_sweeps=4, theta=0.01, seed=0)
    for rp2, ci2 in ((np.array([0, 2, 1, 4], np.uint32), ci), (rp, np.array([1, 0, 7, 1], np.uint32)),
                     (rp, np.array([1, 2, 0, 1], np.uint32))):
        lab, ncl, mod, info = np.empty(3, np.int32), np.empty(1, np.int32), np.empty(1), LeidenInfo()
        res = np.array([1.0])
        rc = h.lib.scl_op_leiden(h.h, N, nnz, ptr(rp2, C.c_uint32), ptr(ci2, C.c_uint32), ptr(v, C.c_double), 1,
                                 ptr(res, C.c_double), C.byref(p), ptr(lab, C.c_int32), ptr(ncl, C.c_int32),
                                 ptr(mod, C.c_double), C.byref(info))
        assert rc == -7
    h.leiden(g, [1.0], 1)                       # the handle still works


def test_ecs_and_ic_against_oracle(h):
    rng = np.random.default_rng(0)
    labs = [rng.integers(0, k, 500) for k in (3, 5, 5, 8, 200)]
    labs.append(labs[1].copy())
    big = np.arange(500) % 130                  # 130 x 200 cells: the global contingency table
    labs.append(big)
    labs.append(np.random.default_rng(1).permutation(500))   # all singletons: 500 x 200 cells
    labs = np.array(labs)
    S = h.label_ecs(labs)
    want = L.ecs_matrix(labs)
    np.testing.assert_allclose(S, want, atol=1e-12, rtol=0)
    assert abs(1 / S.mean() - L.ic(want)) < 1e-12


def test_search_on_ten_cluster_mixture(h):
    from sklearn.metrics import adjusted_rand_score
    X, truth = mixture(500, 10, 10, seed=8)
    g = umap_graph(h, X)
    found, (eg, em), info = h.cluster(g, 2, 12, 10, seed=0)
    assert 10 in found
    f = found[10]
    assert adjusted_rand_score(truth, f["labels"]) >= 0.99
    assert f["ic"] < 1.005
    assert info.n_found == len(found) and info.n_evaluated == len(eg)


def test_clustering_end_to_end_and_repeatable():
    X = make_counts(600, 900, seed=31, K=4, de_prob=0.3, lfc_sd=1.5)
    res = sclens(X, n_perturb=4, verbose=False)
    N = len(res["cell_id"])
    apply_umap(res)
    assert clustering(res, k_max=8, n_trials=8) is res
    for key in ("graph", "n_cluster", "ic", "l_df", "cluster_obj"):
        assert key in res
    assert res["graph"].shape == (N, N) and len(res["ic"]) == len(res["n_cluster"]) >= 1
    df = res["l_df"]
    assert list(df.columns) == ["cell"] + [f"k_{k}" for k in res["n_cluster"]] and len(df) == N
    for k in res["n_cluster"]:
        assert sorted(np.unique(df[f"k_{k}"])) == list(range(1, k + 1))
    first = df.copy()
    clustering(res, k_max=8, n_trials=8)
    assert first.equals(res["l_df"])
    r2 = {"pca_n1": res["pca_n1"], "cell_id": res["cell_id"]}     # no graph: built from the signals
    clustering(r2, k_max=6, n_trials=4)
    assert r2["graph"].shape == (N, N)


def test_clustering_z785_signals():
    z = np.load(os.path.join(ROOT, "tests", "golden", "z785_oracle.npz"))
    sig = z["sig_id"]
    X = (z["signal_evec"][:, sig] * np.sqrt(z["signal_ev"][sig])[None, :]).astype(np.float32)
    res = clustering({"pca_n1": X}, k_max=10, n_trials=10)
    assert len(res["n_cluster"]) >= 1 and (res["ic"] >= 1 - 1e-12).all()
    for k in res["n_cluster"]:
        assert sorted(np.unique(res["l_df"][f"k_{k}"])) == list(range(1, k + 1))
