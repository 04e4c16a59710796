"""-m gpu parity of apply_umap! (:863-873) on the device (scl_op_knn / scl_op_umap) against the oracle's restatement
(oracle/umap_ref.py): kNN, fuzzy graph, spectral / random start, the synchronous layout, determinism, quality, and the
end-to-end call on a sclens() result."""
import os

import numpy as np
import pytest
from scipy.linalg import subspace_angles

from oracle import umap_ref as U
from sclens_b200 import Handle, apply_umap, sclens
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


def z785_pca_n1():
    z = np.load(os.path.join(ROOT, "tests", "golden", "z785_oracle.npz"))
    sig = z["sig_id"]
    return (z["signal_evec"][:, sig] * np.sqrt(z["signal_ev"][sig])[None, :]).astype(np.float32)


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
@pytest.mark.parametrize("N,d,k", [(1001, 1, 2), (777, 40, 15), (2051, 7, 64), (300, 10, 15)])
def test_knn_matches_oracle(h, metric, N, d, k):
    rng = np.random.default_rng(N + d + k)
    X = rng.standard_normal((N, d)).astype(np.float32)
    X[5] = X[17]                        # duplicate points
    X[40:43] = X[41]
    if metric == "cosine":
        X[60] = 0                       # a zero row: distance 1 from everything
    idx, dist = h.knn(X, k, metric)
    idx2, dist2 = h.knn(X, k, metric)
    assert idx.tobytes() == idx2.tobytes() and dist.tobytes() == dist2.tobytes()
    widx, wdist = U.knn(X.astype(np.float64), k + 1, metric)
    np.testing.assert_allclose(dist, wdist[:, :k], rtol=1e-5, atol=1e-6)
    gap = (wdist[:, k] - wdist[:, k - 1]) > 1e-6 * np.maximum(wdist[:, k], 1e-30)
    for i in np.nonzero(gap)[0]:
        assert set(idx[i]) == set(widx[i, :k]), i
    assert (idx != np.arange(N)[:, None]).all()
    assert (np.diff(dist, axis=1) >= 0).all()


@pytest.mark.parametrize("metric", ["euclidean", "cosine"])
def test_graph_matches_oracle_on_device_knn(h, metric):
    X, _ = mixture(250, 4, 6, seed=3)
    h.umap(X, 15, 2, metric=metric, n_epochs=0, init="random")
    g = h.umap_graph()
    idx, dist = h.umap_knn()
    want = U.graph_from_knn(idx, dist, 15)
    np.testing.assert_array_equal(g.indptr, want.indptr)
    np.testing.assert_array_equal(g.indices, want.indices)
    np.testing.assert_allclose(g.data, want.data, rtol=1e-5)
    assert abs(g - g.T).max() == 0


def ritz(g, P):
    deg = np.asarray(g.sum(1)).ravel()
    dinv = 1 / np.sqrt(deg)
    Q, _ = np.linalg.qr(P.astype(np.float64))
    S = (g.multiply(dinv[:, None]).multiply(dinv[None, :])).tocsr()
    return np.sort(np.linalg.eigvalsh(Q.T @ (S @ Q)))[::-1]


@pytest.mark.parametrize("n_clusters,sep", [(3, 2.0), (3, 200.0)])   # connected graph (gap 0.11 below the wanted pair); three components
def test_spectral_start_matches_eigsh(h, n_clusters, sep):
    X, _ = mixture(300, n_clusters, 5, seed=4, sep=sep)
    P, info = h.umap(X, 15, 2, metric="euclidean", n_epochs=0)
    assert info.init_fallback == 0 and info.spectral_iters >= 1
    g = h.umap_graph()
    vals, V = U.spectral_vectors(g, 2)
    assert np.max(subspace_angles(P.astype(np.float64), V)) <= 1e-3
    np.testing.assert_allclose(ritz(g, P), vals, atol=1e-4)
    assert abs(P.max() - 10) < 1e-2


def test_spectral_fallback_and_random_start(h):
    X, _ = mixture(200, 3, 5, seed=5)
    P, info = h.umap(X, 15, 2, metric="euclidean", n_epochs=0, spectral_maxiter=1, seed=9)
    assert info.init_fallback == 1
    np.testing.assert_array_equal(P, U.random_start(len(X), 2, 9))
    P2, info2 = h.umap(X, 15, 3, n_epochs=0, init="random", seed=11)
    assert info2.init_fallback == 0
    np.testing.assert_array_equal(P2, U.random_start(len(X), 3, 11))


@pytest.mark.parametrize("epochs", [1, 5])
def test_layout_matches_layout_sync(h, epochs):
    """The repulsive step grows as 1 / (0.001 + d^2), so Float32 rounding is amplified between near-coincident points:
    the start is a spread-out grid with jitter, not uniform draws, to keep such pairs out of a parity test."""
    X, _ = mixture(120, 5, 6, seed=6)
    side = int(np.ceil(np.sqrt(len(X))))
    grid = np.stack(np.meshgrid(np.arange(side), np.arange(side)), -1).reshape(-1, 2)[:len(X)]
    P0 = (grid * (20.0 / side) - 10.0 + 0.1 * U.random_start(len(X), 2, 1) / 10).astype(np.float32)
    P, info = h.umap(X, 15, 2, n_epochs=epochs, init_embedding=P0, seed=3)
    g = h.umap_graph()
    want = U.layout_sync(g, P0, epochs, info.a, info.b, seed=3)
    extent = np.ptp(want, axis=0).max()
    assert np.abs(P - want).max() <= 1e-4 * extent


def test_full_run_is_bitwise_deterministic(h):
    X, _ = mixture(500, 6, 7, seed=7)
    P1, _ = h.umap(X, 15, 2, seed=5)
    P2, _ = h.umap(X, 15, 2, seed=5)
    assert P1.tobytes() == P2.tobytes()
    P3, _ = h.umap(X, 15, 2, seed=6)
    assert P3.tobytes() != P1.tobytes()


def test_quality_on_ten_cluster_mixture(h):
    from sklearn.manifold import trustworthiness
    from sklearn.neighbors import KNeighborsClassifier
    X, lab = mixture(2000, 10, 10, seed=8)
    P, info = h.umap(X, 15, 2, metric="euclidean")
    assert info.init_fallback == 0
    rng = np.random.default_rng(0)
    sub = rng.choice(len(X), 4000, replace=False)
    assert trustworthiness(X[sub], P[sub], n_neighbors=15) >= 0.95
    knn = KNeighborsClassifier(n_neighbors=6).fit(P, lab)
    nb = knn.kneighbors(P, return_distance=False)[:, 1:]
    assert (lab[nb] == lab[:, None]).mean() >= 0.98


def test_z785_quality_against_sequential_layout(h):
    from sklearn.manifold import trustworthiness
    X = z785_pca_n1()
    P, info = h.umap(X, 15, 2, metric="cosine")
    g = h.umap_graph()
    _, V = U.spectral_vectors(g, 2)
    seq = U.layout_sequential(g, V * (10.0 / V.max()), 300, info.a, info.b, seed=0)
    t_dev = trustworthiness(X, P, n_neighbors=15, metric="cosine")
    t_seq = trustworthiness(X, seq, n_neighbors=15, metric="cosine")
    assert t_dev >= t_seq - 0.02, (t_dev, t_seq)


def test_apply_umap_end_to_end():
    X = make_counts(600, 900, seed=31, K=4, de_prob=0.3, lfc_sd=1.5)
    res = sclens(X, n_perturb=4, verbose=False)
    N = len(res["cell_id"])
    assert apply_umap(res) is res
    assert res["umap"].shape == (N, 2) and np.isfinite(res["umap"]).all()
    obj = res["umap_obj"]
    assert obj["graph"].shape == (N, N) and obj["knns"].shape == (N, 15) and obj["dists"].shape == (N, 15)
    assert abs(obj["a"] - 1.57694) < 1e-4
    r2 = dict(res)
    r2["pca_n1"] = res["pca_n1"].iloc[:, :1]          # only the "cell" column left: the :pca path
    apply_umap(r2, seed=1)
    assert r2["umap"].shape == (N, 2)
    want = apply_umap({"pca": res["pca"]}, seed=1)["umap"]
    np.testing.assert_array_equal(r2["umap"], want)
