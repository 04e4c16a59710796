"""apply_umap! (src/scLENS.jl:863-873) and UMAP.jl 0.1.11 UMAP_, restated in numpy / scipy.

Neither UMAP.jl nor the reference runs in this repository's test environment: every function below restates the
maintainers' recollection of UMAP.jl, not checked code, and is the contract the device implementation
(sclens_b200/csrc/umap.cu) is tested against.  Two deliberate deviations from UMAP.jl (DESIGN.md): exact kNN at every N
(UMAP.jl uses NN-descent from 4096 points on), and a synchronous epoch (``layout_sync``) instead of UMAP.jl's
edge-by-edge updates (``layout_sequential``, kept only to judge that deviation).
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp


# ---- counter-based draws (the device's, bit for bit) -------------------------------------------------------------------
def mix64(x):
    """splitmix64 finaliser on uint64 arrays / scalars (wrapping arithmetic)."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint64(30))
        x = x * np.uint64(0xBF58476D1CE4E5B9)
        x = x ^ (x >> np.uint64(27))
        x = x * np.uint64(0x94D049BB133111EB)
        x = x ^ (x >> np.uint64(31))
    return x


def stream_key(seed, stream, epoch):
    """Key of one (seed, stream, epoch): streams 1 = edge firing, 2 = negative samples, 3 = random start,
    4 = spectral-start noise, 5 = start block of the spectral iteration."""
    with np.errstate(over="ignore"):
        s = np.uint64(seed & 0xFFFFFFFFFFFFFFFF) ^ (np.uint64(0x9E3779B97F4A7C15) * np.uint64(stream + 1))
    return mix64(mix64(s) ^ np.uint64(epoch))


def draw_bits(key, vertex, slot):
    v = np.asarray(vertex, dtype=np.uint64)
    s = np.asarray(slot, dtype=np.uint64)
    return mix64(mix64(np.uint64(key) ^ ((v << np.uint64(32)) | s)))


def draw_unit(key, vertex, slot):
    """Uniform in [0, 1) with 24 bits (exact in Float32)."""
    return (draw_bits(key, vertex, slot) >> np.uint64(40)).astype(np.float64) / 16777216.0


def draw_index(key, vertex, slot, n):
    """Uniform vertex in [0, n): high 32 bits scaled by n."""
    return (((draw_bits(key, vertex, slot) >> np.uint64(32)) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


# ---- kNN --------------------------------------------------------------------------------------------------------------
def knn(X, k, metric="cosine"):
    """Exact kNN in Float64, self excluded, ascending (distance, index).  Cosine: 1/2 |x^ - y^|^2 of unit rows (= 1 - cos);
    a zero row is at distance 1 from everything.  Returns (idx, dist), N x k."""
    X = np.asarray(X, dtype=np.float64)
    N = X.shape[0]
    zero = None
    if metric == "cosine":
        nrm = np.linalg.norm(X, axis=1)
        zero = nrm == 0
        X = X / np.where(zero, 1.0, nrm)[:, None]
    sq = (X * X).sum(1)
    idx = np.empty((N, k), np.int64)
    dist = np.empty((N, k))
    m = min(k + 8, N - 1)
    for b0 in range(0, N, 512):
        rows = np.arange(b0, min(N, b0 + 512))
        D = np.maximum(sq[rows, None] + sq[None, :] - 2 * X[rows] @ X.T, 0)
        D[np.arange(len(rows)), rows] = np.inf
        cand = np.argpartition(D, m - 1, axis=1)[:, :m]            # then exact distances of the candidates
        d2 = ((X[cand] - X[rows, None, :]) ** 2).sum(-1)
        dd = 0.5 * d2 if metric == "cosine" else np.sqrt(d2)
        if zero is not None and zero.any():
            dd = np.where(zero[rows][:, None] | zero[cand], 1.0, dd)
        order = np.lexsort((cand, dd), axis=1)[:, :k]
        idx[rows] = np.take_along_axis(cand, order, axis=1)
        dist[rows] = np.take_along_axis(dd, order, axis=1)
    return idx, dist


# ---- fuzzy simplicial set -----------------------------------------------------------------------------------------------
def smooth_knn_dists(dists, k, local_connectivity=1.0, niter=64, ktol=1e-5):
    """UMAP.jl smooth_knn_dists (recalled): rho_i = the local_connectivity-th non-zero distance (interpolated), sigma_i by
    bisection of sum_j exp(-max(0, d_ij - rho_i) / sigma) = log2(k) (64 steps, tolerance 1e-5).  Float64."""
    dists = np.asarray(dists, dtype=np.float64)
    N = dists.shape[0]
    rho, sigma = np.zeros(N), np.zeros(N)
    target = np.log2(k)
    index = int(np.floor(local_connectivity))
    interp = local_connectivity - index
    for i in range(N):
        d = dists[i]
        nz = d[d > 0]
        if len(nz) >= local_connectivity:
            if index > 0:
                rho[i] = nz[index - 1]
                if interp > 1e-5:
                    rho[i] += interp * (nz[index] - nz[index - 1])
            else:
                rho[i] = interp * nz[0]
        elif len(nz) > 0:
            rho[i] = nz.max()
        lo, mid, hi = 0.0, 1.0, np.inf
        for _ in range(niter):
            psum = np.exp(-np.maximum(d - rho[i], 0.0) / mid).sum()
            if abs(psum - target) < ktol:
                break
            if psum > target:
                hi = mid
                mid = (lo + hi) / 2
            else:
                lo = mid
                mid = mid * 2 if np.isinf(hi) else (lo + hi) / 2
        sigma[i] = mid
    return rho, sigma


def memberships(dists, rho, sigma):
    """w_ij = exp(-max(0, d_ij - rho_i) / sigma_i)."""
    return np.exp(-np.maximum(np.asarray(dists, np.float64) - rho[:, None], 0.0) / sigma[:, None])


def fuzzy_union(knn_idx, w):
    """A + A^T - A o A^T as CSR with sorted columns; the pattern is the union of the kNN edges and their reverses
    (an edge whose membership underflows stays stored).  Values Float64."""
    N, k = knn_idx.shape
    rows = np.repeat(np.arange(N), k)
    cols = np.asarray(knn_idx).ravel()
    A = sp.csr_matrix((np.asarray(w).ravel(), (rows, cols)), shape=(N, N))
    pat = sp.csr_matrix((np.ones(N * k), (rows, cols)), shape=(N, N))
    pat = ((pat + pat.T) > 0).astype(np.float64).tocsr()
    pat.sort_indices()
    r, c = np.repeat(np.arange(N), np.diff(pat.indptr)), pat.indices
    a = np.asarray(A[r, c]).ravel()
    b = np.asarray(A[c, r]).ravel()
    return sp.csr_matrix((a + b - a * b, pat.indices.copy(), pat.indptr.copy()), shape=(N, N))


def fit_ab(min_dist, spread=1.0):
    """UMAP.jl fit_ab (recalled): least squares of 1 / (1 + a x^(2b)) against exp(-(x - min_dist) / spread) (1 below
    min_dist) on 300 points of [0, 3 spread], from (1, 1)."""
    from scipy.optimize import curve_fit
    xs = np.linspace(0.0, 3.0 * spread, 300)
    ys = np.where(xs >= min_dist, np.exp(-(xs - min_dist) / spread), 1.0)
    (a, b), _ = curve_fit(lambda x, a, b: 1.0 / (1.0 + a * x ** (2 * b)), xs, ys, p0=[1.0, 1.0], xtol=1e-14, ftol=1e-14,
                          gtol=1e-14, maxfev=100000)
    return float(a), float(b)


# ---- starts -----------------------------------------------------------------------------------------------------------
def spectral_vectors(graph, nc):
    """Eigenvectors 2..nc+1 of I - D^-1/2 A D^-1/2 (= the top nc + 1 of S = D^-1/2 A D^-1/2 without the first) and their
    eigenvalues of S, by scipy eigsh.  Returns (values, vectors N x nc)."""
    from scipy.sparse.linalg import eigsh
    deg = np.asarray(graph.sum(axis=1)).ravel()
    dinv = np.where(deg > 0, 1.0 / np.sqrt(np.where(deg > 0, deg, 1.0)), 0.0)
    S = sp.diags(dinv) @ graph.astype(np.float64) @ sp.diags(dinv)
    vals, vecs = eigsh(S, k=nc + 1, which="LA", tol=1e-10)
    # the first vector is D^1/2 1 / |.|; with a repeated eigenvalue 1 (disconnected graph) eigsh returns any basis of the
    # eigenspace, so project that vector out explicitly and keep a basis of what is left
    v0 = np.sqrt(deg) / np.sqrt(deg.sum())
    W = vecs - np.outer(v0, v0 @ vecs)
    U_, _, _ = np.linalg.svd(W, full_matrices=False)
    V = U_[:, :nc]
    w, R = np.linalg.eigh(V.T @ (S @ V))
    order = np.argsort(-w)
    return w[order], V @ R[:, order]


def random_start(N, nc, seed):
    """Uniform in [-10, 10] per coordinate (stream 3), Float32."""
    i = np.repeat(np.arange(N), nc)
    c = np.tile(np.arange(nc), N)
    u = draw_unit(stream_key(seed, 3, 0), i, c)
    return (u * 20.0 - 10.0).astype(np.float32).reshape(N, nc)


# ---- layouts ----------------------------------------------------------------------------------------------------------
def _attr_delta(sd, a, b):
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(sd > 0, (-2.0 * a * b * np.power(sd, b - 1.0)) / (1.0 + a * np.power(sd, b)), 0.0)


def layout_sync(graph, P0, n_epochs, a, b, seed, learning_rate=1.0, gamma=1.0, neg_rate=5):
    """The device's synchronous epoch restated: every epoch reads the positions of the epoch's start.  Vertex i gathers,
    for each stored edge e = (i, j) of its row (slot s = e - rowptr[i]):
      * when e fires (draw(stream 1, epoch, i, s) <= p_e): the attractive step clip(delta (x_i - x_j), +-4) and
        neg_rate repulsive steps against k = draw(stream 2, epoch, i, s * neg_rate + t) (skipped when k == i; grad 4 per
        coordinate at distance 0);
      * when the reverse edge (j, i) fires: -clip(delta (x_j - x_i), +-4) (UMAP.jl's move_ref).
    x_i += alpha * sum of the steps, alpha = lr (1 - e / n_epochs)."""
    g = graph.tocsr()
    g.sort_indices()
    N = g.shape[0]
    ptr, col = g.indptr.astype(np.int64), g.indices.astype(np.int64)
    p = g.data.astype(np.float32).astype(np.float64)
    row = np.repeat(np.arange(N), np.diff(ptr))
    slot = np.arange(len(col)) - ptr[row]
    key_rev = col.astype(np.int64) * N + row          # position of (j, i): search the sorted (row, col) keys
    rev = np.searchsorted(row * N + col, key_rev)
    P = np.asarray(P0, dtype=np.float64).copy()
    for e in range(n_epochs):
        alpha = np.float32(learning_rate * (1.0 - e / n_epochs))
        kf, kn = stream_key(seed, 1, e), stream_key(seed, 2, e)
        fired = draw_unit(kf, row, slot) <= p
        f2 = fired[rev]
        G = np.zeros_like(P)
        diff = P[row] - P[col]
        sd = (diff ** 2).sum(1)
        dl = _attr_delta(sd, a, b)
        att = np.clip(dl[:, None] * diff, -4, 4)
        np.add.at(G, row[fired], att[fired])
        np.add.at(G, row[f2], -np.clip(dl[f2, None] * (-diff[f2]), -4, 4))
        fe = np.nonzero(fired)[0]
        for t in range(neg_rate):
            i = row[fe]
            kk = draw_index(kn, i, slot[fe] * neg_rate + t, N)
            keep = kk != i
            i, kk = i[keep], kk[keep]
            dn = P[i] - P[kk]
            sk = (dn ** 2).sum(1)
            with np.errstate(divide="ignore", invalid="ignore"):
                rep = np.where(sk > 0, (2.0 * gamma * b) / ((1e-3 + sk) * (1.0 + a * np.power(sk, b))), 0.0)
            step = np.where(rep[:, None] > 0, np.clip(rep[:, None] * dn, -4, 4), 4.0)
            np.add.at(G, i, step)
        P = (P + float(alpha) * G).astype(np.float32).astype(np.float64)   # positions are stored in Float32
    return P


def layout_sequential(graph, P0, n_epochs, a, b, seed, learning_rate=1.0, gamma=1.0, neg_rate=5):
    """UMAP.jl optimize_embedding (recalled), edge by edge in CSR order with immediate updates and move_ref; draws from
    numpy (the order of draws differs from the device's anyway)."""
    g = graph.tocsr()
    g.sort_indices()
    N = g.shape[0]
    ptr, col, p = g.indptr, g.indices, g.data.astype(np.float64)
    P = [list(map(float, r)) for r in np.asarray(P0, dtype=np.float64)]
    nc = len(P[0])
    rng = np.random.default_rng(seed)
    alpha = learning_rate
    for e in range(n_epochs):
        u = rng.random(len(col))
        negs = rng.integers(0, N, size=(len(col), neg_rate))
        for i in range(N):
            xi = P[i]
            for ind in range(ptr[i], ptr[i + 1]):
                if u[ind] > p[ind]:
                    continue
                j = col[ind]
                xj = P[j]
                sd = sum((xi[d] - xj[d]) ** 2 for d in range(nc))
                delta = (-2.0 * a * b * sd ** (b - 1.0)) / (1.0 + a * sd ** b) if sd > 0 else 0.0
                for d in range(nc):
                    gr = min(4.0, max(-4.0, delta * (xi[d] - xj[d])))
                    xi[d] += alpha * gr
                    xj[d] -= alpha * gr
                for kk in negs[ind]:
                    if kk == i:
                        continue
                    xk = P[kk]
                    sk = sum((xi[d] - xk[d]) ** 2 for d in range(nc))
                    dn = (2.0 * gamma * b) / ((1e-3 + sk) * (1.0 + a * sk ** b)) if sk > 0 else 0.0
                    for d in range(nc):
                        gr = min(4.0, max(-4.0, dn * (xi[d] - xk[d]))) if dn > 0 else 4.0
                        xi[d] += alpha * gr
        alpha = learning_rate * (1.0 - (e + 1) / n_epochs)
    return np.array(P)


def graph_from_knn(idx, dist, k, local_connectivity=1.0):
    """smooth_knn_dists + memberships + fuzzy union of a given kNN."""
    rho, sigma = smooth_knn_dists(dist, k, local_connectivity)
    return fuzzy_union(np.asarray(idx), memberships(dist, rho, sigma))
