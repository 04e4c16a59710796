"""Reference restatement of the clustering pieces of sclens_b200/csrc/leiden.cu: the element-centric similarity (ECS)
of two partitions, the inconsistency coefficient (IC) of a set of labelings, the fixed-point exponent of a graph and
one planning step of the resolution search.

scICE (the method behind the reference's clustering step) is not available here: ECS, IC and the search are stated as
this project defines them, recalled from the scICE paper and unverified against its code."""
from __future__ import annotations

import math

import numpy as np


def ecs_pair(a, b):
    """ECS(A, B) from the contingency table: 1/N sum_ab n_ab [1 - 1/2 (n_ab |1/|a| - 1/|b|| + (|a| - n_ab)/|a|
    + (|b| - n_ab)/|b|)], affinity 1/|cluster| inside a cluster."""
    a = np.unique(np.asarray(a), return_inverse=True)[1].ravel()
    b = np.unique(np.asarray(b), return_inverse=True)[1].ravel()
    N = len(a)
    ka, kb = a.max() + 1, b.max() + 1
    n = np.zeros((ka, kb), np.int64)
    np.add.at(n, (a, b), 1)
    A = np.bincount(a, minlength=ka).astype(np.float64)[:, None]
    B = np.bincount(b, minlength=kb).astype(np.float64)[None, :]
    x = n.astype(np.float64)
    t = x * (1.0 - 0.5 * (x * np.abs(1.0 / A - 1.0 / B) + (A - x) / A + (B - x) / B))
    return float(t[n > 0].sum() / N)


def ecs_brute(a, b):
    """ECS by its definition: mean over cells i of 1 - 1/2 sum_j |p^A_ij - p^B_ij|, p_ij = 1/|C(i)| for j in C(i)."""
    a, b = np.asarray(a), np.asarray(b)
    N = len(a)
    s = 0.0
    for i in range(N):
        pa = np.where(a == a[i], 1.0 / np.sum(a == a[i]), 0.0)
        pb = np.where(b == b[i], 1.0 / np.sum(b == b[i]), 0.0)
        s += 1.0 - 0.5 * np.abs(pa - pb).sum()
    return s / N


def ecs_matrix(labels):
    labels = np.asarray(labels)
    T = len(labels)
    S = np.eye(T)
    for i in range(T):
        for j in range(i + 1, T):
            S[i, j] = S[j, i] = ecs_pair(labels[i], labels[j])
    return S


def ic(S):
    """IC = 1 / (p^T S p) with p uniform over the trials (identical labelings have ECS 1, so this equals the weighting
    over distinct labelings)."""
    S = np.asarray(S, dtype=np.float64)
    p = np.full(len(S), 1.0 / len(S))
    return float(1.0 / (p @ S @ p))


def representative(S, counts, k):
    """Of the trials with exactly k clusters, the one with the largest row sum of S, ties to the lowest."""
    rows = np.asarray(S).sum(axis=1)
    rows = np.where(np.asarray(counts) == k, rows, -np.inf)
    return int(np.argmax(rows))


def weight_shift(maxw, nnz):
    """Fixed-point exponent: the largest s <= 32 with (nnz + 1) maxw 2^s <= 2^61 (maxw < 2^e, nnz + 1 <= 2^lg)."""
    _, e = math.frexp(maxw if maxw > 0 else 1.0)
    lg = 0
    while (1 << lg) < nnz + 1:
        lg += 1
    return min(32, 61 - lg - e)


def modal_count(counts):
    """Most frequent cluster count of the trials at one resolution, ties to the smaller count."""
    vals, cnt = np.unique(np.asarray(counts), return_counts=True)
    return int(vals[np.argmax(cnt)])


def start_grid(gamma_lo=0.01, gamma_hi=10.0, n=16):
    l0, l1 = math.log(gamma_lo), math.log(gamma_hi)
    return [math.exp(l0 + i * ((l1 - l0) / (n - 1))) for i in range(n)]


def plan(gammas, modes, k_min, k_max, lo_limit, hi_limit):
    """Next resolutions from the evaluated (gamma, modal count) pairs: gamma_min / 10 while k_min is not bracketed from
    below, gamma_max * 10 while k_max is not bracketed from above (within the limits), and for every k without a
    resolution of modal count k the geometric midpoint of its brackets lo = max{gamma : mode < k} and
    hi = min{gamma > lo : mode > k}.  Ascending, duplicates removed; empty when the search is done."""
    out = []
    if not len(gammas):
        return out
    order = sorted(range(len(gammas)), key=lambda i: gammas[i])
    g = [gammas[i] for i in order]
    m = [modes[i] for i in order]
    if m[0] > k_min and g[0] / 10 >= lo_limit * (1 - 1e-9):
        out.append(g[0] / 10)
    if m[-1] < k_max and g[-1] * 10 <= hi_limit * (1 + 1e-9):
        out.append(g[-1] * 10)
    for k in range(k_min, k_max + 1):
        if k in m:
            continue
        lows = [gi for gi, mi in zip(g, m) if mi < k]
        if not lows:
            continue
        lo = max(lows)
        his = [gi for gi, mi in zip(g, m) if gi > lo and mi > k]
        if not his:
            continue
        hi = min(his)
        if hi <= lo * (1 + 1e-9):
            continue
        out.append(math.sqrt(lo * hi))
    return sorted(set(out))


def search(count_of, k_min=2, k_max=20, gamma_lo=0.01, gamma_hi=10.0, n_grid=16, max_rounds=12, max_widen=4):
    """The search with count_of(gamma) giving the modal count at gamma: returns the evaluated (gamma, mode) pairs."""
    lo_lim, hi_lim = gamma_lo * 10.0 ** -max_widen, gamma_hi * 10.0 ** max_widen
    gs = start_grid(gamma_lo, gamma_hi, n_grid)
    eg, em = [], []
    for rnd in range(max_rounds + 1):
        for x in gs:
            eg.append(x)
            em.append(count_of(x))
        if rnd >= max_rounds:
            break
        gs = plan(eg, em, k_min, k_max, lo_lim, hi_lim)
        if not gs:
            break
    return eg, em


# ---- the device's synchronous Leiden, restated step for step ---------------------------------------------------------
# Every quantity is what leiden.cu computes: integer weights and totals (Python ints), Float64 gains from them with the
# same operation order (Python floats round to nearest and never contract to FMA), the same hashes and tie rules.  One
# trial at a time: a trial's labels do not depend on the rest of the device batch.  Python's math.log and the device's
# double log may differ by an ulp, so a refinement choice between two candidates whose Gumbel-perturbed scores lie within
# ~1e-16 of each other could differ; with 53-bit draws that does not happen on the graphs the tests use.

M64 = (1 << 64) - 1
PHI = 0x9E3779B97F4A7C15
MAX_LEVELS = 256


def mix64s(x):
    x &= M64
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & M64
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & M64
    x ^= x >> 31
    return x


def stream_key(key, stream, word):
    """mix(mix(key ^ phi (stream + 1)) ^ word): umap_stream_key, and step_key with word = it << 48 | level << 32 | sweep."""
    return mix64s(mix64s(key ^ ((PHI * (stream + 1)) & M64)) ^ word)


def copy_key(seed, trial):
    return stream_key(seed & M64, 6, trial)


def step_key(key, stream, it, level, sweep):
    return stream_key(key, stream, (it << 48) | (level << 32) | sweep)


def draw_bits(key, a, b):
    return mix64s(mix64s(key ^ ((a << 32) | b)))


def gumbel(key, a, b):
    u = (float(draw_bits(key, a, b) >> 11) + 0.5) * 1.1102230246251565e-16
    return -math.log(-math.log(u))


def fixed_graph(graph):
    """CSR (scipy, symmetric, sorted columns) -> (rows [(cols, ws)], deg, shift) with ws = max(1, round(w 2^shift))."""
    import scipy.sparse as sp
    g = sp.csr_matrix(graph)
    g.sort_indices()
    maxw = float(g.data.max()) if g.nnz else 0.0
    s = weight_shift(maxw, g.nnz)
    rows = []
    for i in range(g.shape[0]):
        cols = [int(c) for c in g.indices[g.indptr[i]:g.indptr[i + 1]]]
        ws = [max(1, int(round(math.ldexp(float(v), s)))) for v in g.data[g.indptr[i]:g.indptr[i + 1]]]
        rows.append((cols, ws))
    return rows, [sum(ws) for _, ws in rows], s


def _totals(p, deg, n):
    K, cnt = [0] * n, [0] * n
    for v in range(n):
        K[p[v]] += deg[v]
        cnt[p[v]] += 1
    return K, cnt


def _score(w, gk, K, inv2m):
    return float(w) - gk * (float(K) * inv2m)


def _well_connected(ext, gamma, KS, KC, inv2m):
    return float(ext) >= (gamma * float(KS)) * (float(KC - KS) * inv2m)


def _ext(rows, n, comm, ref):
    ext = [0] * n
    for v in range(n):
        a, r = comm[v], ref[v]
        ext[r] += sum(w for x, w in zip(*rows[v]) if x != v and comm[x] == a and ref[x] != r)
    return ext


def canonical(raw):
    """Ids by cluster size, descending, ties by smallest member."""
    first = {}
    for lab in raw:
        if lab not in first:
            first[lab] = len(first)
    sizes = [0] * len(first)
    for lab in raw:
        sizes[first[lab]] += 1
    order = sorted(range(len(sizes)), key=lambda c: -sizes[c])       # stable: ties keep first-appearance order
    rank = {c: r for r, c in enumerate(order)}
    return np.array([rank[first[lab]] for lab in raw], dtype=np.int32)


def leiden(graph, gamma, seed=0, trial=0, max_iterations=10, max_sweeps=64, theta=0.01, stats=None):
    """One trial of the device Leiden: canonical labels (int32, N).  ``stats`` (a dict) receives iterations and levels."""
    rows0, deg0, shift = fixed_graph(graph)
    N = len(rows0)
    two_m = sum(deg0)
    inv2m = 1.0 / float(two_m) if two_m else 0.0
    ctheta = math.ldexp(1.0 / theta, -shift)
    key = copy_key(seed, trial)
    prev, fin = None, None
    max_levels = 0
    its = 0
    for it in range(max_iterations):
        its = it + 1
        if it == 0:
            comm = list(range(N))
        else:
            low = {}
            for v in range(N):
                low.setdefault(fin[v], v)
            comm = [low[fin[v]] for v in range(N)]
        rows, deg, n = rows0, list(deg0), N
        map0 = list(range(N))
        for level in range(MAX_LEVELS):
            max_levels = max(max_levels, level + 1)
            # (1) local moving
            K, csize = _totals(comm, deg, n)
            level_moved = 0
            for sweep in range(max_sweeps):
                moved = 0
                k7 = step_key(key, 7, it, level, sweep)
                for sub in (0, 1):
                    new = list(comm)
                    for v in range(n):
                        if (draw_bits(k7, v, 0) & 1) != sub:
                            continue
                        tab = {}
                        for x, w in zip(*rows[v]):
                            if x != v:
                                tab[comm[x]] = tab.get(comm[x], 0) + w
                        a, kv = comm[v], deg[v]
                        gk = gamma * float(kv)
                        single = csize[a] == 1
                        best, bid = -math.inf, None
                        for c, w in tab.items():
                            if c == a or (single and csize[c] == 1 and c > a):
                                continue
                            s = _score(w, gk, K[c], inv2m)
                            if s > best or (s == best and c < bid):
                                best, bid = s, c
                        stay = _score(tab.get(a, 0), gk, K[a] - kv, inv2m)
                        if bid is not None and best > stay:
                            new[v] = bid
                            moved += 1
                    comm = new
                    K, csize = _totals(comm, deg, n)
                level_moved += moved
                if moved == 0:
                    break
            # (2) refinement
            ref = list(range(n))
            Kr, rsize = list(deg), [1] * n
            ext = _ext(rows, n, comm, ref)
            for sub in (0, 1):
                k8 = step_key(key, 8, it, level, 0)
                k9 = step_key(key, 9, it, level, sub)
                new = list(ref)
                for v in range(n):
                    if (draw_bits(k8, v, 0) & 1) != sub or ref[v] != v or rsize[v] != 1:
                        continue
                    a, kv = comm[v], deg[v]
                    gk = gamma * float(kv)
                    if not _well_connected(ext[v], gamma, kv, K[a], inv2m):
                        continue
                    tab = {}
                    for x, w in zip(*rows[v]):
                        if x != v and comm[x] == a:
                            tab[ref[x]] = tab.get(ref[x], 0) + w
                    best, bid = gumbel(k9, v, v), v
                    for S, w in tab.items():
                        if rsize[S] == 1 and (draw_bits(k8, S, 0) & 1) == sub:
                            continue
                        if not _well_connected(ext[S], gamma, Kr[S], K[a], inv2m):
                            continue
                        gain = _score(w, gk, Kr[S], inv2m)
                        if not gain >= 0.0:
                            continue
                        s = gain * ctheta + gumbel(k9, v, S)
                        if s > best or (s == best and S < bid):
                            best, bid = s, S
                    if bid != v:
                        new[v] = bid
                ref = new
                Kr, rsize = _totals(ref, deg, n)
                ext = _ext(rows, n, comm, ref)
            # (3) stop when the level neither moved nor merged
            live = [s for s in range(n) if rsize[s] > 0]
            if (len(live) == n and level_moved == 0) or level + 1 >= MAX_LEVELS:
                fin = [comm[map0[v]] for v in range(N)]
                break
            # (4) aggregation of the refined subsets
            nid = {s: t for t, s in enumerate(live)}
            nc = len(live)
            cmin = {}
            for s in live:
                cmin[comm[s]] = min(cmin.get(comm[s], nc), nid[s])
            ccomm = [cmin[comm[s]] for s in live]
            cdeg = [Kr[s] for s in live]
            map0 = [nid[ref[map0[v]]] for v in range(N)]
            acc = [dict() for _ in range(nc)]
            for u in range(n):
                t = nid[ref[u]]
                for x, w in zip(*rows[u]):
                    c = nid[ref[x]]
                    acc[t][c] = acc[t].get(c, 0) + w
            rows = [(sorted(d), [d[c] for c in sorted(d)]) for d in acc]
            comm, deg, n = ccomm, cdeg, nc
        labels = canonical(fin)
        if prev is not None and np.array_equal(labels, prev):
            break
        prev = labels
    if stats is not None:
        stats.update(iterations=its, max_levels=max_levels)
    return prev if prev is not None else labels
