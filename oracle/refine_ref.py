"""CPU restatement (numpy, Float64) of the Rayleigh-Ritz refinement of sclens_b200/csrc/refine.cu.

TEST INFRASTRUCTURE ONLY - imported by tests/ (and nothing else).  It restates, step for step, what refine_eigenvalues
computes from an FP32 matrix G and FP32 eigenvectors V (rows), so the device can be checked against it to the last FP32 bit:

  band     H[i][d] = v_i' G v_(i+d) / (|v_i| |v_(i+d)|) on the diagonals d = 0 .. KBAND, in Float64
  links    i and j (j - i <= KBAND) belong to one cluster when |H_ij| > LINK |H_jj - H_ii|; a cluster grows while a member
           links past its end and is cut at MAX_CLUSTER members (the source's loop order, below)
  values   singletons keep their Rayleigh quotient H_ii; a cluster takes the eigenvalues of H restricted to it, band only
  output   sorted, rounded to FP32

The device forms the band from 128 x 128 tiles of V G in Float64 and reduces the tile partials in a fixed order, and solves a
cluster by cyclic Jacobi; the restatement uses one Float64 product and LAPACK.  Both are accurate to a few Float64 ulps of the
block, far below one FP32 ulp of every value the tests use, so the two agree within one FP32 ulp.
"""
import numpy as np

KBAND = 8
MAX_CLUSTER = 96
LINK = 0.02


def band(G, V):
    """Hb[i, d] = v_i' G v_(i+d) / (|v_i| |v_(i+d)|), 0 where i + d >= n (n x (KBAND + 1), Float64)."""
    G64 = np.asarray(G, np.float64)
    V64 = np.asarray(V, np.float64)
    n = V64.shape[0]
    Z = V64 @ G64
    nrm = np.sqrt(np.einsum("ij,ij->i", V64, V64))
    Hb = np.zeros((n, KBAND + 1))
    for d in range(min(KBAND, n - 1) + 1):
        Hb[: n - d, d] = np.einsum("ij,ij->i", Z[: n - d], V64[d:]) / (nrm[: n - d] * nrm[d:])
    return Hb


def clusters(Hb):
    """[(i, hi)] inclusive index ranges in ascending order, exactly as refine_eigenvalues forms them."""
    n = Hb.shape[0]

    def H(i, j):
        return Hb[i, j - i]

    out = []
    i = 0
    while i < n:
        hi = i
        a = i
        while a <= hi and hi - i + 1 < MAX_CLUSTER:
            for b in range(max(a + 1, hi + 1), min(n - 1, a + KBAND) + 1):
                if abs(H(a, b)) > LINK * abs(H(b, b) - H(a, a)):
                    hi = max(hi, b)
            a += 1
        hi = min(hi, i + MAX_CLUSTER - 1)
        out.append((i, hi))
        i = hi + 1
    return out


def refine(G, V, return_parts=False):
    """The refined eigenvalues (FP32, ascending).  return_parts: also the unsorted Float64 values by vector index, the
    clusters, and stats = [clusters of more than one member, size of the largest (1 when there is none)]."""
    Hb = band(G, V)
    n = Hb.shape[0]
    vals = np.empty(n)
    cl = clusters(Hb)
    multi = [(i, hi) for i, hi in cl if hi > i]
    for i, hi in cl:
        if hi == i:
            vals[i] = Hb[i, 0]
            continue
        m = hi - i + 1
        blk = np.zeros((m, m))
        for a in range(m):
            for b in range(a, min(m, a + KBAND + 1)):
                blk[a, b] = blk[b, a] = Hb[i + a, b - a]
        vals[i: hi + 1] = np.linalg.eigvalsh(blk)
    out = np.sort(vals).astype(np.float32)
    if not return_parts:
        return out
    stats = [len(multi), max([hi - i + 1 for i, hi in multi], default=1)]
    return out, vals, cl, stats
