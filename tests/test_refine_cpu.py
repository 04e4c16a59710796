"""CPU check of oracle/refine_ref.py, the restatement of the Float64 Rayleigh-Ritz refinement (sclens_b200/csrc/refine.cu)
that the device is compared with bit for bit in tests/test_refine_calibration_gpu.py: the band of H, the linking rule with
its cap, and what the refined values are on matrices whose spectrum is known."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import refine_ref as rr  # noqa: E402


def designed(n, lam, seed):
    Q = np.linalg.qr(np.random.default_rng(seed).standard_normal((n, n)))[0]
    return (Q * lam) @ Q.T, Q.T.copy()          # G, exact eigenvectors as rows


def rotate_rows(V, idx, seed):
    """Mix the rows idx by a random orthogonal matrix (an arbitrary basis of their span)."""
    R = np.linalg.qr(np.random.default_rng(seed).standard_normal((len(idx), len(idx))))[0]
    V = V.copy()
    V[idx] = R @ V[idx]
    return V


def test_band_is_the_normalised_band_of_v_g_vt():
    rng = np.random.default_rng(1)
    n = 40
    G = rng.standard_normal((n, n))
    G = G + G.T
    V = rng.standard_normal((n, n))
    Hb = rr.band(G, V)
    nrm = np.linalg.norm(V, axis=1)
    H = (V @ G @ V.T) / np.outer(nrm, nrm)
    for d in range(rr.KBAND + 1):
        np.testing.assert_allclose(Hb[: n - d, d], np.diag(H, d), rtol=1e-12, atol=1e-12)
        assert np.all(Hb[n - d:, d] == 0)


def test_exact_eigenvectors_are_singletons_with_their_eigenvalues():
    n = 300
    lam = np.linspace(0.5, 3.0, n)
    G, V = designed(n, lam, 2)
    out, vals, cl, stats = rr.refine(G, V * np.linspace(0.5, 2.0, n)[:, None], return_parts=True)
    assert stats == [0, 1] and len(cl) == n
    np.testing.assert_allclose(vals, lam, rtol=0, atol=1e-13)
    np.testing.assert_array_equal(out, lam.astype(np.float32))


def test_rotated_pair_is_recovered():
    """DESIGN's case: two eigenvalues 4e-5 apart whose vectors came out rotated by 43 degrees: the Rayleigh quotients are off
    by sin^2(43) x 4e-5, the 2 x 2 Ritz values are exact."""
    n, k = 200, 77
    lam = np.linspace(0.5, 3.0, n)
    lam[k + 1] = lam[k] + 4e-5
    G, V = designed(n, lam, 3)
    t = np.deg2rad(43.0)
    V[[k, k + 1]] = np.array([[np.cos(t), np.sin(t)], [-np.sin(t), np.cos(t)]]) @ V[[k, k + 1]]
    out, vals, cl, stats = rr.refine(G, V, return_parts=True)
    assert stats == [1, 2] and (k, k + 1) in cl
    Hb = rr.band(G, V)
    assert abs(Hb[k, 0] - lam[k]) > 1e-5                   # the plain Rayleigh quotient is wrong
    np.testing.assert_allclose(vals[[k, k + 1]], lam[[k, k + 1]], rtol=0, atol=1e-13)


@pytest.mark.parametrize("run,want", [(20, [1, 20]), (150, [2, rr.MAX_CLUSTER])])
def test_runs_longer_than_the_band_and_the_cap(run, want):
    """A run of near-equal eigenvalues with an arbitrary basis: one chain longer than the band (20), or a run the 96-member
    cap splits (150 -> 96 + 54).  Either way every Ritz value lies inside the run's spread, and the trace of each block is
    kept (the band drops off-diagonal entries only)."""
    n, k = 400, 120
    lam = np.linspace(0.5, 3.0, n)
    lam[k: k + run] = lam[k] + 1e-6 * np.arange(run)
    lam = np.sort(lam)
    G, V = designed(n, lam, 4)
    V = rotate_rows(V, np.arange(k, k + run), 5)
    out, vals, cl, stats = rr.refine(G, V, return_parts=True)
    assert stats == want
    if run == 150:
        assert (k, k + 95) in cl and (k + 96, k + 149) in cl
    else:
        assert (k, k + run - 1) in cl
    lo, hi = lam[k], lam[k + run - 1]
    assert np.all(vals[k: k + run] > lo - 1e-12) and np.all(vals[k: k + run] < hi + 1e-12)
    for i, j in cl:
        Hb = rr.band(G, V)
        np.testing.assert_allclose(vals[i: j + 1].sum(), Hb[i: j + 1, 0].sum(), rtol=1e-14)
    rest = np.setdiff1d(np.arange(n), np.arange(k, k + run))
    np.testing.assert_allclose(vals[rest], lam[rest], rtol=0, atol=1e-13)


def test_loop_order_matches_a_plain_restatement():
    """The linking loop against a second, literal transcription of the C++ loop on random bands (cap included)."""
    rng = np.random.default_rng(7)
    n = 500
    Hb = np.zeros((n, rr.KBAND + 1))
    Hb[:, 0] = np.cumsum(rng.uniform(0, 1, n))
    Hb[:, 1:] = rng.standard_normal((n, rr.KBAND)) * np.where(rng.uniform(size=(n, rr.KBAND)) < 0.3, 1.0, 1e-6)

    def literal(Hb):
        res, i = [], 0
        while i < n:
            hi, a = i, i
            while True:
                if not (a <= hi and hi - i + 1 < rr.MAX_CLUSTER):
                    break
                b = max(a + 1, hi + 1)
                end = min(n - 1, a + rr.KBAND)
                while b <= end:
                    if abs(Hb[a, b - a]) > rr.LINK * abs(Hb[b, 0] - Hb[a, 0]):
                        hi = max(hi, b)
                    b += 1
                a += 1
            hi = min(hi, i + rr.MAX_CLUSTER - 1)
            res.append((i, hi))
            i = hi + 1
        return res

    got = rr.clusters(Hb)
    assert got == literal(Hb)
    assert max(j - i + 1 for i, j in got) == rr.MAX_CLUSTER      # the cap was reached
