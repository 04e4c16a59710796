"""-m gpu tests of the own eigensolver at the orders production solves (n = 20 000 for the data and null matrices of the
benchmark workloads, 25 000 for the largest), against spectra known by construction.

The matrices are built on the device in Float64: G64 = Q diag(lam) Q' with Q from the QR of a seeded Gaussian, and
G = fp32(G64).  |G - G64|_2 < 1e-7 lam_max (checked by power iteration), so the designed lam is the reference at the
tolerances below, and no Float64 eigh of order 25 000 is needed.  Every check runs in Float64 on the device.

Two code paths run only at these orders, and the cases are chosen (from the SM count) to reach them:
- the stage-2 back-transformation kernel k_q2_apply_h<12>, which apply_q2 picks when a CTA needs more than 8 warps
  (more than 8 x SMs x 16 vectors), next to k_q2_apply_h<8> with and without CTAs that take one extra tile;
- the batch loop of the tridiagonal stage, which builds the vectors in batches of Bmax = 4 GiB / (8 n) when more are asked
  for (all vectors from n > 23 170 on), with and without an index range starting above 0.
The arithmetic of both is restated below as it is in backtrans.cu and tridiag.cu."""
import ctypes as C
import math
import time

import numpy as np
import pytest
import torch

from sclens_b200 import Handle
from sclens_b200._lib import ptr

pytestmark = pytest.mark.gpu


# ---- launch shapes, restated --------------------------------------------------------------------------------------------

def q2_launch(m, sms):
    """apply_q2 (backtrans.cu): 16-vector tiles, one warp each, at most 12 warps per CTA, as few waves as that allows."""
    tiles = (m + 15) // 16
    waves = (tiles + sms * 12 - 1) // (sms * 12)
    grid = min(tiles, sms * waves)
    base, extra = tiles // grid, tiles % grid
    warps = base + (1 if extra else 0)
    return dict(tiles=tiles, grid=grid, base=base, extra=extra, warps=warps, kernel=8 if warps <= 8 else 12)


def tri_batches(n, m):
    """tridiag_eigen (tridiag.cu): vectors in batches of Bmax = max(128, min(m, 4 GiB / (8 n)))."""
    if m == 0:
        return 0
    bmax = max(128, min(m, (4 << 30) // (n * 8)))
    return math.ceil(m / bmax)


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def plan(sms):
    """The solves of this file: (name, n, v0, v1).  n1 = 20 000 unless this SM count would take every tile of an all-vector
    solve in 8 warps; the 25 000 solves batch on any card (Bmax does not depend on it)."""
    n1 = 20000 if q2_launch(20000, sms)["warps"] > 8 else 16 * (8 * sms + sms // 2)
    edge = 16 * 8 * sms
    assert edge <= n1
    e0 = (n1 - edge) // 2
    return [("mp_all", n1, 0, n1), ("mp_range", n1, 3, n1 // 2 + 40), ("mp_values", n1, 0, 0), ("mp_edge", n1, e0, e0 + edge),
            ("mp25_all", 25000, 0, 25000), ("mp25_range", 25000, 1000, 24000), ("graded_all", 19997, 0, 19997)]


def test_cases_reach_both_kernels_and_the_batch_loop():
    sms = sm_count()
    shapes = []
    for name, n, v0, v1 in plan(sms):
        m = v1 - v0
        if m:
            q = q2_launch(m, sms)
            shapes.append((name, q, tri_batches(n, m)))
            print(f"{name}: n={n} vectors [{v0},{v1}) SMs={sms} grid={q['grid']} warps={q['warps']} extra={q['extra']} "
                  f"k_q2_apply_h<{q['kernel']}> tridiagonal batches={tri_batches(n, m)}")
    assert any(q["warps"] <= 8 for _, q, _ in shapes) and any(q["warps"] > 8 for _, q, _ in shapes)
    assert any(q["extra"] == 0 for _, q, _ in shapes) and any(q["extra"] > 0 and q["warps"] <= 8 for _, q, _ in shapes)
    assert any(b >= 2 and name == "mp25_all" for name, _, b in shapes) and any(b >= 2 and name == "mp25_range" for name, _, b in shapes)
    edge = [q for name, q, _ in shapes if name == "mp_edge"][0]
    assert edge["warps"] == 8 and edge["extra"] == 0          # the last shape that takes k_q2_apply_h<8>


# ---- matrices and checks -------------------------------------------------------------------------------------------------

def mp_spectrum(n, ratio, spikes):
    """Marchenko-Pastur bulk (variance 1, aspect ratio `ratio`) at the quantiles (k + 1/2) / n_bulk, plus spikes."""
    a, b = (1 - math.sqrt(ratio)) ** 2, (1 + math.sqrt(ratio)) ** 2
    x = np.linspace(a, b, 2_000_001)
    pdf = np.sqrt(np.maximum((b - x) * (x - a), 0)) / (2 * math.pi * ratio * x)
    cdf = np.concatenate([[0], np.cumsum((pdf[1:] + pdf[:-1]) / 2 * np.diff(x))])
    cdf /= cdf[-1]
    nb = n - len(spikes)
    bulk = np.interp((np.arange(nb) + 0.5) / nb, cdf, x)
    return np.sort(np.concatenate([bulk, spikes]))


SPIKES = np.array([3.0, 3.6, 4.4, 5.5, 7.0, 9.5, 14.0])


def build(n, lam, seed):
    """Host FP32 matrix G = fp32(Q diag(lam) Q') and |G - G64|_2 (20 power iterations), the device freed afterwards."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    Q, _ = torch.linalg.qr(torch.randn(n, n, dtype=torch.float64, device=dev, generator=g))
    G64 = (Q * torch.as_tensor(lam, device=dev)) @ Q.T
    del Q
    G64 = (G64 + G64.T) * 0.5
    G = G64.float()
    E = G.double() - G64
    del G64
    x = torch.randn(n, dtype=torch.float64, device=dev, generator=g)
    for _ in range(20):
        x = E @ x
        x /= torch.linalg.vector_norm(x)
    e2 = float(torch.linalg.vector_norm(E @ x))
    fro = float(torch.linalg.matrix_norm(G.double()))
    del E
    Gh = G.cpu().numpy()
    del G
    torch.cuda.empty_cache()
    assert e2 < 1e-7 * float(np.max(np.abs(lam))), e2
    return Gh, e2, fro


def solve(h, G, v0, v1):
    n = G.shape[0]
    L, V, out = np.empty(n, np.float32), np.empty((max(1, v1 - v0), n), np.float32), np.zeros(6)
    st = np.zeros(8)
    t = time.perf_counter()
    h._ck(h.lib.scl_op_syevd_tri(h.h, n, ptr(G, C.c_float), v0, v1, ptr(L, C.c_float), ptr(V, C.c_float), ptr(out, C.c_double)))
    wall = time.perf_counter() - t
    h._ck(h.lib.scl_debug_last_solve(h.h, ptr(st, C.c_double)))
    print(f"n={n} vectors [{v0},{v1}): {wall:.2f} s with copies; stages (ms) {np.round(st[:5], 1).tolist()}")
    assert out[5] == 0 and st[5] == 1 and st[6] == 0 and st[7] == 0, ("the two-stage path did not produce the result", out, st)
    return L, V[: v1 - v0]


def check_values(L, lam):
    lmax = float(np.max(np.abs(lam)))
    np.testing.assert_allclose(L.astype(np.float64), lam, rtol=2e-5, atol=3e-6 * lmax)


def check_vectors(G, L, V, lam):
    """max |G V - V diag(L)| < 5e-5 max(1, lam_max) and max |V'V - I| < 5e-5, in Float64 on the device (V: rows)."""
    dev = torch.device("cuda")
    lmax = float(np.max(np.abs(lam)))
    Vd = torch.from_numpy(V).to(dev).double()
    Gd = torch.from_numpy(G).to(dev).double()
    R = Vd @ Gd
    del Gd
    R -= torch.from_numpy(L).to(dev).double()[:, None] * Vd
    res = float(R.abs().max())
    del R
    O = Vd @ Vd.T
    O.diagonal().sub_(1.0)
    orth = float(O.abs().max())
    del O, Vd
    torch.cuda.empty_cache()
    assert res < 5e-5 * max(1.0, lmax), res
    assert orth < 5e-5, orth


def check_range(Vr, V, v0):
    """| |cos| - 1 | < 1e-5 between the range solve's vectors and the full solve's."""
    dev = torch.device("cuda")
    a = torch.from_numpy(Vr).to(dev).double()
    b = torch.from_numpy(V[v0: v0 + Vr.shape[0]]).to(dev).double()
    cos = (a * b).sum(dim=1).abs()
    err = float((cos - 1).abs().max())
    del a, b
    torch.cuda.empty_cache()
    assert err < 1e-5, err


@pytest.fixture(scope="module")
def h():
    with Handle() as hh:
        yield hh


@pytest.fixture(scope="module")
def cases():
    return {name: (n, v0, v1) for name, n, v0, v1 in plan(sm_count())}


@pytest.fixture(scope="module")
def mp1(cases):
    n = cases["mp_all"][0]
    lam = mp_spectrum(n, n / 68000, SPIKES)
    G, e2, fro = build(n, lam, 20000)
    return G, lam, fro


def test_mp_20000_all_vectors_range_and_values(h, mp1, cases):
    """All vectors (k_q2_apply_h<12>, 9 warps on 148 SMs; stage 1 over 40 block reflectors), the range of a sparsity-search
    step (k_q2_apply_h<8> with CTAs of one extra tile), values only, and a range of exactly 8 x SMs x 16 vectors (the last
    shape k_q2_apply_h<8> takes, no extra tile).  Range and values-only eigenvalues equal the full solve's bit for bit."""
    G, lam, _ = mp1
    n, _, _ = cases["mp_all"]
    L, V = solve(h, G, 0, n)
    check_values(L, lam)
    check_vectors(G, L, V, lam)
    for name in ("mp_range", "mp_edge"):
        _, v0, v1 = cases[name]
        L2, V2 = solve(h, G, v0, v1)
        np.testing.assert_array_equal(L2, L)
        check_range(V2, V, v0)
        del V2
    L3, _ = solve(h, G, 0, 0)
    np.testing.assert_array_equal(L3, L)


@pytest.mark.parametrize("e", [-20, 20])
def test_mp_20000_scaled_values(h, mp1, e):
    """The same matrix times 2^-20 and 2^20 (exact in FP32): its Frobenius norm leaves [n / 8192, 1024] on both sides, so
    stage 1 multiplies in three-term TF32 instead of split binary16."""
    G, lam, fro = mp1
    n = G.shape[0]
    Gs = np.ascontiguousarray(G * np.float32(2.0 ** e))
    fro *= 2.0 ** e
    assert not (n / 8192 <= fro <= 1024), fro
    L, _ = solve(h, Gs, 0, 0)
    check_values(L, lam * 2.0 ** e)


def test_mp_25000_batched_tridiagonal_vectors(h, cases):
    """n = 25 000: all vectors (two batches of the tridiagonal stage, 21 474 + 3 526, and k_q2_apply_h<12> with 11 warps on
    148 SMs) and the range [1000, 24000) (two batches with v0 > 0)."""
    n, _, _ = cases["mp25_all"]
    lam = mp_spectrum(n, n / 68000, SPIKES)
    G, e2, fro = build(n, lam, 25000)
    L, V = solve(h, G, 0, n)
    check_values(L, lam)
    check_vectors(G, L, V, lam)
    _, v0, v1 = cases["mp25_range"]
    L2, V2 = solve(h, G, v0, v1)
    np.testing.assert_array_equal(L2, L)
    check_range(V2, V, v0)
    check_vectors(G, L[v0:v1], V2, lam)


def test_graded_19997(h, cases):
    """n = 19 997 (not a multiple of 4 or 64: the padded copy and a short last panel) with eigenvalues graded over six
    decades: the Frobenius norm is above 1024, so stage 1 runs in three-term TF32 at scale."""
    n, _, _ = cases["graded_all"]
    lam = np.logspace(-3, 3, n)
    G, e2, fro = build(n, lam, 19997)
    assert not (n / 8192 <= fro <= 1024), fro
    L, V = solve(h, G, 0, n)
    check_values(L, lam)
    check_vectors(G, L, V, lam)
