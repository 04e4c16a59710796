"""-m gpu tests of the tcgen05 GEMM (gemm_umma.cu) through scl_debug_gemm, entry by entry and bit for bit.

Operands are small integers (hi, lo in {-3 .. 3}).  Every product and every partial sum, split mode and split-K included, is
then an integer below 2^24, so the tensor core's truncation, the promotion of accumulation chunks and the reduction of
split-K partials are exact, and the only rounding left is the one FP32 multiply by alpha (or by the reduce scale):
expected = float32(S) * float32(alpha), with S = hi hi' (+ hi lo' + lo hi' in split mode, and no lo lo' term).  S is
formed on the device with FP32 matrix products, exact for these integers (checked against Float64 once).

Every case also guards what the kernel must not touch or read: binary16 NaN in the pad columns between K and the leading
dimension and in rows after each operand (a TMA read of them turns the result into NaN), and NaN around the result - spare
columns (ldc larger than the row, +8 where the caller's ldc is the row length) and a tail - that must survive.  The launch
the hook reports must equal the restatement (oracle/gemm_ref.py) at the device's SM count.

The cases: every production call site at its 68 000 x 20 000 shape and configuration, the sharded Gram's operand window,
edges of m, n, K and the syrk triangle, the empty split-K partition, and - the one thing integer operands cannot see - that
chunked accumulation bounds the tensor core's truncation bias."""
import ctypes as C
import os
import sys
import zlib

import numpy as np
import pytest

from sclens_b200 import Handle

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import gemm_ref as gr  # noqa: E402

pytestmark = pytest.mark.gpu

GUARD_ROWS = 256
GUARD_TAIL = 4096
NAN16 = 0x7E00


@pytest.fixture(scope="module")
def torch():
    import torch as t
    assert t.cuda.is_available()
    return t


@pytest.fixture(scope="module")
def h():
    with Handle() as hh:
        yield hh


@pytest.fixture(scope="module")
def sms(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


def nan16(torch, rows, ld):
    return torch.full((rows, ld), NAN16, dtype=torch.int16, device="cuda").view(torch.float16)


def int_operand(torch, gen, rows, K, ld, split):
    """(hi, lo) binary16 [rows + GUARD_ROWS, ld]: integers in [:rows, :K], NaN in the pad columns and the guard rows."""
    out = []
    for _ in range(2 if split else 1):
        x = nan16(torch, rows + GUARD_ROWS, ld)
        x[:rows, :K] = torch.randint(-3, 4, (rows, K), generator=gen, device="cuda", dtype=torch.int8).half()
        out.append(x)
    return out[0], (out[1] if split else None)


def exact_product(torch, A, B, m, n, K):
    """S = hi_a hi_b' (+ hi_a lo_b' + lo_a hi_b'): FP32 products of integers below 2^24, exact."""
    ah, bh = A[0][:m, :K].float(), B[0][:n, :K].float()
    if A[1] is None:
        return ah @ bh.T
    S = ah @ (bh + B[1][:n, :K].float()).T
    S += A[1][:m, :K].float() @ bh.T
    return S


def ptr(x):
    return None if x is None else x.data_ptr()


def call(h, m, n, K, A, lda, B, ldb, alpha, epi, syrk, splits, split_stride, chunk_kb, cg, Cbuf, ldc, red=None, red_scale=1.0):
    launch = np.zeros(7, np.int32)
    rc = h.lib.scl_debug_gemm(h.h, m, n, K, ptr(A[0]), ptr(A[1]), lda, ptr(B[0]), ptr(B[1]), ldb, float(alpha), epi, int(syrk),
                              splits, split_stride, chunk_kb, cg, ptr(Cbuf), ldc, ptr(red), float(red_scale),
                              launch.ctypes.data_as(C.POINTER(C.c_int32)))
    return rc, [int(v) for v in launch]


def run_case(torch, h, sms, c, cg, seed, A=None, a_off=0):
    """Runs one case (a dict as gemm_ref builds them) and checks every entry, the guards and the reported launch.
    A / a_off: a prepared operand and an element offset into it (the sharded Gram's window)."""
    torch.cuda.synchronize()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    m, n, K, split, epi, syrk = c["m"], c["n"], c["K"], c["split"], c["epi"], c["syrk"]
    if A is None:
        A = int_operand(torch, gen, m, K, c["lda"], split)
    A = tuple(None if x is None else x.view(-1)[a_off:] for x in A)   # the operand as the kernel sees it
    B = A if syrk else int_operand(torch, gen, n, K, c["ldb"], split)
    rows, cols = {gr.STORE: (m, n), gr.STORE_T: (n, m), gr.COLABSMAX: (1, n)}[epi]
    ldc = n if epi == gr.COLABSMAX else (c["ldc"] if c["ldc"] > cols else c["ldc"] + 8)
    extent = rows * ldc
    splits = c["splits"]
    reduce = splits > 1 and c["reduce"] is not None
    alpha = np.float32(1.0) if reduce else c["alpha"]
    stride = extent if splits > 1 else 0
    Cbuf = torch.full(((splits - 1) * stride + extent + GUARD_TAIL,), float("nan"), device="cuda")
    if epi == gr.COLABSMAX:
        Cbuf[:n] = 0
    red = torch.full((stride + GUARD_TAIL,), float("nan"), device="cuda") if reduce else None
    torch.cuda.synchronize()
    rc, launch = call(h, m, n, K, A, c["lda"], B, c["ldb"], alpha, epi, syrk, splits, stride, c["chunk_kb"], cg, Cbuf, ldc,
                      red, c["reduce"] if reduce else 1.0)
    h._ck(rc)
    r = gr.resolve(m, n, K, split=split, cg=cg, syrk=syrk, epi=epi, splits=splits, chunk_kb=c["chunk_kb"], sms=sms)
    assert launch == gr.report(r), (launch, gr.report(r))

    rows_of = lambda x, r, ld: None if x is None else x.reshape(-1)[: r * ld].view(r, ld)   # noqa: E731
    S = exact_product(torch, [rows_of(x, m, c["lda"]) for x in A], [rows_of(x, n, c["ldb"]) for x in B], m, n, K)
    del A, B
    scale = torch.tensor(float(c["reduce"] if reduce else alpha), dtype=torch.float32, device="cuda")
    if epi == gr.COLABSMAX:
        want = S.abs().amax(dim=0) * scale
        assert torch.equal(Cbuf[:n], want), float((Cbuf[:n] - want).abs().max())
        assert torch.isnan(Cbuf[n:]).all()
        return launch
    want = S * scale
    if epi == gr.STORE_T:
        want = want.T
    out = (red if reduce else Cbuf)[:extent].view(rows, ldc)
    bad = (out[:, :cols] != want) | torch.isnan(out[:, :cols])
    assert not bad.any(), (int(bad.sum()), torch.nonzero(bad)[:5].tolist())
    assert torch.isnan(Cbuf[(splits - 1) * stride + extent:]).all(), "result written past its extent"
    if reduce:
        assert torch.isnan(red[extent:]).all()
    for s in range(splits):
        part = Cbuf[s * stride: s * stride + extent].view(rows, ldc)
        assert torch.isnan(part[:, cols:]).all(), f"spare columns written (partition {s})"
        assert not torch.isnan(part[:, :cols]).any(), f"partition {s} not written"
        if s * r["kb_per_split"] >= r["kblocks"]:
            assert not part[:, :cols].any(), f"empty partition {s} is not zero"
    return launch


def case_list(sms):
    out = []
    for c in gr.production_cases(sms):
        for cg in ([c["cg"]] if c["cg"] else [2, 1]):
            out.append(pytest.param(c["name"], cg, id=f"{c['name']}-cg{cg}"))
    return out


def test_fp32_products_are_exact(torch):
    gen = torch.Generator(device="cuda").manual_seed(1)
    A = int_operand(torch, gen, 300, 5000, 5008, True)
    B = int_operand(torch, gen, 200, 5000, 5008, True)
    S = exact_product(torch, A, B, 300, 200, 5000)
    a = [x[:300, :5000].double() for x in A]
    b = [x[:200, :5000].double() for x in B]
    S64 = a[0] @ b[0].T + a[0] @ b[1].T + a[1] @ b[0].T
    assert torch.equal(S.double(), S64)


@pytest.mark.parametrize("name,cg", case_list(148))
def test_production_call_site(torch, h, sms, name, cg):
    c = [c for c in gr.production_cases(sms) if c["name"] == name][0]
    run_case(torch, h, sms, c, cg, seed=zlib.crc32(name.encode()))


@pytest.mark.parametrize("rank", [0, 1])
def test_sharded_gram_window(torch, h, sms, rank):
    """gram_of on rank `rank` of two: the operand from hi + k0 over the rank's K window, the columns after it holding data."""
    M, N = 4000, 68000
    ld = gr.round8(N)
    kblocks = (N + 63) // 64
    per = (kblocks + 1) // 2
    k0 = min(ld, rank * per * 64)
    k1 = ld if rank == 1 else min(ld, (rank + 1) * per * 64)
    Ks = min(N, k1) - k0
    gen = torch.Generator(device="cuda").manual_seed(7)
    A = int_operand(torch, gen, M, N, ld, False)
    c = dict(m=M, n=M, K=Ks, lda=ld, ldb=ld, split=False, syrk=True, epi=gr.STORE, splits=1, chunk_kb=0, ldc=M,
             alpha=np.float32(1.0) / np.float32(M), reduce=None)
    run_case(torch, h, sms, c, 2, seed=0, A=A, a_off=k0)


EDGE = [1, 31, 32, 33, 127, 128, 129, 255, 256, 257]
EDGE_K = [8, 63, 64, 65, 1000, 4097]


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("cg", [2, 1])
def test_edges(torch, h, sms, cg, split):
    """m x n over the edge sizes, K cycling through its edges, Store and StoreTransposed, a positive and a negative alpha
    that round; K padded to ld = round8(K) + 8."""
    for i, m in enumerate(EDGE):
        for j, n in enumerate(EDGE):
            K = EDGE_K[(i + j) % len(EDGE_K)]
            ld = gr.round8(K) + 8
            epi = gr.STORE if (i + j) % 2 == 0 else gr.STORE_T
            c = dict(m=m, n=n, K=K, lda=ld, ldb=ld, split=split, syrk=False, epi=epi, splits=1, chunk_kb=0,
                     ldc=n if epi == gr.STORE else m, alpha=np.float32(0.3 if i % 2 else -0.7), reduce=None)
            run_case(torch, h, sms, c, cg, seed=100 * i + j)


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("cg", [2, 1])
def test_syrk_edges(torch, h, sms, cg, split):
    """The lower tile triangle and its mirror at 1, 129 and 257 rows, and at 4 100 rows, whose triangle has more tiles than
    there are units; also split-K with the mirror and with chunking."""
    for rows, K, splits, chunk_kb in ((1, 65, 1, 0), (129, 1000, 1, 0), (257, 4097, 1, 0), (4100, 1000, 1, 0),
                                      (257, 4097, 3, 2), (1000, 4097, 5, 3)):
        ld = gr.round8(K) + 8
        c = dict(m=rows, n=rows, K=K, lda=ld, ldb=ld, split=split, syrk=True, epi=gr.STORE, splits=splits, chunk_kb=chunk_kb,
                 ldc=rows, alpha=np.float32(1.0) / np.float32(3.0), reduce=np.float32(0.1) if splits > 1 else None)
        launch = run_case(torch, h, sms, c, cg, seed=rows + K)
        if rows == 4100:
            assert launch[1] > launch[2]


@pytest.mark.parametrize("cg", [1, 2])
def test_empty_split_partition(torch, h, sms, cg):
    """25 k-blocks in 6 splits: the last partition is empty and comes out zero; on the units that meet it a partition with
    work follows on the same accumulator stage."""
    c = [c for c in gr.empty_split_cases() if c["cg"] == cg][0]
    launch = run_case(torch, h, sms, c, cg, seed=cg)
    assert launch[3] == 6 and launch[6] >= 2


def same_sign_operand(torch, rows, K, seed):
    """Rows with a common positive component (same-sign off-diagonal sums, as normalised expression data): the case where
    the tensor core's truncation accumulates; hi + lo = the FP32 rows."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn((rows, K), generator=g, device="cuda") * 0.5 + torch.randn((1, K), generator=g, device="cuda").abs()
    hi = A.half()
    lo = (A - hi.float()).half()
    return hi, lo


@pytest.mark.parametrize("split,chunk_kb", [(False, 0), (True, 0), (True, gr.Q1_CHUNK_KB)])
def test_chunked_accumulation_bounds_the_truncation_bias(torch, h, sms, split, chunk_kb):
    """The mean relative shortfall of the off-diagonal of a same-sign Gram is above 0 and at most L 2^-23, L the MMAs of one
    accumulation chain as resolved; with one chain over the whole K it exceeds that bound."""
    rows, K = 256, 68000
    hi, lo = same_sign_operand(torch, rows, K, 5)
    lo = lo if split else None
    h64 = hi.double()
    E = h64 @ h64.T
    if split:
        l64 = lo.double()
        E = E + h64 @ l64.T + l64 @ h64.T
    off = ~torch.eye(rows, dtype=torch.bool, device="cuda")

    def shortfall(ckb):
        G = torch.empty((rows, rows), device="cuda")
        torch.cuda.synchronize()
        rc, launch = call(h, rows, rows, K, (hi, lo), K, (hi, lo), K, 1.0, gr.STORE, True, 1, 0, ckb, 2, G, rows)
        h._ck(rc)
        return float(((E - G.double()) / E)[off].mean()), launch

    r = gr.resolve(rows, rows, K, split=split, cg=2, syrk=True, chunk_kb=chunk_kb, sms=sms)
    bound = r["mmas_per_chunk"] * 2.0 ** -23
    s, launch = shortfall(chunk_kb)
    assert launch[5] == 1 and launch[4] == r["chunk_kb"]
    assert 0 < s <= bound, (s, bound)
    if chunk_kb == 0:
        s_off, launch = shortfall(r["kblocks"])
        assert launch[5] == 0
        assert s_off > bound, (s_off, bound)


def test_invalid_arguments_are_refused(torch, h):
    gen = torch.Generator(device="cuda").manual_seed(3)
    A = int_operand(torch, gen, 64, 128, 128, True)
    B = int_operand(torch, gen, 32, 128, 128, True)
    Cb = torch.zeros(64 * 64 * 4, device="cuda")
    ok = dict(m=64, n=32, K=128, A=A, lda=128, B=B, ldb=128, alpha=1.0, epi=0, syrk=False, splits=1, split_stride=0,
              chunk_kb=0, cg=2, Cbuf=Cb, ldc=32)

    def rc(**kw):
        a = dict(ok, **kw)
        return call(h, a["m"], a["n"], a["K"], a["A"], a["lda"], a["B"], a["ldb"], a["alpha"], a["epi"], a["syrk"], a["splits"],
                    a["split_stride"], a["chunk_kb"], a["cg"], a["Cbuf"], a["ldc"])[0]

    assert rc() == 0
    bad = [dict(syrk=True), dict(syrk=True, n=64, B=(A[0], None)), dict(A=(A[0], None)), dict(lda=120),
           dict(ldb=100), dict(lda=132), dict(A=(A[0].view(-1)[4:], A[1])), dict(ldc=31), dict(epi=1, ldc=63),
           dict(splits=0), dict(chunk_kb=-1), dict(cg=3), dict(cg=0), dict(epi=3), dict(epi=-1), dict(splits=2, split_stride=10),
           dict(syrk=True, n=64, B=A, epi=1, ldc=64), dict(m=0), dict(K=0)]
    for kw in bad:
        assert rc(**kw) == -1, kw
