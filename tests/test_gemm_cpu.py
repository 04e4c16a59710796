"""CPU checks of oracle/gemm_ref.py, the restatement of the tcgen05 GEMM's launch arithmetic (sclens_b200/csrc/gemm_umma.cu
launch() and build_tiles(), gemm_splitk's pick_splits, apply_G's split choice) and of its barrier protocol.

They pin down what the cases of tests/test_gemm_gpu.py reach at 148 SMs - several tile-splits per persistent unit in both
accumulator modes, 1, 2 and many accumulation chunks, split-K with and without chunking, an empty split-K partition
followed on the same unit by one with work - and show, by running the three roles' mbarrier waits and arrivals against
each other, that the protocol before the empty-partition fix let the epilogue read an accumulator before its MMAs were
committed, and that the fixed protocol never does."""
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import gemm_ref as gr  # noqa: E402

SMS = 148


def resolved(c, cg=None):
    return gr.resolve(c["m"], c["n"], c["K"], split=c["split"], cg=cg or c["cg"], syrk=c["syrk"], epi=c["epi"],
                      splits=c["splits"], chunk_kb=c["chunk_kb"], sms=SMS)


def all_cases():
    out = []
    for c in gr.production_cases(SMS) + gr.empty_split_cases():
        for cg in ([c["cg"]] if c["cg"] else [2, 1]):
            out.append((c, cg, resolved(c, cg)))
    return out


def chunks_of(r):
    return -(-r["kb_per_split"] // r["chunk_kb"])


def test_build_tiles_lower_triangle_and_order():
    t = gr.build_tiles(20, 3, 2, False, 128, 256)
    assert len(t) == 120 and t[:4] == [(0, 0, 0), (0, 0, 1), (0, 1, 0), (0, 1, 1)]
    assert t[6] == (1, 0, 0)                       # rows of one 8 x 8 super-tile first
    assert t[48] == (8, 0, 0)                      # then the next super-tile
    tri = gr.build_tiles(10, 5, 1, True, 128, 256)
    # a tile is kept when its first column is not above its last row
    assert sorted(tri) == sorted((tm, tn, 0) for tm in range(10) for tn in range(5) if tn * 256 <= tm * 128 + 127)


def test_block_n_and_chunk_rules():
    assert [gr.block_n_of(n, False) for n in (1, 31, 32, 33, 75, 256, 257)] == [32, 32, 32, 64, 96, 256, 256]
    assert gr.block_n_of(7, True) == 256
    r = gr.resolve(20000, 20000, 68000, split=False, cg=2, syrk=True)
    assert (r["chunk_kb"], chunks_of(r), r["mmas_per_chunk"]) == (63, 17, 252)
    r = gr.resolve(20000, 20000, 68000, split=True, cg=2, syrk=True)
    assert (r["chunk_kb"], chunks_of(r), r["mmas_per_chunk"]) == (21, 51, 252)
    r = gr.resolve(512, 19997, 19933, split=True, cg=2, chunk_kb=4)
    assert (r["chunk_kb"], r["mmas_per_chunk"]) == (4, 48)
    # ColAbsMax: one chunk whatever K; chunk_kb = all k-blocks switches chunking off
    assert gr.resolve(20000, 10000, 20000, split=True, cg=2, epi=gr.COLABSMAX)["chunked"] == 0
    assert gr.resolve(256, 256, 68000, split=False, cg=2, syrk=True, chunk_kb=1063)["chunked"] == 0
    # more splits than k-blocks are clamped
    assert gr.resolve(128, 128, 100, split=False, cg=1, splits=9)["splits"] == 2


def test_production_launches_match_the_callers():
    by = {(c["name"], cg): r for c, cg, r in all_cases()}
    g = by[("gram_single", 2)]
    assert (g["n_tiles"], g["units"], g["max_per_unit"], chunks_of(g), g["chunk_kb"]) == (3160, 74, 43, 17, 63)
    g = by[("gram_split", 1)]
    assert (g["max_per_unit"], chunks_of(g), g["chunk_kb"]) == (43, 51, 21)
    c = by[("corr_colabsmax", 2)]
    assert (c["max_per_unit"], c["chunked"], c["kblocks"]) == (43, 0, 313)
    b = by[("back_project", 2)]
    assert (b["block_n"], b["max_per_unit"], chunks_of(b)) == (96, 4, 15)
    a = by[("apply_G_cg2", 2)]
    assert (a["splits"], a["max_per_unit"], chunks_of(a)) == (7, 8, 3)
    y = by[("q1_Y", 2)]
    assert (y["max_per_unit"], y["chunk_kb"], chunks_of(y)) == (3, 4, 78)
    u = by[("q1_U", 2)]
    assert (u["max_per_unit"], chunks_of(u)) == (84, 2)
    assert gr.apply_g_splits(20000, 2, SMS) == 7


def test_cases_reach_what_they_claim():
    cases = all_cases()
    # several tile-splits per unit with two accumulator stages and with the chunked single stage
    assert any(r["max_per_unit"] >= 2 and not r["chunked"] for _, _, r in cases)
    assert any(r["max_per_unit"] >= 2 and r["chunked"] for _, _, r in cases)
    # 1, 2 and many accumulation chunks
    counts = {chunks_of(r) for _, _, r in cases}
    assert 1 in counts and 2 in counts and max(counts) >= 50
    # split-K with and without chunking, and split-K with the syrk mirror
    assert any(r["splits"] > 1 and r["chunked"] for _, _, r in cases)
    assert any(r["splits"] > 1 and not r["chunked"] for _, _, r in cases)
    assert any(r["splits"] > 1 and c["syrk"] for c, _, r in cases)
    # ldc larger than the row length, and a negative alpha
    assert any(c["ldc"] and c["epi"] == gr.STORE and not c["syrk"] and c["ldc"] > c["n"] for c, _, _ in cases)
    assert any(c["alpha"] < 0 for c, _, _ in cases)


def empty_then_work(r):
    """(unit, items) of the first unit that meets an empty partition and, two items later (the same accumulator stage of
    the protocol that advanced on every item), a partition with work."""
    for u in range(r["units"]):
        it = gr.unit_items(r, u)
        for j in range(len(it) - 2):
            if it[j][1] <= it[j][0] and it[j + 2][1] > it[j + 2][0]:
                return u, it
    return None


@pytest.mark.parametrize("cg", [1, 2])
def test_empty_split_case_reaches_an_empty_partition_before_work(cg):
    c = [c for c in gr.empty_split_cases() if c["cg"] == cg][0]
    r = resolved(c)
    assert r["kblocks"] == 25 and r["kb_per_split"] == 5 and r["splits"] == 6
    assert (r["n_tiles"], r["max_per_unit"], r["chunked"]) == ((900, 7, 0) if cg == 1 else (480, 7, 0))
    assert empty_then_work(r) is not None


def test_production_split_rules_leave_no_empty_partition_before_work():
    """gemm_splitk makes at most one tile-split per unit; apply_G's rule makes no empty partition below n = 30 000."""
    for cg in (1, 2):
        units = SMS // cg
        for tiles in range(1, units + 1):
            for K in range(64, 70000, 97):
                assert tiles * gr.pick_splits(tiles, K, cg, SMS) <= units
        for n in range(64, 30000, 7):
            s = gr.apply_g_splits(n, cg, SMS)
            kb = (n + 63) // 64
            assert (s - 1) * (-(-kb // s)) < kb, (n, cg, s)


def test_protocol_before_the_fix_reads_before_the_commit():
    for c in gr.empty_split_cases():
        r = resolved(c)
        _, items = empty_then_work(r)
        found, _ = gr.check_protocol(items, r["chunk_kb"], r["chunked"], gr.stages(c["cg"], c["split"]), fixed=False)
        assert any(v[0] == "early tmem_full" for v in found), found
        found, dead = gr.check_protocol(items, r["chunk_kb"], r["chunked"], gr.stages(c["cg"], c["split"]), fixed=True)
        assert found == [] and not dead


@pytest.mark.parametrize("chunked", [0, 1])
def test_fixed_protocol_on_synthetic_item_sequences(chunked):
    """Empty items first, last, in runs and between chunked items: no early wait and no deadlock in any role order."""
    seqs = [[(0, 0), (0, 5)], [(0, 5), (5, 5)], [(3, 3), (3, 3), (0, 9), (9, 9), (0, 2), (4, 4), (0, 7)],
            [(0, 4), (4, 8), (8, 8), (0, 4), (8, 8), (8, 8), (4, 8)], [(12, 10), (0, 6), (12, 10), (6, 10)]]
    for items in seqs:
        for ring in (2, 3):
            found, dead = gr.check_protocol(items, 2 if chunked else 64, chunked, ring, fixed=True)
            assert found == [] and not dead, (items, ring, found)
    # and the old protocol fails on the same kind of sequence
    found, _ = gr.check_protocol([(0, 4), (4, 4), (0, 4), (0, 4)], 64, 0, 3, fixed=False)
    assert found


@pytest.mark.parametrize("name", ["apply_G_cg2", "q1_U", "back_project"])
def test_fixed_protocol_on_production_units(name):
    c = [c for c in gr.production_cases(SMS) if c["name"] == name][0]
    cg = c["cg"] or 2
    r = resolved(c, cg)
    items = gr.unit_items(r, 0)
    found, dead = gr.check_protocol(items, r["chunk_kb"], r["chunked"], gr.stages(cg, c["split"]), fixed=True)
    assert found == [] and not dead
