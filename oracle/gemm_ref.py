"""CPU restatement of the launch arithmetic and the barrier protocol of the tcgen05 GEMM (sclens_b200/csrc/gemm_umma.cu).

TEST INFRASTRUCTURE ONLY - imported by tests/ (and nothing else).

  launch    block_n, the tile list of build_tiles() (8 x 8 super-tiles, split index innermost, syrk: lower tile triangle),
            the effective split count, the accumulation chunks and the persistent units, as launch() resolves them
  callers   pick_splits() of gemm_splitk (pipeline.cu) and the split choice of apply_G (subspace.cu)
  cases     the production call sites at the 68 000 cells x 20 000 genes workload, restated from their callers, and the
            cases that reach the empty split-K partition; tests/test_gemm_gpu.py runs them, tests/test_gemm_cpu.py checks
            what they reach
  protocol  the three roles of k_gemm_umma (TMA producer, MMA issuer, epilogue) as sequences of mbarrier waits and
            arrivals over one unit's items, and a scheduler that runs them against each other and reports every wait
            that passes before the event it stands for
"""
import itertools
import math

import numpy as np

KBLOCK = 64          # binary16 elements per k-block
TILE_ROWS_A = 128    # A rows per CTA: UMMA M = 128 * cta_group
MAX_BLOCK_N = 256
SMEM_BUDGET = 192 * 1024
STORE, STORE_T, COLABSMAX = 0, 1, 2
UNIT_SCALE = np.float32(1024.0)   # kUnitScale (pipeline.cu)
G_SCALE = np.float32(64.0)        # kGScale (subspace.cu)
Q1_PANELS, Q1_BAND, Q1_CHUNK_KB = 8, 64, 4   # kQ1Panels, kBand, kQ1ChunkKb (backtrans.cu)


def round8(x):
    return (x + 7) // 8 * 8


def block_n_of(n_rows, syrk):
    if syrk:
        return MAX_BLOCK_N
    return max(32, min(MAX_BLOCK_N, (n_rows + 31) // 32 * 32))


def build_tiles(tiles_m, tiles_n, splits, syrk, tile_m, tile_n):
    out = []
    S = 8
    for sm in range(0, tiles_m, S):
        for sn in range(0, tiles_n, S):
            for tm in range(sm, min(tiles_m, sm + S)):
                for tn in range(sn, min(tiles_n, sn + S)):
                    if syrk and tn * tile_n > (tm + 1) * tile_m - 1:
                        continue
                    out.extend((tm, tn, s) for s in range(splits))
    return out


def stages(cg, split):
    rows_b = MAX_BLOCK_N // cg
    return SMEM_BUDGET // ((TILE_ROWS_A * 128 + rows_b * 128) * (2 if split else 1))


def resolve(m, n, K, *, split, cg, syrk=False, epi=STORE, splits=1, chunk_kb=0, sms=148):
    """What launch() makes of a call: the fields scl_debug_gemm reports, the tile list and the per-split k-block count."""
    tile_m = TILE_ROWS_A * cg
    bn = block_n_of(n, syrk)
    kblocks = (K + KBLOCK - 1) // KBLOCK
    s = max(1, min(splits, kblocks))
    tiles = build_tiles((m + tile_m - 1) // tile_m, (n + bn - 1) // bn, s, syrk, tile_m, bn)
    kbs = (kblocks + s - 1) // s
    want = 1 << 30 if epi == COLABSMAX else (chunk_kb if chunk_kb > 0 else (21 if split else 64))
    n_chunks = max(1, (kbs + want - 1) // want)
    ckb = max(1, (kbs + n_chunks - 1) // n_chunks)
    units = min(sms // cg, len(tiles))
    return dict(block_n=bn, n_tiles=len(tiles), units=units, splits=s, chunk_kb=ckb, chunked=int(n_chunks > 1),
                max_per_unit=(len(tiles) + units - 1) // units, tiles=tiles, kblocks=kblocks, kb_per_split=kbs,
                mmas_per_chunk=ckb * (KBLOCK // 16) * (3 if split else 1))


def report(r):
    """The seven launch fields in the order scl_debug_gemm reports them."""
    return [r[k] for k in ("block_n", "n_tiles", "units", "splits", "chunk_kb", "chunked", "max_per_unit")]


def unit_items(r, unit):
    """(kb0, kb1) of every tile-split the unit walks, in order (kb1 <= kb0: an empty split-K partition)."""
    kbs, kb = r["kb_per_split"], r["kblocks"]
    return [(t[2] * kbs, min(kb, t[2] * kbs + kbs)) for t in r["tiles"][unit::r["units"]]]


def n_chunks(kb0, kb1, chunk_kb):
    """Passes of the issuer's and the epilogue's do-while over one item (one for an empty item)."""
    return max(1, -(-(kb1 - kb0) // chunk_kb))


def pick_splits(tiles, K, cg, sms=148):
    """gemm_splitk (pipeline.cu)."""
    units = sms // cg
    kblocks = (K + 63) // 64
    s = max(1, units // max(1, tiles))
    return max(1, min(s, max(1, kblocks // 4)))


def splitk_tiles(m, n, cg):
    """The tile count gemm_splitk hands pick_splits (block_n 256 whatever n is, the full rectangle also for syrk)."""
    tile_m = 128 * cg
    return ((m + tile_m - 1) // tile_m) * ((n + 255) // 256)


def apply_g_splits(n, cg, sms=148):
    """apply_G (subspace.cu): the split count with the fewest waves per unit of work."""
    units = sms // cg
    tiles = (n + 128 * cg - 1) // (128 * cg)
    kblocks = (n + 63) // 64
    best, best_cost = 1, 1e30
    s = 1
    while s <= 16 and s * 8 <= kblocks:
        cost = math.ceil(tiles * s / units) / s + 0.02 * s
        if cost < best_cost:
            best_cost, best = cost, s
        s += 1
    return best


# ---- the call sites ---------------------------------------------------------------------------------------------------

def production_cases(sms=148, N=68000, M=20000, k=75, n_perturb=20, min_pc=75, n_eig=19997):
    """Every call of gemm_umma the 68 000 x 20 000 workload makes, with the fields its caller sets.  Each case: m, n, K,
    lda, ldb, split, cg, syrk, epi, splits, chunk_kb, ldc, alpha, reduce (the scale of the caller's reduce_splits, or
    None).  `cg` None: the handle's cta_group (the test runs both)."""
    f32 = np.float32
    cases = []

    def add(name, m, n, K, ld_a, ld_b, split, cg, *, syrk=False, epi=STORE, splits=1, chunk_kb=0, ldc=None, alpha=1.0,
            reduce=None):
        cases.append(dict(name=name, m=m, n=n, K=K, lda=ld_a, ldb=ld_b, split=split, cg=cg, syrk=syrk, epi=epi,
                          splits=splits, chunk_kb=chunk_kb, ldc=ldc, alpha=f32(alpha), reduce=reduce))

    # gram_of (gene side: rows = genes, contraction over cells), scale 1/M; single-pass and split operands
    for split in (False, True):
        add(f"gram_{'split' if split else 'single'}", M, M, N, round8(N), round8(N), split, None, syrk=True, ldc=M,
            alpha=f32(1.0) / f32(M))
    # corr_colabsmax: |V' W| column maxima, unit vectors pre-scaled by kUnitScale
    add("corr_colabsmax", M, M // 2, M, round8(M), round8(M), True, None, epi=COLABSMAX, ldc=0,
        alpha=f32(1.0) / (UNIT_SCALE * UNIT_SCALE))
    # back_project: X (cells x genes) * V', StoreTransposed into [k][N]
    add("back_project", N, k, M, round8(M), round8(M), True, None, epi=STORE_T, ldc=N)
    # gene_basis: X (genes x cells) * nV', Store with ldc = k
    add("gene_basis", M, k, N, round8(N), round8(N), True, None, ldc=k,
        alpha=f32(1.0) / np.sqrt(f32(M)) / UNIT_SCALE)
    # apply_G of the subspace iteration: G (n x n) * Q', StoreTransposed, split-K with its own rule, reduced by 1/kGScale
    for cg in (2, 1):
        s = apply_g_splits(M, cg, sms)
        add(f"apply_G_cg{cg}", M, k, M, round8(M), round8(M), True, cg, epi=STORE_T, splits=s, ldc=M,
            reduce=f32(1.0) / G_SCALE)
    # score_sets: nV' * sets (Store) and the stack's pairwise products (syrk), both through gemm_splitk
    tot = n_perturb * min_pc
    R = n_perturb * k
    for cg in (2, 1):
        add(f"score_sets_store_cg{cg}", k, tot, N, round8(N), round8(N), True, cg, ldc=tot,
            splits=pick_splits(splitk_tiles(k, tot, cg), N, cg, sms), reduce=f32(1.0) / (UNIT_SCALE * UNIT_SCALE))
        add(f"score_sets_syrk_cg{cg}", R, R, N, round8(N), round8(N), True, cg, syrk=True, ldc=R,
            splits=pick_splits(splitk_tiles(R, R, cg), N, cg, sms), reduce=f32(1.0) / (UNIT_SCALE * UNIT_SCALE))
    # apply_q1_umma, the first (largest) block of an n_eig solve with all vectors: cta_group 2 (the GemmArgs default)
    ncols = Q1_PANELS * Q1_BAND
    m = n_eig - Q1_BAND
    ldk, ldo, mvec = round8(m), ncols, n_eig
    add("q1_Y", ncols, mvec, m, ldk, ldk, True, 2, chunk_kb=Q1_CHUNK_KB, ldc=round8(mvec),
        alpha=f32(1.0) / (f32(1024.0) * f32(1024.0)))
    add("q1_syrk", ncols, ncols, m, ldk, ldk, True, 2, syrk=True, ldc=ldo, alpha=f32(1.0) / (f32(1024.0) * f32(1024.0)))
    add("q1_U", mvec, m, ncols, ldo, ldo, True, 2, chunk_kb=Q1_CHUNK_KB, ldc=ldk, alpha=-f32(1.0) / (f32(256.0) * f32(64.0)))
    return cases


def empty_split_cases():
    """cta_group 1 and 2: 1 920 x 2 560, K = 1 600 in 6 splits = 25 k-blocks as [0,5) ... [20,25) and the empty [25,25)."""
    return [dict(name=f"empty_split_cg{cg}", m=1920, n=2560, K=1600, lda=1600, ldb=1600, split=False, cg=cg, syrk=False,
                 epi=STORE, splits=6, chunk_kb=0, ldc=2560, alpha=np.float32(1.0), reduce=np.float32(0.5)) for cg in (1, 2)]


# ---- the barrier protocol ---------------------------------------------------------------------------------------------

def role_programs(items, chunk_kb, chunked, ring, fixed):
    """The waits and arrivals of the three roles of one unit, restated from k_gemm_umma.  fixed=False: the protocol before
    empty split-K partitions were skipped (the issuer waited tmem_empty and advanced its stage for an empty item without a
    commit; the epilogue released and advanced without a wait).  Ops: ("wait", bar, parity, tag) / ("arrive", bar, tag)."""
    n_acc = 1 if chunked else 2
    prod, iss, epi = [], [], []
    stage = phase = 0
    for kb0, kb1 in items:
        for _ in range(kb0, kb1):
            prod += [("wait", ("empty", stage), phase ^ 1, None), ("arrive", ("full", stage), None)]
            stage, phase = (0, phase ^ 1) if stage + 1 == ring else (stage + 1, phase)
    stage = phase = acc = acc_phase = 0
    for i, (kb0, kb1) in enumerate(items):
        if fixed and kb1 <= kb0:
            continue
        kb, c = kb0, 0
        while True:
            kend = min(kb1, kb + chunk_kb)
            iss.append(("wait", ("tmem_empty", acc), acc_phase ^ 1, ("mma", i, c, acc)))
            while kb < kend:
                iss += [("wait", ("full", stage), phase, None), ("arrive", ("empty", stage), None)]
                stage, phase = (0, phase ^ 1) if stage + 1 == ring else (stage + 1, phase)
                kb += 1
            if fixed or kb1 > kb0:
                iss.append(("arrive", ("tmem_full", acc), ("commit", i, c)))
            acc, acc_phase = (0, acc_phase ^ 1) if acc + 1 == n_acc else (acc + 1, acc_phase)
            c += 1
            if not kb < kb1:
                break
    acc = acc_phase = 0
    for i, (kb0, kb1) in enumerate(items):
        have = kb1 > kb0
        kb, c = kb0, 0
        while True:
            kb = min(kb1, kb + chunk_kb)
            if have:
                epi.append(("wait", ("tmem_full", acc), acc_phase, ("read", i, c)))
            if have or not fixed:
                epi.append(("arrive", ("tmem_empty", acc), ("release", i, c)))
                acc, acc_phase = (0, acc_phase ^ 1) if acc + 1 == n_acc else (acc + 1, acc_phase)
            c += 1
            if not kb < kb1:
                break
    return {"epilogue": epi, "producer": prod, "issuer": iss}


def simulate(programs, order):
    """Run the roles against each other, each step the first role in `order` that can go on (an mbarrier wait on parity P
    passes once the barrier's completed phases have the other parity; every barrier here completes on one arrival).
    Returns (violations, deadlocked): a violation is an epilogue read whose MMAs were not committed yet, or an MMA chain
    started on an accumulator stage whose previous chain the epilogue had not released yet."""
    done = {}                 # barrier -> completed phases
    pc = {r: 0 for r in programs}
    committed, released = set(), set()
    occupant = {}             # accumulator stage -> the (item, chunk) whose MMAs last went there
    violations = []
    while True:
        moved = False
        for r in order:
            prog = programs[r]
            if pc[r] == len(prog):
                continue
            op = prog[pc[r]]
            if op[0] == "wait":
                _, bar, parity, tag = op
                if (done.get(bar, 0) & 1) == parity:
                    continue
                if tag and tag[0] == "read" and (tag[1], tag[2]) not in committed:
                    violations.append(("early tmem_full", tag[1], tag[2]))
                if tag and tag[0] == "mma":
                    prev = occupant.get(tag[3])
                    if prev is not None and prev not in released:
                        violations.append(("early tmem_empty", tag[1], tag[2]))
                    occupant[tag[3]] = (tag[1], tag[2])
            else:
                _, bar, tag = op
                done[bar] = done.get(bar, 0) + 1
                if tag and tag[0] == "commit":
                    committed.add((tag[1], tag[2]))
                if tag and tag[0] == "release":
                    released.add((tag[1], tag[2]))
            pc[r] += 1
            moved = True
            break
        if not moved:
            return violations, any(pc[r] < len(programs[r]) for r in programs)


def check_protocol(items, chunk_kb, chunked, ring, fixed):
    """simulate() under every priority order of the three roles: (all violations, any deadlock)."""
    progs = role_programs(items, chunk_kb, chunked, ring, fixed)
    found, dead = [], False
    for order in itertools.permutations(progs):
        v, d = simulate(progs, order)
        found += v
        dead |= d
    return found, dead
