"""The launch plans of the estimator sweeps (plan_fast and plan_terms in kgl_gene_b200/csrc/terms_launch.cuh), compiled as a host
program (tests/terms_plan_probe.cu) and checked without a GPU.

k_terms_fast gives each warp `slots` genome blocks, spreads ceil(gblocks / (warps * slots)) rows of CTAs over grid.y and the
256-locus tiles of the selection window over grid.x in chunks; every CTA holds one tile's table and the accumulators of all its
slots in shared memory. A plan whose shared memory exceeds the device's opt-in limit cannot launch; an empty row of CTAs, a chunk
outside the window or a selected row outside it would lose or double terms. k_genome_terms (loglik_grid, the exact Newton
fallback) cuts the words into chunks of whole 4-word tiles. tests/test_gpu_sweep_plans.py runs the kernels at the plans pinned
by test_plan_regimes_at_148_sms."""
import numpy as np
import pytest

import terms_plan_probe as TP

SMS = (1, 2, 132, 148, 160)
LIMIT = TP.B200_SMEM_OPTIN
GBLOCKS = np.arange(1, 4001)
# sample-major words (multiples of 4) around the 8-word tile: one tile, a last tile of 4 words, config 2 (1.1 M loci) and 20 M loci
WORDS = (4, 8, 12, 16, 100, 628, 1252, 34_376, 625_000)
# selection windows [lo, hi) in rows, -1: none; around the 256-row tile boundaries
WINDOWS = ((0, -1), (0, 0), (300, 480), (100, 513), (255, 257), (256, 512), (511, 1_000_000), (39_000, 40_000), (5, 7))


@pytest.fixture(scope="module")
def probe():
    try:
        TP.probe_binary()
    except FileNotFoundError:
        pytest.skip("nvcc is not installed")
    return TP


def cdiv(a, b):
    return -(-a // b)


def smem_bytes(mode, slots, warps):
    """6 population rows of (256 loci x 4 codes + 4) entries of 1 or 2 doubles, the slot accumulators of every thread (1, 2 or 3
    doubles), the RITLAND masks."""
    entry = np.where((mode == 3) | (mode == 4), 2, 1)
    n_acc = np.where(mode == 1, 1, np.where(mode == 4, 3, 2))
    return 6 * 1028 * entry * 8 + slots * warps * 32 * n_acc * 8 + 6 * 8 * 2 * 4


def restated(c, fit_only):
    """The plan as launch_fast chose it before terms_launch.cuh (fit_only=False: whatever its shared memory), or with the search
    limited to the shapes that fit (fit_only=True), restated in numpy. -> dict of arrays."""
    mode, gb, nw, lo, hi, sms, limit = (c[f] for f in ("mode", "gblocks", "n_words", "sel_row_lo", "sel_row_hi", "sm_count", "smem_limit"))
    warps, best = np.zeros_like(gb), np.full(gb.shape, -1.0)
    for w in range(16, 25):
        sl = np.minimum(8, cdiv(gb, w))
        rows = cdiv(gb, w * sl)
        filled = gb / (rows * sl * w)
        take = filled >= best
        if fit_only:
            take &= smem_bytes(mode, sl, w) <= limit
        best = np.where(take, filled, best)
        warps = np.where(take, w, warps)
    small = gb <= 8
    warps = np.where(small, np.where(gb <= 4, 4, 8), warps)
    ctas = np.where(small, 4, 1)
    slots = np.minimum(8, cdiv(gb, np.maximum(warps, 1)))
    smem = smem_bytes(mode, slots, warps)
    ok = (warps > 0) & (smem <= limit) if fit_only else np.ones(gb.shape, dtype=bool)
    gy = cdiv(gb, np.maximum(warps * slots, 1))
    all_tiles = cdiv(nw, 8)
    tb = np.minimum(all_tiles, lo // 256)
    te = np.maximum(tb, np.minimum(all_tiles, np.where(hi < 0, all_tiles, cdiv(hi, 256))))
    n_tiles = np.maximum(1, te - tb)
    want = np.maximum(1, sms * ctas // np.maximum(gy, 1))
    tpc = np.maximum(1, cdiv(n_tiles, want))
    return dict(ok=ok, warps=warps, ctas_per_sm=ctas, slots=slots, gy=gy, tile_begin=tb, tile_end=te, tiles_per_chunk=tpc,
                n_chunks=cdiv(n_tiles, tpc), smem=smem)


def sweep(sms, modes=range(5), limit=LIMIT):
    """Every genome-block count 1..4,000 x every mode, with the words and windows cycling through WORDS and WINDOWS."""
    req = []
    for m in modes:
        for g in GBLOCKS.tolist():
            nw = WORDS[(g + m) % len(WORDS)]
            lo, hi = WINDOWS[(g // 3 + m) % len(WINDOWS)]
            req.append((m, g, nw, lo, hi, sms, limit))
    return req


def assert_no_violation(cols, checks):
    bad = {name: np.flatnonzero(m) for name, m in checks.items() if m.any()}
    if bad:
        lines = []
        for name, idx in bad.items():
            i = int(idx[0])
            lines.append(f"{name}: {idx.size} plans, e.g. " + ", ".join(f"{f}={int(v[i])}" for f, v in cols.items()))
        pytest.fail("\n".join(lines))


def violations(c):
    gb, w, sl, gy, ctas = c["gblocks"], c["warps"], c["slots"], c["gy"], c["ctas_per_sm"]
    tb, te, tpc, nc, last = c["tile_begin"], c["tile_end"], c["tiles_per_chunk"], c["n_chunks"], c["last_chunk_tiles"]
    nw, lo, hi = c["n_words"], c["sel_row_lo"], c["sel_row_hi"]
    rows = np.minimum(np.where(hi < 0, nw * 32, hi), nw * 32)         # selectable rows end (the matrix has nw * 32 rows at most)
    window = rows > lo
    return {
        "a plan for every shape (ok)": c["ok"] != 1,
        "smem <= the opt-in limit": c["smem"] > c["smem_limit"],
        "smem as stated": c["smem"] != smem_bytes(c["mode"], sl, w),
        "warps 16..24, or 4 / 8 with 4 CTAs per SM when gblocks <= 8":
            np.where(gb <= 8, (w != np.where(gb <= 4, 4, 8)) | (ctas != 4), (w < 16) | (w > 24) | (ctas != 1)),
        "slots 1..8": (sl < 1) | (sl > 8),
        "gy * warps * slots >= gblocks": gy * w * sl < gb,
        "no empty row of CTAs": (gy - 1) * w * sl >= gb,
        "chunks cover the tiles": nc * tpc < np.maximum(1, te - tb),
        "no empty chunk": (nc < 1) | ((nc - 1) * tpc >= np.maximum(1, te - tb)),
        "last chunk as stated": (last < 1) | (last > tpc) | ((nc - 1) * tpc + last != np.maximum(1, te - tb)),
        "window inside the matrix": (tb > te) | (te > cdiv(nw, 8)),
        "window covers every selectable row": window & ((tb * 256 > lo) | (te * 256 < rows)),
        "window has no tile without a selectable row": window & ((tb + 1) * 256 <= lo) | window & ((te - 1) * 256 >= rows),
        "k_genome_terms chunks whole tiles": (c["term_words_per_chunk"] < 4) | (c["term_words_per_chunk"] % 4 != 0),
        "k_genome_terms chunks cover the words": c["term_n_chunks"] * c["term_words_per_chunk"] < nw,
        "k_genome_terms: no empty chunk": (c["term_last_chunk_words"] < 1) | (c["term_last_chunk_words"] > c["term_words_per_chunk"]),
        "k_genome_terms: one CTA per 8 genome blocks": c["term_gx"] != cdiv(gb, 8),
    }


@pytest.mark.parametrize("sms", SMS)
def test_plan_invariants_over_the_sweep(probe, sms):
    """20,000 plans per SM count (every mode x genome blocks 1..4,000, which include every list length of a late Newton sweep):
    none may break an invariant. Before terms_launch.cuh the unphased root search (NEWTON_U) broke the shared-memory limit at
    8 slots and 22 or more warps, first at 169 genome blocks."""
    consts, cols = probe.plans(sweep(sms))
    assert consts == {"tile_loci": 256, "tile_words": 8, "max_warps": 24, "max_pop": 6, "term_warps": 8, "term_tile_words": 4}
    assert_no_violation(cols, violations(cols))
    # the sweep reaches the small CTAs, 8 slots, several rows of CTAs, several tiles per chunk, an empty window
    assert (cols["warps"] == 4).any() and (cols["warps"] == 8).any() and (cols["slots"] == 8).any() and (cols["gy"] > 1).any()
    assert (cols["tiles_per_chunk"] > 1).any() and (cols["tile_end"] == cols["tile_begin"]).any()


def test_plan_invariants_over_every_sm_count(probe):
    """SM counts 1..160 x every mode x the genome-block counts around the small CTAs, the 8-slot threshold and the NEWTON_U
    overflow ranges (plus a spread to 4,000), each with every window: the invariants, and the restated rule."""
    blocks = sorted(set(range(1, 20)) | set(range(120, 200)) | set(range(380, 400)) | set(range(200, 4001, 97)) | {3_125})
    req = [(m, g, WORDS[(g + s) % len(WORDS)], lo, hi, s, LIMIT) for s in range(1, 161) for m in range(5) for g in blocks
           for lo, hi in WINDOWS[(g + s) % 3::3]]
    _, c = probe.plans(req)
    assert_no_violation(c, violations(c))
    new = restated(c, fit_only=True)
    for f in ("warps", "slots", "gy", "tile_begin", "tile_end", "tiles_per_chunk", "n_chunks", "smem"):
        assert np.array_equal(c[f], new[f]), f


@pytest.mark.parametrize("sms", SMS)
def test_plan_is_the_rule_it_replaced_wherever_that_fits(probe, sms):
    """RITLAND / HALL / NEWTON / LIMITS: the plan is launch_fast's former rule, restated, everywhere (it always fit). NEWTON_U:
    the same wherever that rule fits (so the chunking, and with it the summation order, did not move), and elsewhere the
    shape of fewest empty slots among those that fit."""
    _, c = probe.plans(sweep(sms))
    old, new = restated(c, fit_only=False), restated(c, fit_only=True)
    fields = ("warps", "ctas_per_sm", "slots", "gy", "tile_begin", "tile_end", "tiles_per_chunk", "n_chunks", "smem")
    fits = old["smem"] <= LIMIT
    u = c["mode"] == 4
    assert fits[~u].all()
    for f in fields:
        assert np.array_equal(c[f][fits], old[f][fits]), f
        assert np.array_equal(c[f], new[f]), f
    assert np.array_equal(c["ok"].astype(bool), new["ok"])
    if sms == 148:
        # the former rule overflows for NEWTON_U from 169 genome blocks on (5,377 unphased genomes)
        over = np.flatnonzero(u & ~fits)
        assert over.size and int(c["gblocks"][over].min()) == 169


def test_newton_u_blocks_the_former_rule_overflowed(probe):
    """The table of the bug report: the former rule's NEWTON_U plan and bytes, and the plan that replaces it."""
    rows = [(169, (22, 8, 234_240), (16, 8, 2, 197_376)), (192, (24, 8, 246_528), (16, 8, 2, 197_376)),
            (3_125, (23, 8, 240_384), (17, 8, 23, 203_520)), (193, (16, 8, 197_376), (16, 8, 2, 197_376)),
            (625, (20, 8, 221_952), (20, 8, 4, 221_952))]
    _, c = probe.plans([(4, g, 628, 0, -1, 148, LIMIT) for g, _, _ in rows])
    old = restated(c, fit_only=False)
    for i, (g, (ow, osl, ob), want) in enumerate(rows):
        assert (old["warps"][i], old["slots"][i], old["smem"][i]) == (ow, osl, ob), g
        assert (c["warps"][i], c["slots"][i], c["gy"][i], c["smem"][i]) == want, g


def test_no_plan_is_an_error_not_a_launch(probe):
    """A limit no shape fits (100,000 B: below NEWTON_U's table and one slot of 4 warps) gives ok = 0 for every genome-block
    count; the other modes still plan."""
    _, c = probe.plans([(m, g, 628, 0, -1, 148, 100_000) for m in range(5) for g in (1, 5, 8, 9, 169, 4000)])
    ok = c["ok"].reshape(5, -1)
    assert not ok[4].any()
    assert ok[1].all()            # HALL: 49,728 B of table, 16 x 8 slots x 256 B = 32,768 B
    _, c = probe.plans([(4, g, 628, 0, -1, 148, 120_000) for g in (1, 9, 4000)])
    assert c["ok"].tolist() == [1, 1, 0] and c["smem"][0] <= 120_000


def test_term_chunks(probe):
    """plan_terms over genome blocks 1..4,000 and words around the 4-word tile and the ~4 waves of CTAs it aims for."""
    req = [(0, g, nw, 0, -1, s, LIMIT) for g in range(1, 4001, 7) for nw in (4, 8, 12, 100, 1004, 4740, 34_376) for s in SMS]
    _, c = probe.plans(req)
    assert_no_violation(c, {k: v for k, v in violations(c).items() if k.startswith("k_genome_terms")})
    gx = cdiv(c["gblocks"], 8)
    want = np.maximum(1, cdiv(c["sm_count"] * 8, gx))
    wpc = np.maximum(4, cdiv(cdiv(c["n_words"], want), 4) * 4)
    assert np.array_equal(c["term_words_per_chunk"], wpc)
    assert (c["term_last_chunk_words"] < c["term_words_per_chunk"]).any()


# Plans of the GPU cases at 148 SMs: (name, mode, gblocks, n_words, sel_row_lo, sel_row_hi) -> (warps, CTAs per SM, slots, gy,
# tile_begin, tile_end, tiles per chunk, chunks, last chunk tiles). tests/test_gpu_sweep_plans.py derives its shapes from the probe
# on the device it runs on; on a B200 they are these, and a planner change that moves one of them off its regime fails here first.
REGIMES_148 = [
    # small CTAs: 100 and 230 genomes x 20,000 loci (628 words, 79 tiles)
    ("4 warps", 0, 4, 628, 0, -1, (4, 4, 1, 1, 0, 79, 1, 79, 1)),
    ("8 warps", 1, 8, 628, 0, -1, (8, 4, 1, 1, 0, 79, 1, 79, 1)),
    # 24 x 8 slots (6,144 genomes), and 22 x 8 = 176 slots for 169 blocks (5,408 genomes)
    ("24 x 8", 2, 192, 628, 0, -1, (24, 1, 8, 1, 0, 79, 1, 79, 1)),
    ("22 x 8, partial row", 3, 169, 628, 0, -1, (22, 1, 8, 1, 0, 79, 1, 79, 1)),
    # the unphased root search at the same sizes: 16 x 8 in two rows of CTAs, two tiles per chunk, the last one short
    ("NEWTON_U 6,144", 4, 192, 628, 0, -1, (16, 1, 8, 2, 0, 79, 2, 40, 1)),
    ("NEWTON_U 5,408", 4, 169, 628, 0, -1, (16, 1, 8, 2, 0, 79, 2, 40, 1)),
    ("LIMITS unphased 5,408", 3, 169, 628, 0, -1, (22, 1, 8, 1, 0, 79, 1, 79, 1)),
    # selection windows over 6,144 genomes x 40,000 loci (1,252 words: 157 tiles, the last of 4 words)
    ("window inside one tile", 2, 192, 1_252, 300, 480, (24, 1, 8, 1, 1, 2, 1, 1, 1)),
    ("window one row past a tile", 2, 192, 1_252, 100, 513, (24, 1, 8, 1, 0, 3, 1, 3, 1)),
    ("window to a 4-word last tile", 2, 192, 1_252, 39_000, 40_000, (24, 1, 8, 1, 152, 157, 1, 5, 1)),
    ("every tile, 2 per chunk", 2, 192, 1_252, 0, 40_000, (24, 1, 8, 1, 0, 157, 2, 79, 1)),
]


@pytest.mark.parametrize("name,mode,gblocks,n_words,lo,hi,want", REGIMES_148, ids=[r[0] for r in REGIMES_148])
def test_plan_regimes_at_148_sms(probe, name, mode, gblocks, n_words, lo, hi, want):
    p = probe.plan({v: k for k, v in TP.MODES.items()}[mode], gblocks, n_words, 148, lo, hi)
    got = tuple(p[f] for f in ("warps", "ctas_per_sm", "slots", "gy", "tile_begin", "tile_end", "tiles_per_chunk", "n_chunks",
                               "last_chunk_tiles"))
    assert p["ok"] == 1 and got == want, TP.describe(name, p)


def test_grid_case_at_148_sms(probe):
    """loglik_grid over 2,048 genomes (64 device genome blocks, 8 CTAs per chunk) x 32,128 loci (1,004 words): 126 chunks of
    8 words, the last of 4."""
    p = probe.plan("RITLAND", TP.device_gblocks(2_048), TP.term_words(32_128), 148)
    assert (p["term_gx"], p["term_n_chunks"], p["term_words_per_chunk"], p["term_last_chunk_words"]) == (8, 126, 8, 4)
