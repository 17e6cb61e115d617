"""The launch plan of pairwise IBS on the popcount kernel (plan_ibs, ibs_words_used and ibs_repair_segments in
kgl_gene_b200/csrc/ibs_launch.cuh), compiled as a host program (tests/ibs_plan_probe.cu) and checked without a GPU.

k_ibs_tiles runs units of (64 x 64 tile, chunk of 32-locus words) round-robin over one persistent CTA per SM and feeds them
through a ring of six 16-word stages; a unit's last stage holds the words left over, and its consumers step two words at a
time. A chunk with no stage, or a stage with an odd or zero word count, would desynchronise the ring's barriers; a unit index
past 2^32 would wrap in the kernel's uint32 arithmetic. k_ibs_missing_fix cuts every genome's dropped rows into `segs` segments
(gridDim.y) and flushes its counters every 32,760 rows. tests/test_gpu_ibs_plans.py runs both kernels at the plans pinned by
test_plan_regimes_at_148_sms."""
import numpy as np
import pytest

import ibs_plan_probe as IP

SMS = (1, 2, 132, 148, 160)
# words_used around the stage (16 words) and split (16 stages) boundaries, config 2 (1.1 M loci = 34,376 words), config 4 (20 M
# loci = 625,000 words) and just under 2^27 words (2^32 loci); odd word counts round up to even
WORDS = [1, 2, 14, 15, 16, 17, 18, 254, 255, 256, 257, 258, 510, 511, 512, 513, 514, 34_376, 625_000, (1 << 27) - 2]
# average dropped rows per genome around the repair's 256-row segment rule
AVG_ROWS = (0, 255, 256, 511, 512, 1_000, 16_384, 10**6)
N_GENOMES = 5_000


@pytest.fixture(scope="module")
def probe():
    try:
        IP.probe_binary()
    except FileNotFoundError:
        pytest.skip("nvcc is not installed")
    return IP


def violations(c):
    """name -> boolean array of the plans that break the invariant."""
    wu, wpc, nc, grid, units = c["words_used"], c["words_per_chunk"], c["n_chunks"], c["grid"], c["units"]
    segs, last, ls, lsw = c["segs"], c["last_chunk_words"], c["last_chunk_stages"], c["last_stage_words"]
    return {
        "words_used = loci in 32-locus words, rounded up to even": wu != (c["n_loci"] + 31) // 32 + ((c["n_loci"] + 31) // 32) % 2,
        "words_per_chunk a positive multiple of 16": (wpc < 16) | (wpc % 16 != 0),
        "stages_per_chunk = words_per_chunk / 16": c["stages_per_chunk"] * 16 != wpc,
        "chunks cover words_used": nc * wpc < wu,
        "no empty chunk": (nc < 1) | ((nc - 1) * wpc >= wu),
        "last chunk as stated": last != wu - (nc - 1) * wpc,
        ">= 256 words per chunk when split": (nc > 1) & (wpc < 256),
        "<= 4,096 chunks": nc > 4096,
        "grid = min(units, SMs)": grid != np.minimum(units, c["sm_count"]),
        "grid >= 1": grid < 1,
        "units = tiles x chunks": units != c["n_tiles"] * nc,
        "unit index fits uint32 (u + grid)": units + grid >= 1 << 32,
        "units per CTA": c["max_units_per_cta"] != -(-units // grid),
        "last stage even, 2..16 words": (lsw < 2) | (lsw > 16) | (lsw % 2 != 0) | ((ls - 1) * 16 + lsw != last),
        "1 <= segs <= 64": (segs < 1) | (segs > 64),
        "segs = 1 from 8 x SMs tiles": (c["n_tiles"] >= 8 * c["sm_count"]) & (segs != 1),
        "segs = 1 below 512 rows per genome": (c["n_dropped"] // c["n_genomes"] < 512) & (segs != 1),
    }


def assert_no_violation(cols, checks):
    bad = {name: np.flatnonzero(m) for name, m in checks.items() if m.any()}
    if bad:
        lines = []
        for name, idx in bad.items():
            i = int(idx[0])
            lines.append(f"{name}: {idx.size} plans, e.g. " + ", ".join(f"{f}={int(v[i])}" for f, v in cols.items()))
        pytest.fail("\n".join(lines))


@pytest.mark.parametrize("sms", SMS)
def test_plan_invariants_over_the_sweep(probe, sms):
    """Every tile count of one launch (1..8,192) x 20 word counts, with the average dropped rows per genome cycling through
    AVG_ROWS (~164,000 plans per SM count): none may break an invariant (none did when this was written)."""
    req = [(t, 32 * w, sms, AVG_ROWS[(t + i) % len(AVG_ROWS)] * N_GENOMES, N_GENOMES)
           for t in range(1, 8193) for i, w in enumerate(WORDS)]
    consts, cols = probe.plans(req)
    assert consts == {"stage_words": 16, "ring": 6, "prefetch": 3, "flush_rows": 32_760, "max_tiles_per_launch": 8192, "tile": 64}
    assert cols["n_tiles"].size == len(req)
    assert_no_violation(cols, violations(cols))
    # the sweep reaches every regime of both kernels: one chunk and split, several units per CTA, a last stage of 2 and of 16
    # words, several repair segments; a split only on more than one SM
    nc = cols["n_chunks"]
    assert (nc == 1).any() and (nc > 1).any() == (sms > 1)
    assert ((nc > 1) & (cols["max_units_per_cta"] >= 3)).any() == (sms > 1)
    assert (cols["last_stage_words"] == 2).any() and (cols["last_stage_words"] == 16).any()
    assert (cols["segs"] > 1).any()


def test_repair_segments(probe):
    """segs = min(ceil(8 SMs / tiles), max(1, floor(avg rows / 256)), 64), and the walk of the longest genome: ceil(rows / segs)
    rows in one counter pass per 32,760 rows."""
    req = [(t, 1000, s, a * N_GENOMES, N_GENOMES, m) for t in (1, 2, 7, 148, 149, 591, 592, 593, 1183, 1184, 1185, 8192)
           for s in SMS for a in (0, 1, 255, 256, 512, 767, 768, 16_383, 16_384, 10**6) for m in (0, 1, 32_760, 32_761, 65_520, 65_521, 10**6)]
    _, c = probe.plans(req)
    t, s, a = c["n_tiles"], c["sm_count"], c["n_dropped"] // c["n_genomes"]
    want = np.minimum(np.minimum(-(-8 * s // t), np.maximum(1, a // 256)), 64)
    assert np.array_equal(c["segs"], want)
    assert np.array_equal(c["walk_rows"], -(-c["max_rows"] // c["segs"]))
    assert np.array_equal(c["walk_passes"], np.maximum(1, -(-c["walk_rows"] // 32_760)))


def test_pairwise_launches():
    """run_pairwise's launches as tests/ibs_plan_probe.py restates them: the whole matrix in upper-tile launches of at most
    8,192 tiles while the result takes at most 2 GiB, otherwise slabs of whole tile rows (at most 1 GiB and 8,192 tiles)."""
    assert IP.pairwise_launches(3_000, 0, 3_000, 16) == [1_128]
    assert IP.pairwise_launches(8_128, 0, 8_128, 16) == [8_128]
    assert IP.pairwise_launches(8_200, 0, 8_200, 16) == [8_192, 193]          # 8,385 upper tiles
    assert IP.pairwise_launches(8_200, 1, 8_200, 16) == [8_127, 8_127, 387]   # 63 tile rows of 129 per slab
    assert IP.pairwise_launches(8_200, 0, 8_200, 8) == [8_192, 193]
    assert IP.pairwise_launches(12_000, 0, 12_000, 16) == [43 * 188] * 4 + [16 * 188]      # > 2 GiB: slabs of 43 tile rows
    for n, r0, r1, b in ((8_200, 1, 8_200, 16), (12_000, 0, 12_000, 16), (40_000, 500, 9_000, 8)):
        side = IP.side(n)
        launches = IP.pairwise_launches(n, r0, r1, b)
        assert all(x % side == 0 and x <= 8192 for x in launches)
        assert sum(launches) // side == -(-r1 // 64) - r0 // 64


# Runs of the GPU tests at 148 SMs (the B200): (name, n_tiles, n_loci, n_dropped, n_genomes, max_rows) -> (n_chunks,
# stages_per_chunk, last_chunk_words, last_stage_words, grid, max units per CTA, segs, walk_passes). tests/test_gpu_ibs_plans.py
# derives its shapes from the probe on the device it runs on; on a B200 they are these, and a planner change that moves one of
# them off its regime fails here first.
REGIMES_148 = [
    # >= 3 multi-stage units per CTA, split, unequal last chunk, partial last stage (whole matrix of 1,100 genomes, saturated)
    ("saturated 1,100 x 25,000", IP.upper_tiles(1_100), 25_000, 0, 1_100, 0, (3, 17, 238, 14, 148, 4, 1, 1)),
    # SMs + 1 one-chunk units: CTA 0 runs two and stores both
    ("SMs + 1 units, 3,000 loci", 149, 3_000, 0, 1_067, 0, (1, 6, 94, 14, 148, 2, 1, 1)),
    # a split whose last stage holds 2 words (498 words)
    ("last stage 2 words, 250 x 15,931", IP.upper_tiles(250), 15_931, 0, 250, 0, (2, 16, 242, 2, 20, 1, 1, 1)),
    # the repair: segs > 1 with one chunk (the J plane cleared by the 2-D memset), segs > 1 split, a counter flush inside each
    # of two segments (split J), two flushes in one segment (stored J, then added)
    ("repair segs 2, one chunk", 592, 40_000, 140_800, 256, 4_400, (1, 79, 1_250, 2, 148, 4, 2, 1)),
    ("repair segs 2, split", 593, 40_000, 140_800, 256, 4_400, (2, 40, 610, 2, 148, 9, 2, 1)),
    ("repair flush, segs 2", 4, 70_000, 76_000, 128, 66_000, (8, 18, 172, 12, 32, 1, 2, 2)),
    ("repair flushes, segs 1", 1_184, 70_000, 76_000, 128, 66_000, (1, 137, 2_188, 12, 148, 8, 1, 3)),
    # slab drivers over 8,200 genomes x 300 loci: the first launch of the whole matrix, its second, one band slab of 63 tile rows
    ("8,200 x 300, 8,192 tiles", 8_192, 300, 0, 8_200, 0, (1, 1, 10, 10, 148, 56, 1, 1)),
    ("8,200 x 300, 193 tiles", 193, 300, 0, 8_200, 0, (1, 1, 10, 10, 148, 2, 1, 1)),
    ("8,200 x 300, band slab", 8_127, 300, 0, 8_200, 0, (1, 1, 10, 10, 148, 55, 1, 1)),
    # tests/test_gpu_gram_plans.py::test_king_band_mirrored_blocks_saturated: 2 tile rows of 19,160 genomes x 30,000 loci with
    # code 3 too dense to index, so IBS runs here with the validity plane: split, 9 units per CTA
    ("KING band 19,160 x 30,000", 2 * IP.side(19_160), 30_000, 0, 19_160, 0, (2, 30, 458, 10, 148, 9, 1, 1)),
    # the widest IBS / KING runs of the other GPU tests, on the popcount kernel when the tensor cores are off
    ("3,000 x 400", IP.upper_tiles(3_000), 400, 0, 3_000, 0, (1, 1, 14, 14, 148, 8, 1, 1)),
    ("2,504 x 40,000", IP.upper_tiles(2_504), 40_000, 0, 2_504, 0, (1, 79, 1_250, 2, 148, 6, 1, 1)),
]


@pytest.mark.parametrize("name,n_tiles,n_loci,n_dropped,n_genomes,max_rows,want", REGIMES_148, ids=[r[0] for r in REGIMES_148])
def test_plan_regimes_at_148_sms(probe, name, n_tiles, n_loci, n_dropped, n_genomes, max_rows, want):
    p = probe.plan(n_tiles, n_loci, 148, n_dropped, n_genomes, max_rows)
    got = tuple(p[f] for f in ("n_chunks", "stages_per_chunk", "last_chunk_words", "last_stage_words", "grid", "max_units_per_cta",
                               "segs", "walk_passes"))
    assert got == want, IP.describe(name, p)
