"""The launch planner of the tensor-core Gram kernel (plan_gram, kgl_gene_b200/csrc/gram_launch.cuh), compiled as a host
program (tests/gram_plan_probe.cu) and checked without a GPU.

k_gram_i8 runs units of (256 x 256 tile, chunk of K) round-robin over its CTAs; the expanders and the MMA warp each derive a
unit's stage count as min(stages_per_chunk, k_stages - chunk * stages_per_chunk). A chunk with no stage would never commit
the accumulator barrier and the kernel would hang; a unit index past 2^32 would wrap in the kernel's uint32_t arithmetic; a
wrong split would only show on a large input. This sweep checks the plan of tile counts from 1 to 80,000 (a 100,000-genome
run_gram has 76,636 tiles) at k-stage counts around every boundary of the planner and on several SM counts.
tests/test_gpu_gram_plans.py runs the kernel at the plans pinned by test_plan_regimes_at_148_sms."""
import numpy as np
import pytest

import gram_plan_probe as GP

SMS = (1, 2, 132, 148, 160)
# k-stages: around the split threshold (64 stages = 8,192 loci per chunk), splits whose last chunk is 1 or 2 stages on few
# tiles (4,097 / 4,161 / 4,162), config 2 (1.1 M loci), 2,048 chunks of 64 stages, config 4 (20 M loci) and 2^22 - 1 (just under
# 2^29 loci, the int32 limit of the accumulators)
K_STAGES = sorted({k + d for k in (1, 63, 64, 127, 128, 129, 4_097, 4_161, 8_594, 131_072, 156_250) for d in (-1, 0, 1) if k + d >= 1}
                  | {(1 << 22) - 2, (1 << 22) - 1})
N_TILES = np.unique(np.concatenate([np.arange(1, 2049), np.geomspace(2049, 80_000, 300).astype(np.int64), [76_636, 80_000]]))


@pytest.fixture(scope="module")
def probe():
    try:
        GP.probe_binary()
    except FileNotFoundError:
        pytest.skip("nvcc is not installed")
    return GP


def violations(c):
    """name -> boolean array of the plans that break the invariant (planner's own choice, no hint)."""
    sp, nc, k = c["stages_per_chunk"], c["n_chunks"], c["k_stages"]
    return {
        "1 <= n_chunks <= 2048": (nc < 1) | (nc > 2048),
        "chunks cover K": nc * sp < k,
        "no empty chunk": (nc - 1) * sp >= k,
        "last chunk as stated": c["last_stages"] != k - (nc - 1) * sp,
        ">= 64 stages per chunk when split": (nc > 1) & (sp < 64),
        "one chunk below 128 stages": (k < 128) & (nc != 1),
        "grid = min(units, SMs)": c["grid"] != np.minimum(c["units"], c["sm_count"]),
        "grid >= 1": c["grid"] < 1,
        "units = tiles x chunks": c["units"] != c["n_tiles"] * nc,
        "unit index fits uint32": c["units"] >= 1 << 32,
        "units per CTA": c["max_units_per_cta"] != -(-c["units"] // c["grid"]),
    }


def assert_no_violation(cols, checks):
    bad = {name: np.flatnonzero(m) for name, m in checks.items() if m.any()}
    if bad:
        lines = []
        for name, idx in bad.items():
            i = int(idx[0])
            lines.append(f"{name}: {idx.size} plans, e.g. " + ", ".join(f"{f}={int(v[i])}" for f, v in cols.items()))
        pytest.fail("\n".join(lines))


def test_plan_invariants_over_the_sweep(probe):
    """Tiles 1..2,048 and 300 more up to 80,000 x 39 k-stage counts x 5 SM counts (~450,000 plans): none may break an
    invariant (none did when this was written)."""
    req = [(t, k, s) for t in N_TILES for k in K_STAGES for s in SMS]
    consts, cols = probe.plans(req)
    assert (consts["ring"], consts["tile"], consts["stage_loci"]) == (3, 256, 128)
    assert cols["n_tiles"].size == len(req)
    assert_no_violation(cols, violations(cols))
    # the sweep reaches every regime the kernel has: one chunk, split-K, several units per CTA, a
    # last chunk of one and of two stages (shorter than the 3-deep stage ring)
    nc = cols["n_chunks"]
    assert (nc == 1).any() and nc.max() > max(SMS)
    assert cols["max_units_per_cta"].max() >= 3
    assert ((nc > 1) & (cols["max_units_per_cta"] >= 2)).any()
    for last in (1, 2):
        assert ((nc > 1) & (cols["last_stages"] == last)).any(), last


@pytest.mark.parametrize("sms", SMS)
def test_short_last_chunk_where_it_occurs(probe, sms):
    """Every k-stage count from 128 to 20,000 on one and on two tiles: a split whose last chunk is shorter than the stage ring
    needs ceil(K / c) to round the chunk count down, which happens only from ~4,096 stages (64 chunks of >= 64 stages) -- the
    GPU cases search this range for theirs."""
    req = [(t, k, sms) for t in (1, 2) for k in range(1, 20_001)]
    _, cols = probe.plans(req)
    assert_no_violation(cols, violations(cols))
    short = (cols["n_chunks"] > 1) & (cols["last_stages"] < 3)
    if sms >= 64:
        assert short.any()
        assert cols["k_stages"][short].min() >= 4_000


@pytest.mark.parametrize("hint", [1, 2, 3, 63, 64, 65, 1000, 8_594])
def test_chunk_hint_is_honoured(probe, hint):
    """chunk_stages_hint (tools: grambench) overrides the search: chunks of at most `hint` stages, ceil(K / hint) of them, none
    empty."""
    ks = [k for k in K_STAGES if k <= 200_000] + [hint - 1, hint, hint + 1, 3 * hint + 1]
    req = [(t, k, s, hint) for t in (1, 7, 153, 5000) for k in ks if k >= 1 for s in (1, 148)]
    _, c = probe.plans(req)
    assert np.all(c["hint"] == hint)
    sp, nc, k = c["stages_per_chunk"], c["n_chunks"], c["k_stages"]
    assert np.all(sp <= hint)
    assert np.all(nc == -(-k // hint))
    assert np.all(((nc - 1) * sp < k) & (k <= nc * sp))
    assert np.all(c["grid"] == np.minimum(c["units"], c["sm_count"]))


# Runs of the GPU tests at 148 SMs (the B200): (name, n_tiles, k_stages) -> (n_chunks, stages_per_chunk, last, grid,
# max units per CTA). tests/test_gpu_gram_plans.py derives its shapes from the probe on the device it runs on; on a B200 they
# are these, and a planner change that moves one of them off its regime fails here first.
REGIMES_148 = [
    # test_gpu_pca.py::test_product_bit_equal, 20,000 genomes x 700 loci, 48 columns: pass 1 split-K, pass 2 two units per CTA
    ("PCA pass 1 (20,000 x 700)", GP.pca_tiles(20_000, 700, 48)[0], GP.k_stages(20_000), 2, 79, 78, 18, 1),
    ("PCA pass 2 (20,000 x 700)", GP.pca_tiles(20_000, 700, 48)[1], GP.k_stages(700), 1, 6, 6, 148, 2),
    # test_gpu_king.py::test_king_modes_and_edges, 600 x 20,000: 6 blocks (3 per side), the M run split in two
    ("KING 600 x 20,000", 6, GP.k_stages(20_000), 2, 79, 78, 12, 1),
    # test_gpu_gram_plans.py: a last chunk of 1 and of 2 stages on one tile / one block (532,557 and 524,365 loci)
    ("last chunk 1 stage", 1, 4_161, 65, 65, 1, 65, 1),
    ("last chunk 2 stages", 1, 4_097, 64, 65, 2, 64, 1),
    # units = SMs + 1, one chunk (enqueue_gram_tiles: every 4th of the 595 tiles of 8,685 genomes, 3,000 loci)
    ("SMs + 1 units", 149, GP.k_stages(3_000), 1, 24, 24, 148, 2),
    # KING band over 75 blocks (19,160 genomes) x 30,000 loci: 3 chunks of unequal length, 2 units per CTA, mirrored blocks
    ("KING band 75 blocks", 75, GP.k_stages(30_000), 3, 79, 77, 148, 2),
    # run_gram over 17 x 17 blocks (4,315 genomes) x 40,013 loci: 5 multi-stage units per CTA, 4 chunks of unequal length
    ("Gram 4,315 x 40,013", GP.upper_tiles(4_315), GP.k_stages(40_013), 4, 79, 76, 148, 5),
]


@pytest.mark.parametrize("name,n_tiles,k_stages,n_chunks,sp,last,grid,per_cta", REGIMES_148, ids=[r[0] for r in REGIMES_148])
def test_plan_regimes_at_148_sms(probe, name, n_tiles, k_stages, n_chunks, sp, last, grid, per_cta):
    p = probe.plan(n_tiles, k_stages, 148)
    assert (p["n_chunks"], p["stages_per_chunk"], p["last_stages"], p["grid"], p["max_units_per_cta"]) == (n_chunks, sp, last, grid, per_cta), \
        GP.describe(name, p)
