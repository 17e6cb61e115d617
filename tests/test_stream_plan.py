"""The launch planner of the streaming pass (plan_stream, kgl_gene_b200/csrc/stream_common.cuh), compiled as a host program
(tests/stream_plan_probe.cu) and checked without a GPU.

Every per-genome count the library returns goes through the V role of the streaming kernels, whose 12-level bit-sliced
counters hold at most 4,095 rows; every `flush_stages` stages they are expanded into the CTA's shared counts. A plan that lets
more rows than that into one chunk, or a V mapping that needs more threads than the kernel has, would be wrong only on inputs
large or wide enough to reach it. This sweep checks the plan of every width up to 8,000 units (512,000 genomes) at loci
counts around every stage, chunk and flush boundary and on several SM counts. tests/test_gpu_stream_plans.py runs the
kernels at the plans pinned by test_plan_regimes_at_148_sms."""
import numpy as np
import pytest

import stream_plan_probe as SP

SMEM_LIMIT = 227 * 1024          # dynamic shared memory of one block on sm_100
SMS = (1, 2, 132, 148, 160)
FIXED_LOCI = (1, 63, 64, 65, 255, 256, 257, 4096, 1_100_000, 20_000_000, 80_000_000)
MAX_UNITS = 8000


@pytest.fixture(scope="module")
def probe():
    try:
        SP.probe_binary()
    except FileNotFoundError:
        pytest.skip("nvcc is not installed")
    return SP


def flush_boundaries(cols):
    """Per row of a large-L plan: the loci at which a CTA's stages reach k * flush_stages (k = 1, 2), and one row either side."""
    step = cols["flush_stages"] * cols["n_ctas"] * cols["rows_per_stage"]
    return [(k * step + d, k, d) for k in (1, 2) for d in (-1, 0, 1)]


def violations(consts, c):
    """name -> boolean array of the rows that break the invariant."""
    R, rl = c["rows_per_stage"], c["v_row_lanes"]
    rows_per_v = R // rl
    max_rows = (1 << consts["levels"]) - 1
    return {
        "R is 64, 128 or 256": ~np.isin(R, (64, 128, 256)),
        "rows per V thread a multiple of 8": (R % rl != 0) | (rows_per_v % 8 != 0),
        "a chunk fits the counter": c["flush_stages"] * rows_per_v > max_rows,
        "a chunk fits the counter's call budget": c["flush_stages"] * (rows_per_v // 8) > consts["max_calls"],
        "flush_stages >= 1": c["flush_stages"] < 1,
        "chunks cover the CTA's stages": c["chunks_per_cta"] != -(-c["stages_per_cta"] // np.maximum(c["flush_stages"], 1)),
        "smem within one block": c["smem"] > SMEM_LIMIT,
        "threads within one block": c["threads"] > 1024,
        "ring depth": (c["n_stages"] < 2) | (c["n_stages"] > consts["max_stages"]),
        "pitch covers the row": c["units_padded"] < c["units"],
        "slices cover the pitch": c["slices"] * c["slice_units"] < c["units_padded"],
        "compile-time shapes: pitch a multiple of the slice": (c["shape"] != 0) & (c["units_padded"] % np.maximum(c["slice_units"], 1) != 0),
        "compile-time shapes: their slice widths": ((c["shape"] == 1) & ((c["slice_units"] != 40) | (R != 64)))
                                                   | ((c["shape"] == 2) & ((c["slice_units"] != 8) | (R != 256))),
        "rows cover the loci": c["padded_rows"] < c["n_loci"],
        "rows fit the device matrix (loci padded to 256)": c["padded_rows"] > (c["n_loci"] + 255) // 256 * 256,
        "CTAs cover the stages": c["n_ctas"] * c["stages_per_cta"] < c["total_stages"],
        "no CTA without a stage": (c["n_ctas"] - 1) * c["stages_per_cta"] >= c["total_stages"],
        "one wave where the SMs allow": c["n_ctas"] * c["slices"] > np.maximum(c["sm_count"], c["slices"]),
        "H role covers the row": (c["h_parts"] * R != 256) | (c["h_parts"] * c["h_units"] < c["slice_units"]),
        "A | B << 16 does not carry": c["slice_units"] * 64 >= 65536,
        "runtime shape: V mapping fits the consumer warps": (c["shape"] == 0) & (4 * c["slice_units"] * rl > consts["consumer_threads"]),
        "runtime shape: slice within the shared-memory stage": (c["shape"] == 0) & (c["slice_units"] > consts["max_slice_units"]),
    }


def assert_no_violation(consts, cols):
    bad = {name: np.flatnonzero(m) for name, m in violations(consts, cols).items() if m.any()}
    if bad:
        lines = []
        for name, idx in bad.items():
            i = int(idx[0])
            lines.append(f"{name}: {idx.size} plans, e.g. " + ", ".join(f"{f}={int(v[i])}" for f, v in cols.items()))
        pytest.fail("\n".join(lines))


def test_plan_invariants_over_the_sweep(probe):
    """Every width of 1..8,000 units x every SM count x loci from one row to 80 M, plus the loci one row either side of the
    first and second flush boundary of each width: 680,000 plans, none may break an invariant (none did when this was
    written)."""
    units = np.arange(1, MAX_UNITS + 1)
    req = [(u, l, s) for u in units for s in SMS for l in FIXED_LOCI]
    consts, cols = probe.plans(req)
    assert consts["levels"] == 12
    assert_no_violation(consts, cols)
    # the boundaries follow from the 80 M plan of each (width, SM count): the CTAs are one wave there
    big = cols["n_loci"] == FIXED_LOCI[-1]
    big_cols = {f: v[big] for f, v in cols.items()}
    assert np.all(big_cols["n_ctas"] == np.maximum(1, big_cols["sm_count"] // big_cols["slices"]))
    bounds = flush_boundaries(big_cols)
    req2 = [(u, l, s) for b, _, _ in bounds for u, l, s in zip(big_cols["units"], b, big_cols["sm_count"])]
    _, cols2 = probe.plans(req2)
    assert_no_violation(consts, cols2)
    n = big_cols["units"].size
    for j, (_, k, d) in enumerate(bounds):
        chunks = cols2["chunks_per_cta"][j * n:(j + 1) * n]
        assert np.all(chunks == (k + 1 if d > 0 else k)), (k, d)      # the boundary is where the chunks change
    total = cols["units"].size + cols2["units"].size
    assert total == MAX_UNITS * len(SMS) * (len(FIXED_LOCI) + 6)
    # every kernel, stage height and row-lane count is in the sweep
    assert set(np.unique(cols["shape"])) == {0, 1, 2}
    assert set(np.unique(cols["rows_per_stage"])) == {64, 128, 256}
    assert set(np.unique(cols["v_row_lanes"])) >= {1, 2, 4, 8}
    assert cols["chunks_per_cta"].max() >= 3


# genomes -> (shape, R, rows per V thread, flush_stages, slices) at 148 SMs, and the loci above which a CTA runs two chunks
REGIMES_148 = [
    ("rt R=256", [g for g in range(1, 641) if not 449 <= g <= 512], 0, 256, 32, 127, 1, 4_811_776),
    ("rt R=128", range(641, 1281), 0, 128, 32, 127, 1, 2_405_888),
    ("rt R=64", range(1281, 2497), 0, 64, 32, 127, 1, 1_202_944),
    ("rt R=64 rl=1", range(2561, 3585), 0, 64, 64, 63, 1, 596_736),
    ("ct<8,256>", range(449, 513), 2, 256, 32, 127, 1, 4_811_776),
    ("ct<40,64>", range(2497, 2561), 1, 64, 32, 127, 1, 1_202_944),
    ("ct<40,64> x 2 slices", range(3585, 5121), 1, 64, 32, 127, 2, 601_472),
]


@pytest.mark.parametrize("name,genomes,shape,R,rows_v,flush,slices,two_chunks", REGIMES_148, ids=[r[0] for r in REGIMES_148])
def test_plan_regimes_at_148_sms(probe, name, genomes, shape, R, rows_v, flush, slices, two_chunks):
    """The kernel, stage height, V rows per thread and flush interval of every width at 148 SMs (the B200), and the loci at
    which a CTA first needs a second counter chunk."""
    units = sorted({SP.units_of(g) for g in genomes})
    _, c = probe.plans([(u, l, 148) for u in units for l in (two_chunks, two_chunks + 1)])
    assert np.all(c["shape"] == shape) and np.all(c["rows_per_stage"] == R) and np.all(c["slices"] == slices)
    assert np.all(c["rows_per_stage"] // c["v_row_lanes"] == rows_v) and np.all(c["flush_stages"] == flush)
    assert np.all(c["chunks_per_cta"] == np.tile([1, 2], len(units)))
    assert np.all(c["flush_stages"] * rows_v <= 4095)
