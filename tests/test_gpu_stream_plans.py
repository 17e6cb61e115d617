"""The streaming count pass at every launch plan, across its counter flushes, against the CPU oracle.

Every per-genome count goes through the V role of k_stream_count_ct<8,256>, k_stream_count_ct<40,64> or k_stream_count_rt,
whose 12-level bit-sliced counters hold at most 4,095 rows: every `flush_stages` stages of a CTA (a chunk) they are expanded
into the CTA's shared counts. Each case here sizes its loci with the planner (tests/stream_plan_probe.cu) on this device's SM
count so that its CTAs run the chunks it names, asserts that plan, and prints it:
  * the flush boundary on the cheapest plan (k_stream_count_rt, R = 256): a CTA of exactly one full chunk, one chunk and
    one stage, two full chunks, two chunks and one stage (both code-3 regimes: indexed, and too many cells to index), and a
    grid whose last CTA and last stage are short;
  * one case per kernel / stage height / V row-lane regime (tests/test_stream_plan.py pins the table), each with two chunks
    or more, populations mixed inside every 32-genome word and a windowed, spaced or AF-filtered selection, so the stage
    summary takes both its uniform and its masked branch and the V role its partial-mask branch;
  * saturated content in several of them: in every row 32 genomes are code 1 and 32 are code 2, so one lo and one hi plane
    word are all ones for every row of every chunk. Their counts are known without the oracle (L each), and a chunk longer
    than the counter holds, or a missing flush, loses 4,096 of them.
Per-locus and per-genome allele counts (the raw path: every row, one population) and the class counts are compared bit for
bit, the expected sums and F at the tolerances of test_gpu_baseline_sizes.py; RitlandLocus on the compile-time shapes.
The oracle adds its per-genome sums with compensation here (oracle_py.inbreed(compensated=True)): the device's sums are
fixed-point and exact at these sizes, while the reference's order -- double, locus by locus -- drifts by up to one rounding
per locus; over the 3.6 M selected rows of the smallest flush case that moves an expected sum by 5e-5 and F by 1e-10.
Populations are generated on the device and downloaded; only saturated ones are uploaded again.

Then the resident pass: back-to-back kgl_b200_enqueue_count_and_inbreed calls on a torch side stream with alternating
selections, closed by kgl_b200_run_count_and_inbreed (the double-buffered preparation and per-CTA counts of the timed step),
and kgl_b200_inbreed_fetch after a resident pass on a fresh context and after an iterative estimator."""
import numpy as np
import pytest

import oracle_py as O
import stream_plan_probe as SP
from conftest import results_matrix

pytestmark = pytest.mark.gpu

SEED = 20261020
# one 128-bit unit (64 genomes): lo plane bytes 0..7, hi plane bytes 8..15 -- genomes 0..31 code 1, genomes 32..63 code 2
SAT_UNIT = np.array([0xFF] * 4 + [0] * 8 + [0xFF] * 4, dtype=np.uint8)


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)) if a.size else 0.0


def assert_results_equal(got, want, what):
    c_got, f_got = results_matrix(got)
    c_want, f_want = results_matrix(want)
    assert np.array_equal(c_got, c_want), what
    assert rel_err(f_got[:, :3], f_want[:, :3]) < 1e-9, what
    a, b = got["inbred_allele_sum"], want["inbred_allele_sum"]
    assert np.array_equal(np.isfinite(a), np.isfinite(b)), what
    fin = np.isfinite(b)
    if fin.any():
        err = np.max(np.abs(a[fin] - b[fin]) / np.maximum(np.abs(b[fin]), 1e-3))
        assert err < 1e-8, (what, err)


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.close()


def loci_for(n_genomes, sms, stages, short=False):
    """Loci whose plan gives every CTA `stages(flush_stages)` stages; short: the last CTA owns flush_stages + 1 of them and its
    last stage is partial. Returns (loci, plan)."""
    units = SP.units_of(n_genomes)
    wave = SP.plan(units, 80_000_000, sms)              # a full wave of CTAs: n_ctas = SMs / slices
    fs, ctas, R = wave["flush_stages"], wave["n_ctas"], wave["rows_per_stage"]
    spc = stages(fs)
    loci = (spc * (ctas - 1) + fs + 1) * R - 37 if short else spc * ctas * R
    p = SP.plan(units, loci, sms)
    assert p["stages_per_cta"] == spc, p
    if short:
        assert p["total_stages"] - (p["n_ctas"] - 1) * spc == fs + 1 and loci % R != 0, p
    return loci, p


def describe(name, p):
    kernel = {0: "k_stream_count_rt", 1: "k_stream_count_ct<40,64>", 2: "k_stream_count_ct<8,256>"}[p["shape"]]
    return (f"{name}: {kernel} x {p['slices']} slice(s), L {p['n_loci']}, R {p['rows_per_stage']}, v_row_lanes {p['v_row_lanes']}, "
            f"{p['n_ctas']} CTAs x {p['stages_per_cta']} stages, flush_stages {p['flush_stages']}, chunks_per_cta {p['chunks_per_cta']}")


def selection(kind, offsets):
    """select_loci keywords: 'window' (uniform stages inside, none outside), 'af' (rows selected for some populations only),
    'spaced' (every third locus), 'window_af' (both)."""
    n = offsets.shape[0]
    window = dict(lower=int(offsets[n // 8]), upper=int(offsets[n - n // 8]))
    af = dict(min_af=0.02, max_af=0.9)
    return {"window": window, "af": af, "spaced": dict(spacing=25), "window_af": {**window, **af}}[kind]


def population(gpu, n, offsets, af, missing_rate, sat_at=None, grouped=False):
    """Generated on the device, downloaded (the oracle's input); a saturated 64-genome block at genome `sat_at` is written
    into the host copy, which is then uploaded."""
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes
    superpop, f = make_genomes(n, SEED, grouped=grouped)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.set_unphased(False)
    gpu.synth_genotypes(SEED, n, offsets.shape[0], f, missing_rate=missing_rate)
    pop = FlatPopulation(offsets, af, superpop, gpu.download_genotypes(), n, False)
    if sat_at is not None:
        assert sat_at % 64 == 0 and sat_at + 64 <= n
        pop.packed[:, sat_at // 4: sat_at // 4 + 16] = SAT_UNIT
        gpu.upload_population(pop)
    return pop


def oracle_genomes(n, sat_at):
    """The genomes the estimators are checked on: the edges of the saturated block and about 48 others."""
    some = np.arange(0, n, max(1, n // 48))
    if sat_at is not None:
        some = np.concatenate([some, sat_at + np.array([0, 1, 31, 32, 33, 63])])
    return np.unique(some).astype(np.int64)


def check_counting(gpu, pop, sel_kw, sat_at=None, ritland=False, code3_indexed=None):
    n, L = pop.n_genomes, pop.n_loci
    olc, ogc = O.allele_count(pop)
    if code3_indexed is not None:
        # the library indexes the code-3 cells when there are at most max(2^16, N L / 64) of them (finish_dropped_index);
        # otherwise the pass sums the CTAs' counts with k_sum_cta_counts and scans the matrix with k_dropped_scan
        n3 = int(ogc[:, 3].sum())
        assert (n3 <= max(1 << 16, n * L // 64)) == code3_indexed, n3
    # raw path: every row, one population
    lc, gc = gpu.allele_count()
    if sat_at is not None:
        assert np.all(gc[sat_at:sat_at + 32] == [0, L, 0, 0]), gc[sat_at:sat_at + 32, 1].min()
        assert np.all(gc[sat_at + 32:sat_at + 64] == [0, 0, L, 0]), gc[sat_at + 32:sat_at + 64, 2].min()
    assert np.array_equal(lc, olc)
    assert np.array_equal(gc, ogc)
    # the selected rows of each genome's population
    gpu.select_loci(**sel_kw)
    sel = O.select_all_pops(pop, **sel_kw)
    some = oracle_genomes(n, sat_at)
    lc2, res = gpu.count_and_inbreed()
    assert np.array_equal(lc2, olc)
    assert_results_equal(res[some], O.inbreed(pop, sel, "Simple", genomes=some, compensated=True), "Simple")
    if ritland:
        assert_results_equal(gpu.inbreed("RitlandLocus")[some], O.inbreed(pop, sel, "RitlandLocus", genomes=some, compensated=True),
                              "RitlandLocus")


# ----------------------------------------------------------------------------------- flush boundary, rt R = 256 ----
# 128 genomes: the saturated block (genomes 0..63) and 64 random genomes of the five super-populations in turn
FLUSH_GENOMES = 128
FLUSH_CASES = [
    # name, stages per CTA from flush_stages, short last CTA, code-3 rate of the random genomes, selection, chunks per CTA
    ("one-full-chunk", lambda fs: fs, False, 0.001, "window", 1),
    ("chunk-plus-one-stage", lambda fs: fs + 1, False, 0.001, "af", 2),
    ("two-full-chunks", lambda fs: 2 * fs, False, 0.001, "spaced", 2),
    ("two-chunks-plus-one-stage-indexed", lambda fs: 2 * fs + 1, False, 0.001, "window_af", 3),
    ("two-chunks-plus-one-stage-not-indexed", lambda fs: 2 * fs + 1, False, 0.05, "window_af", 3),
    ("short-last-cta", lambda fs: 2 * fs + 1, True, 0.001, "af", 3),
]


@pytest.fixture(scope="module")
def flush_loci(sms):
    """Offsets and frequencies for the longest flush case; every case takes a prefix."""
    from kgl_gene_b200.synth import make_loci
    longest = max(loci_for(FLUSH_GENOMES, sms, c[1], c[2])[0] for c in FLUSH_CASES)
    return make_loci(longest, SEED)


@pytest.mark.parametrize("name,stages,short,missing_rate,sel_kind,chunks", FLUSH_CASES, ids=[c[0] for c in FLUSH_CASES])
def test_flush_boundary(gpu, sms, flush_loci, name, stages, short, missing_rate, sel_kind, chunks):
    L, p = loci_for(FLUSH_GENOMES, sms, stages, short)
    print(describe(name, p))
    assert p["shape"] == 0 and p["rows_per_stage"] == 256 and p["chunks_per_cta"] == chunks
    offsets, af = flush_loci
    offsets, af = offsets[:L], np.ascontiguousarray(af[:, :L])
    pop = population(gpu, FLUSH_GENOMES, offsets, af, missing_rate, sat_at=0)
    check_counting(gpu, pop, selection(sel_kind, offsets), sat_at=0, code3_indexed=missing_rate < 0.01)


# ------------------------------------------------------------------------------ one case per kernel regime ----
REGIME_CASES = [
    # name, genomes, (shape, R, rows per V thread, slices), saturated block, selection, RitlandLocus
    ("rt-R128", 700, (0, 128, 32, 1), None, "af", False),
    ("rt-R64", 1300, (0, 64, 32, 1), None, "spaced", False),
    ("rt-R64-one-row-lane", 2600, (0, 64, 64, 1), 1280, "window", False),
    ("ct8x256", 500, (2, 256, 32, 1), 0, "af", True),
    ("ct40x64", 2504, (1, 64, 32, 1), None, "window_af", True),
    ("ct40x64-two-slices", 4100, (1, 64, 32, 2), 2560, "spaced", False),
]


@pytest.mark.parametrize("name,n,regime,sat_at,sel_kind,ritland", REGIME_CASES, ids=[c[0] for c in REGIME_CASES])
def test_kernel_regime_over_two_chunks(gpu, sms, name, n, regime, sat_at, sel_kind, ritland):
    from kgl_gene_b200.synth import make_loci
    L, p = loci_for(n, sms, lambda fs: fs + 4)          # a full chunk and one of four stages
    print(describe(name, p))
    shape, R, rows_v, slices = regime
    assert (p["shape"], p["rows_per_stage"], p["rows_per_stage"] // p["v_row_lanes"], p["slices"]) == regime
    assert p["chunks_per_cta"] >= 2
    offsets, af = make_loci(L, SEED + n)
    pop = population(gpu, n, offsets, af, 0.001, sat_at=sat_at)
    check_counting(gpu, pop, selection(sel_kind, offsets), sat_at=sat_at, ritland=ritland)


# ------------------------------------------------------------------------- back-to-back resident passes ----
CHAIN_GENOMES = 2504
CHAIN_SELECTIONS = [dict(), dict(spacing=25)]


@pytest.fixture(scope="module")
def chain_population(sms):
    """The bench width (2,504 genomes, grouped super-populations, k_stream_count_ct<40,64>) with two chunks per CTA, and the
    oracle's results for both selections."""
    from kgl_gene_b200.capi import KglB200
    from kgl_gene_b200.synth import make_loci
    L, p = loci_for(CHAIN_GENOMES, sms, lambda fs: fs + 4)
    print(describe("resident chain", p))
    assert p["shape"] == 1 and p["slices"] == 1 and p["chunks_per_cta"] >= 2
    offsets, af = make_loci(L, SEED + 1)
    ctx = KglB200(0)
    try:
        pop = population(ctx, CHAIN_GENOMES, offsets, af, 0.001, grouped=True)
        some = oracle_genomes(CHAIN_GENOMES, None)
        want = [O.inbreed(pop, O.select_all_pops(pop, **kw), "Simple", genomes=some, compensated=True)
                for kw in CHAIN_SELECTIONS]
        yield ctx, pop, some, want, O.allele_count(pop)[0]
    finally:
        ctx.close()


@pytest.mark.parametrize("k", [1, 2, 5])
def test_back_to_back_resident_passes(chain_population, k):
    """k resident passes with alternating selections (select_loci and nothing else between them) on a torch side stream, then
    the one-call pass: its results and the locus counts are those of the last selection."""
    import torch
    ctx, pop, some, want, olc = chain_population
    stream = torch.cuda.Stream(priority=-1)
    ctx.set_stream(stream.cuda_stream)
    try:
        with torch.cuda.stream(stream):
            for i in range(k):
                ctx.select_loci(**CHAIN_SELECTIONS[i % 2])
                ctx.enqueue_count_and_inbreed()
            ctx.select_loci(**CHAIN_SELECTIONS[k % 2])
            _, res = ctx.count_and_inbreed(want_loci=False)
            lc = ctx.fetch_locus_counts()
            fetched = ctx.inbreed_fetch()
    finally:
        ctx.set_stream(None)
    assert_results_equal(res[some], want[k % 2], ("k", k))
    assert np.array_equal(lc, olc)
    assert fetched.tobytes() == res.tobytes()


# ------------------------------------------------------------------------- kgl_b200_inbreed_fetch after a resident pass ----
@pytest.mark.parametrize("before", [None, "HallME", "Loglikelihood"])
def test_inbreed_fetch_after_resident_pass(before):
    """kgl_b200_inbreed_fetch returns the resident pass's Simple results on a fresh context and after an iterative estimator
    (whose coefficient must not be stored over them)."""
    from kgl_gene_b200.capi import KglB200
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(300, 20_000, seed=91, missing_rate=0.002)
    sel = O.select_all_pops(pop, spacing=15)
    want = O.inbreed(pop, sel, "Simple", compensated=True)
    ctx = KglB200(0)
    try:
        ctx.upload_population(pop)
        ctx.select_loci(spacing=15)
        if before is not None:
            other = ctx.inbreed(before)
            assert np.nanmax(np.abs(other["inbred_allele_sum"] - want["inbred_allele_sum"])) > 1e-6    # a different estimate
        ctx.enqueue_count_and_inbreed()
        got = ctx.inbreed_fetch()
        assert_results_equal(got, want, before)
        assert np.array_equal(ctx.fetch_locus_counts(), O.allele_count(pop)[0])
    finally:
        ctx.close()
