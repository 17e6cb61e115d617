"""GPU parity tests: every call goes through the C ABI (kgl_gene_b200/libkgl_b200.so) and is compared with
(a) the committed golden vectors produced by the reference's own code and (b) the CPU oracle on seeded inputs.
Integer results (allele counts, class counts, locus selection, IBS) must be bit-exact; floating-point results must
agree within 1e-6 relative (BASELINE.json north_star) -- the assertions below use far tighter bounds where the
arithmetic allows it."""
import os

import numpy as np
import pytest

import oracle_py as O
from conftest import results_matrix

pytestmark = pytest.mark.gpu

SUPER_POPS = ["AFR", "AMR", "EAS", "EUR", "SAS", "ALL"]
REL = 1e-6          # the contract
TIGHT = 1e-11       # what double arithmetic in a different summation order actually gives


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.close()


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)) if a.size else 0.0


def sel_bits(sel):   # uint8 [6, L] -> bit mask per locus
    return np.bitwise_or.reduce(sel.astype(np.uint8) << np.arange(sel.shape[0], dtype=np.uint8)[:, None], axis=0).astype(np.uint8)


# ---------------------------------------------------------------------------------------------- golden (reference) ----
def test_golden_locus_selection(gpu, golden):
    name, pop, ref, sel_kw = golden
    gpu.upload_population(pop)
    counts = gpu.select_loci(**sel_kw)
    bits = gpu.get_locus_selection()
    for k, sp in enumerate(SUPER_POPS):
        chosen = pop.offsets[(bits >> k) & 1 == 1]
        assert np.array_equal(chosen, ref["selected_offsets_" + sp]), (name, sp)
        assert counts[k] == len(ref["selected_offsets_" + sp])


def test_golden_simple_and_counts(gpu, golden):
    name, pop, ref, sel_kw = golden
    gpu.upload_population(pop)
    gpu.select_loci(**sel_kw)
    lc, res = gpu.count_and_inbreed()
    counts, freqs = results_matrix(res)
    present = ref["genome_present"] == 1
    assert np.array_equal(counts[present], ref["Simple_counts"][present])                 # bit-exact, MINOR_HETEROZYGOUS included
    assert rel_err(freqs[present][:, :3], ref["Simple_freqs"][present][:, :3]) < TIGHT
    if pop.n_multi:     # the sum over i < j of 2 p_i p_j at the multi-allelic loci (freq.cpp:166-174)
        assert np.all(ref["Simple_freqs"][present][:, 3] > 0) and rel_err(freqs[present][:, 3], ref["Simple_freqs"][present][:, 3]) < TIGHT
    else:
        assert np.all(freqs[:, 3] == 0.0)
    assert rel_err(res["inbred_allele_sum"][present], ref["Simple_coeff"][present]) < 1e-9
    # per-locus allele counts vs VariantDBVariant::summaryByVariant
    m = ref["variant_present"] == 1
    if pop.n_multi:     # one column per allele there: kgl_b200_run_multi_allele_count, slot 0 = the harness' "A>G" column
        mc = gpu.multi_allele_count(pop.n_multi)
        cells = pop.multi_cells.astype(np.int64)
        for a in range(3):
            copies = ((cells & 15) == a + 1).astype(np.int64) + ((cells >> 4) == a + 1).astype(np.int64)
            copies[cells == 0xFF] = 0
            for c in range(3):
                assert np.array_equal(mc[:, a, c], (copies == c).sum(axis=1))
        no3 = ~(cells == 0xFF).any(axis=1) & m[pop.multi_rows]
        assert np.array_equal(mc[no3, 0, 1], ref["summary_by_variant"][pop.multi_rows][no3, 1])
        assert np.array_equal(mc[no3, 0, 2], ref["summary_by_variant"][pop.multi_rows][no3, 2])
        m = m.copy(); m[pop.multi_rows] = False
    sv = ref["summary_by_variant"]
    assert np.array_equal(lc[m, 1], sv[m, 1]) and np.array_equal(lc[m, 2], sv[m, 2])
    assert np.array_equal((lc[m, 0] + lc[m, 3]).astype(np.uint64), sv[m, 0])


def test_golden_allele_count(gpu, golden):
    name, pop, ref, _ = golden
    gpu.upload_population(pop)
    lc, gc = gpu.allele_count()
    olc, ogc = O.allele_count(pop)
    assert np.array_equal(lc, olc) and np.array_equal(gc, ogc)
    if pop.n_multi:
        return          # summaryByGenome also runs over the per-allele columns of the multi-allelic loci
    sg = ref["summary_by_genome"]
    present = ref["genome_present"] == 1
    assert np.array_equal(sg[present, 1], gc[present, 1] + gc[present, 3]) and np.array_equal(sg[present, 2], gc[present, 2])


def test_golden_ritland(gpu, golden):
    name, pop, ref, sel_kw = golden
    gpu.upload_population(pop)
    gpu.select_loci(**sel_kw)
    res = gpu.inbreed("RitlandLocus")
    counts, freqs = results_matrix(res)
    present = ref["genome_present"] == 1
    assert np.array_equal(counts[present], ref["RitlandLocus_counts"][present])
    assert rel_err(res["inbred_allele_sum"][present], ref["RitlandLocus_coeff"][present]) < 1e-9


def test_golden_hallme_fifty_sweeps(gpu, golden):
    name, pop, ref, sel_kw = golden
    gpu.upload_population(pop)
    gpu.select_loci(**sel_kw)
    start = np.full(pop.n_genomes, ref["hall_start_sequence"][4])
    res = gpu.inbreed("HallME", hall_start=start, hall_sweeps=50)
    present = ref["genome_present"] == 1
    assert rel_err(res["inbred_allele_sum"][present], ref["HallME_coeff"][present]) < 1e-9


def test_golden_loglikelihood(gpu, golden):
    name, pop, ref, sel_kw = golden
    gpu.upload_population(pop)
    gpu.select_loci(**sel_kw)
    present = ref["genome_present"] == 1
    ll = gpu.loglik_grid(ref["ll_grid"])
    assert rel_err(ll[present], ref["ll_grid_values"][present]) < 1e-12
    res = gpu.inbreed("Loglikelihood")
    sel = O.select_all_pops(pop, **sel_kw)
    opt = O.inbreed(pop, sel, "Loglikelihood")["inbred_allele_sum"]
    # converged optimum of the same objective: <= 1e-9 (SURVEY 8c); the reference's own Nelder-Mead stops at xtol 1e-6
    assert np.max(np.abs(res["inbred_allele_sum"][present] - opt[present])) < 1e-9
    close = np.abs(res["inbred_allele_sum"][present] - ref["Loglikelihood_coeff"][present]) < 2e-6
    # multi_allelic_unphased: for two genomes the reference's Nelder-Mead ends outside the feasible region (see the waiver in
    # tests/test_oracle_vs_reference.py::test_loglikelihood_optimum_within_optimiser_tolerance)
    assert np.all(close) or (name == "multi_allelic_unphased" and close.sum() >= close.size - 2)


# ------------------------------------------------------------------------------------------------ oracle, seeded ----
CASES = [
    dict(n_genomes=300, n_loci=20000, seed=1, spectrum="sfs", grouped=True),
    dict(n_genomes=257, n_loci=9000, seed=2, spectrum="dense", grouped=False),             # mixed-population units
    dict(n_genomes=64, n_loci=4097, seed=3, spectrum="sfs", unphased=True),
    dict(n_genomes=1, n_loci=100, seed=4, spectrum="dense"),                                # single genome
    dict(n_genomes=2504, n_loci=3000, seed=5, spectrum="sfs", missing_rate=0.02, missing_af_rate=0.02),
    dict(n_genomes=130, n_loci=31, seed=6, spectrum="dense"),                               # fewer loci than one word
    # BASELINE config 1 width (449..512 genomes = 8 units: k_stream_count_ct<8,256>), phased and unphased (SURVEY 8d, Q6),
    # every row selected (even seeds: spacing 0) and a spaced, masked selection (odd seeds: spacing 20)
    dict(n_genomes=500, n_loci=30000, seed=7, spectrum="sfs", missing_rate=0.004, missing_af_rate=0.01),
    dict(n_genomes=500, n_loci=30000, seed=8, spectrum="sfs", unphased=True),
    dict(n_genomes=449, n_loci=12001, seed=9, spectrum="dense", unphased=True, grouped=False, missing_af_rate=0.03),
    dict(n_genomes=512, n_loci=25600, seed=10, spectrum="sfs", grouped=False),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"N{c['n_genomes']}xL{c['n_loci']}")
def test_all_estimators_match_oracle(gpu, case):
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(**case)
    if case["seed"] == 1:   # exercise q <= 0.01 rows and p <= 0.001 on a big case
        pop.af[:, ::97] = np.float32(0.996)
        pop.af[:, 5::89] = np.float32(0.0004)
    sel_kw = dict(spacing=20 if case["seed"] % 2 else 0, min_af=0.0, max_af=1.0)
    sel = O.select_all_pops(pop, **sel_kw)
    gpu.upload_population(pop)
    gpu.select_loci(**sel_kw)
    assert np.array_equal(gpu.get_locus_selection(), sel_bits(sel))

    lc, gc = gpu.allele_count()
    olc, ogc = O.allele_count(pop)
    assert np.array_equal(lc, olc) and np.array_equal(gc, ogc)

    lc2, res = gpu.count_and_inbreed()
    assert np.array_equal(lc2, olc)
    for algo, got in (("Simple", res), ("RitlandLocus", gpu.inbreed("RitlandLocus"))):
        want = O.inbreed(pop, sel, algo)
        c_got, f_got = results_matrix(got)
        c_want, f_want = results_matrix(want)
        assert np.array_equal(c_got, c_want), algo
        assert rel_err(f_got[:, :3], f_want[:, :3]) < TIGHT, algo
        ok = c_want[:, 4] > 0
        assert np.max(np.abs(got["inbred_allele_sum"][ok] - want["inbred_allele_sum"][ok])
                      / np.maximum(np.abs(want["inbred_allele_sum"][ok]), 1e-3)) < 1e-8, algo

    start = np.linspace(0.05, 0.5, pop.n_genomes)
    got = gpu.inbreed("HallME", hall_start=start, hall_sweeps=50)
    want = O.inbreed(pop, sel, "HallME", start=start, sweeps=50)
    ok = results_matrix(want)[0][:, 4] > 0
    assert rel_err(got["inbred_allele_sum"][ok], want["inbred_allele_sum"][ok]) < 1e-9

    grid = np.array([-0.4, -0.05, 0.0, 0.07, 0.3, 0.9])
    assert rel_err(gpu.loglik_grid(grid)[ok], O.loglik_grid(pop, sel, grid)[ok]) < 1e-12
    got = gpu.inbreed("Loglikelihood")
    want = O.inbreed(pop, sel, "Loglikelihood")
    assert np.max(np.abs(got["inbred_allele_sum"][ok] - want["inbred_allele_sum"][ok])) < 1e-9


@pytest.mark.parametrize("unphased,sel_kw", [(False, dict(spacing=0)), (False, dict(spacing=25, min_af=0.01, max_af=0.9)),
                                             (True, dict(spacing=15, lower=20_000, upper=150_000))],
                         ids=["phased", "phased-spaced", "unphased-window"])
def test_multi_allelic_loci_match_oracle(gpu, unphased, sel_kw):
    """Loci with two or three alternate alleles (kgl_b200_upload_multi_allelic): selection (they take part in the spaced accept
    chain), class counts incl. MINOR_HETEROZYGOUS bit-exact, the four expected sums incl. the sum of 2 p_i p_j, and all four
    estimators against the oracle, whose general forms are pinned bit for bit to the reference (golden multi_allelic*)."""
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    pop, _ = make_population(600, 20_000, seed=91, missing_rate=0.004, missing_af_rate=0.01, unphased=unphased, grouped=False)
    add_multi_allelic(pop, 700, seed=92)
    sel = O.select_all_pops(pop, **sel_kw)
    gpu.upload_population(pop)
    counts = gpu.select_loci(**sel_kw)
    assert np.array_equal(gpu.get_locus_selection(), sel_bits(sel))
    assert np.array_equal(counts[:6], sel.sum(axis=1).astype(np.uint64))
    assert sel[:, pop.multi_rows].sum() > 100                                   # multi-allelic loci are selected
    lc, res = gpu.count_and_inbreed()
    assert np.array_equal(lc, O.allele_count(pop)[0])
    start = np.linspace(0.05, 0.5, pop.n_genomes)
    for algo, kw, okw in (("Simple", None, {}), ("RitlandLocus", {}, {}), ("HallME", dict(hall_start=start, hall_sweeps=50), dict(start=start, sweeps=50)),
                          ("Loglikelihood", {}, {})):
        got = res if kw is None else gpu.inbreed(algo, **kw)
        want = O.inbreed(pop, sel, algo, **okw)
        c_got, f_got = results_matrix(got)
        c_want, f_want = results_matrix(want)
        assert np.array_equal(c_got, c_want), algo
        assert c_want[:, 3].sum() > 0
        assert rel_err(f_got, f_want) < TIGHT, algo
        assert np.max(np.abs(got["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-9, algo
    grid = np.array([-0.4, -0.05, 0.0, 0.07, 0.3, 0.9, -0.9, 0.5, 0.2])          # nine points: two launches of the grid kernel
    assert rel_err(gpu.loglik_grid(grid), O.loglik_grid(pop, sel, grid)) < 1e-12
    # without the side structures the same matrix is a population whose multi-allelic loci are absent: results must differ
    gpu.upload_multi_allelic(None, None, None)
    gpu.select_loci(**sel_kw)
    assert not np.array_equal(results_matrix(gpu.count_and_inbreed()[1])[0], results_matrix(O.inbreed(pop, sel, "Simple"))[0])


@pytest.mark.parametrize("kw", [
    dict(spacing=1),                                             # below the 10 bp locus spacing: every candidate is accepted
    dict(spacing=10), dict(spacing=11), dict(spacing=1000),
    dict(spacing=1000, lower=123_456, upper=2_000_000, min_af=0.02, max_af=0.4),
    dict(spacing=10**7),                                         # one accepted locus per population
    dict(spacing=250, lower=5_000_000, upper=6_000_000),         # empty window
], ids=lambda kw: "-".join(f"{k}{v}" for k, v in kw.items()))
def test_spaced_selection_on_the_device(gpu, kw):
    """getAllelesFromTo with SamplingDistance > 0 (kga_analysis_inbreed_locus.cpp:21-72): the accept chain is marked on the device
    by pointer doubling (locus_kernels.cuh); bit-exact against the oracle's sequential walk, per super-population, on a
    population large enough for many 256-locus blocks and missing frequencies; the first locus sits at offset 0."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(64, 300_000, seed=77, missing_af_rate=0.1)
    pop.offsets = (pop.offsets - pop.offsets[0]).astype(np.uint32)          # offsets 0, 10, 20, ...: the previous_offset == 0 rule
    gpu.upload_population(pop)
    counts = gpu.select_loci(**kw)
    want = O.select_all_pops(pop, **kw)
    assert np.array_equal(gpu.get_locus_selection(), sel_bits(want))
    assert np.array_equal(counts[: want.shape[0]], want.sum(axis=1).astype(np.uint64))


@pytest.mark.parametrize("unphased", [False, True], ids=["phased", "unphased"])
def test_loglikelihood_clamped_terms(gpu, unphased):
    """The likelihood's clamps (calc.cpp:108-124). Heterozygous cells at loci with 2 p q < 1e-10 are clamped at every f: the
    table-driven Newton sweep hands such genomes to the cell-by-cell kernel (terms_fast.cuh, state 2). In an unphased
    population a hom-alt pair is the heterozygous term 2 (1-f) p p, clamped from above where it exceeds 1: the sweep counts
    those cells per genome and f. Both must land on the oracle's optimum."""
    from kgl_gene_b200.flatfile import pack_codes, unpack_codes
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(96, 5000, seed=31, unphased=unphased)
    pop.af[:, ::50] = np.float32(1e-11)
    pop.af[:, 3::40] = np.float32(0.95)
    codes = unpack_codes(pop.packed, pop.n_genomes)
    codes[::50, ::3] = 1                      # every third genome is heterozygous at the 1e-11 loci
    pop.packed = pack_codes(codes)
    sel = O.select_all_pops(pop)
    gpu.upload_population(pop)
    gpu.select_loci()
    got = gpu.inbreed("Loglikelihood")
    want = O.inbreed(pop, sel, "Loglikelihood")
    c_got, _ = results_matrix(got)
    c_want, _ = results_matrix(want)
    assert np.array_equal(c_got, c_want)
    assert np.max(np.abs(got["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-9
    grid = np.array([-0.2, 0.0, 0.1, 0.6])
    assert rel_err(gpu.loglik_grid(grid), O.loglik_grid(pop, sel, grid)) < 1e-12


def test_hallme_fixed_point(gpu):
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(96, 6000, seed=11)
    sel = O.select_all_pops(pop)
    gpu.upload_population(pop)
    gpu.select_loci()
    got = gpu.inbreed("HallME", hall_sweeps=-1)
    want = O.inbreed(pop, sel, "HallME", sweeps=-1)
    assert np.max(np.abs(got["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-9


@pytest.mark.parametrize("case", [
    dict(n_genomes=300, n_loci=20000, seed=41, spectrum="sfs", grouped=True),
    dict(n_genomes=257, n_loci=9000, seed=42, spectrum="dense", grouped=False),                 # every tile holds every population
    dict(n_genomes=500, n_loci=30000, seed=43, spectrum="sfs", missing_rate=0.01, missing_af_rate=0.01),
    dict(n_genomes=96, n_loci=12000, seed=44, spectrum="sfs", unphased=True),
], ids=lambda c: f"N{c['n_genomes']}xL{c['n_loci']}")
def test_moment_tables_agree_with_exact_sweeps(gpu, case):
    """HallME and the likelihood root search from the per-genome moment tables (terms_moments.cuh) against the kernels that
    evaluate every cell in every sweep (terms_fast.cuh) and against the oracle -- with the frequencies that bend the tables:
    a == 1 in one population (t = 0 cells), exactly 1/2, the ends of the bin range, rare homozygous cells far left."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(**case)
    pop.af[1, ::61] = np.float32(1.0)
    pop.af[:, 7::53] = np.float32(0.5)
    pop.af[:, 11::211] = np.float32(1e-11)
    pop.af[:, 13::199] = np.float32(0.9999)
    pop.af[2, 17::97] = np.float32(0.75)
    unphased = bool(case.get("unphased"))
    for sel_kw in (dict(spacing=0), dict(spacing=15, lower=int(pop.offsets[pop.n_loci // 5]), upper=int(pop.offsets[pop.n_loci // 2]))):
        sel = O.select_all_pops(pop, **sel_kw)
        gpu.upload_population(pop)
        gpu.select_loci(**sel_kw)
        start = np.linspace(0.0, 1.0, pop.n_genomes)
        want = O.inbreed(pop, sel, "HallME", start=start, sweeps=50)
        ok = results_matrix(want)[0][:, 4] > 0
        fast = gpu.inbreed("HallME", hall_start=start, hall_sweeps=50)
        assert gpu.used_moment_tables() == 2                      # tables built on the tensor cores (k_mom_mma)
        gpu.select_loci(**sel_kw)                                 # a new selection: the tables are rebuilt, now on the CUDA cores
        cores = gpu.inbreed("HallME", hall_start=start, hall_sweeps=50, moments_on_cuda_cores=True)
        assert gpu.used_moment_tables() == 1
        assert np.array_equal(fast["inbred_allele_sum"], cores["inbred_allele_sum"], equal_nan=True)     # the same integers
        steps = gpu.inbreed("HallME", hall_start=start, hall_sweeps=50, sweep_by_sweep=True)     # the protocol of a locus-sharded caller
        assert gpu.used_moment_tables() and np.max(np.abs(fast["inbred_allele_sum"][ok] - steps["inbred_allele_sum"][ok])) < 1e-13
        exact = gpu.inbreed("HallME", hall_start=start, hall_sweeps=50, exact_sweeps=True)
        assert not gpu.used_moment_tables()
        assert np.max(np.abs(fast["inbred_allele_sum"][ok] - exact["inbred_allele_sum"][ok])) < 1e-10
        assert rel_err(fast["inbred_allele_sum"][ok], want["inbred_allele_sum"][ok]) < 1e-9
        fast = gpu.inbreed("Loglikelihood")
        if not unphased:
            gpu.select_loci(**sel_kw)
            cores = gpu.inbreed("Loglikelihood", moments_on_cuda_cores=True)
            assert gpu.used_moment_tables() == 1
            assert np.max(np.abs(fast["inbred_allele_sum"][ok] - cores["inbred_allele_sum"][ok])) < 1e-12
            gpu.select_loci(**sel_kw)
            fast = gpu.inbreed("Loglikelihood")
        assert bool(gpu.used_moment_tables()) == (not unphased)       # Q6: the upper clamp of 2 (1-f) p p needs the cells
        steps = gpu.inbreed("Loglikelihood", sweep_by_sweep=True)
        assert np.max(np.abs(fast["inbred_allele_sum"][ok] - steps["inbred_allele_sum"][ok])) < 1e-12
        exact = gpu.inbreed("Loglikelihood", exact_sweeps=True)
        assert not gpu.used_moment_tables()
        want = O.inbreed(pop, sel, "Loglikelihood")
        assert np.max(np.abs(fast["inbred_allele_sum"][ok] - exact["inbred_allele_sum"][ok])) < 1e-10
        assert np.max(np.abs(fast["inbred_allele_sum"][ok] - want["inbred_allele_sum"][ok])) < 1e-9
        assert np.array_equal(results_matrix(fast)[0], results_matrix(want)[0])
    # a HallME start outside [0,1], and a frequency below the bins (1e-13): the exact kernels take over, same results
    start = np.linspace(-0.3, 1.2, pop.n_genomes)
    got = gpu.inbreed("HallME", hall_start=start, hall_sweeps=10)
    assert not gpu.used_moment_tables()
    pop.af[0, 19::301] = np.float32(1e-13)
    gpu.upload_population(pop)
    gpu.select_loci()
    sel = O.select_all_pops(pop)
    got = gpu.inbreed("HallME", hall_sweeps=50)
    assert not gpu.used_moment_tables()
    want = O.inbreed(pop, sel, "HallME", sweeps=50)
    ok = results_matrix(want)[0][:, 4] > 0
    assert rel_err(got["inbred_allele_sum"][ok], want["inbred_allele_sum"][ok]) < 1e-9


def test_moment_tables_left_of_zero(gpu):
    """Outbred and negatively inbred genomes: the root search runs at f < 0, where the bins of the octaves below 4|f| give way
    to the list of the genome's rare homozygous cells; genomes left of the tables' domain (f < -0.2) take the exact kernel."""
    from kgl_gene_b200.flatfile import pack_codes
    from kgl_gene_b200.synth import make_loci, make_genomes, synth_codes
    from kgl_gene_b200.flatfile import FlatPopulation, row_bytes_for
    n, l = 200, 16000
    offsets, af = make_loci(l, 51, spectrum="dense")
    superpop, _ = make_genomes(n, 51)
    inbreeding = np.linspace(-0.45, 0.05, n)                # excess heterozygosity
    codes = synth_codes(51, af, superpop, inbreeding, missing_rate=0.002)
    pop = FlatPopulation(offsets, af, superpop, pack_codes(codes), n, False)
    sel = O.select_all_pops(pop)
    gpu.upload_population(pop)
    gpu.select_loci()
    want = O.inbreed(pop, sel, "Loglikelihood")
    fast = gpu.inbreed("Loglikelihood")
    assert gpu.used_moment_tables()
    assert want["inbred_allele_sum"].min() < -0.25 and (want["inbred_allele_sum"] > -0.15).sum() > 20
    assert np.max(np.abs(fast["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-9


@pytest.mark.parametrize("n,l,miss", [(130, 40_000, 0.012), (70, 2_400_000, 0.014)], ids=["segments", "counter-flush"])
def test_ibs_sparse_repair_at_scale(gpu, n, l, miss):
    """The sparse repair of code-3 cells (k_ibs_missing_fix) where it splits a genome's dropped rows into segments (few tiles,
    many rows) and where one thread's rows exceed a counter flush (> 32,760 dropped rows per genome), against the naive
    O(N^2 L) oracle loop."""
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    offsets, af = make_loci(l, 91)
    superpop, f = make_genomes(n, 91)
    packed = O.synth_genotypes(91, n, l, af, superpop, f, missing_rate=miss)
    pop = FlatPopulation(offsets, af, superpop, packed, n, False)
    gpu.upload_population(pop)
    assert np.array_equal(gpu.ibs(), O.ibs(pop))


def test_ibs_matches_oracle(gpu):
    """Indexed code-3 cells: two-plane kernel on pre-masked planes + sparse repair (ibs_tile.cuh)."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(150, 3001, seed=21, missing_rate=0.03)
    gpu.upload_population(pop)
    want = O.ibs(pop)
    for tensor in (True, False):                       # dense part on the tensor cores (ibs_gram.cuh) and on the popcount kernel
        gpu.set_ibs_tensor_cores(tensor)
        assert np.array_equal(gpu.ibs(), want)
        assert gpu.ibs_used_tensor_cores() == tensor
        assert np.array_equal(gpu.ibs(64, 130), want[64:130])
        assert np.array_equal(gpu.ibs(149, 150), want[149:150])
    gpu.set_ibs_tensor_cores(True)


@pytest.mark.parametrize("n,l,miss", [(70, 999, 0.0),        # no code-3 cell: the sample-major planes as they are
                                      (300, 20000, 0.03),    # too many code-3 cells to index: in-kernel validity plane
                                      (64, 64, 0.5),         # exactly one tile, two words, half the cells dropped
                                      (1, 40, 0.1),          # a single genome
                                      (129, 33000, 0.002)])  # several word chunks per tile
def test_ibs_modes_and_edges(gpu, n, l, miss):
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(n, l, seed=3 + n, missing_rate=miss)
    gpu.upload_population(pop)
    want = O.ibs(pop)
    for tensor in (True, False):
        gpu.set_ibs_tensor_cores(tensor)
        got = gpu.ibs()
        assert gpu.ibs_used_tensor_cores() == (tensor and n != 300)       # 300 x 20000 at 3 %: too many code-3 cells to index -> popcount kernel with a validity plane
        assert np.array_equal(got, want)
        assert np.array_equal(got, got.transpose(1, 0, 2))
        assert np.array_equal(got[..., :3].sum(-1), got[..., 3])
    gpu.set_ibs_tensor_cores(True)


def test_ibs_tiles_dealt_to_ranks(gpu):
    """The multi-GPU decomposition on one device: every 'rank' computes tiles rank, rank + world, ...; assembled = oracle."""
    from kgl_gene_b200 import shards
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(200, 2500, seed=8, missing_rate=0.01)
    gpu.upload_population(pop)
    side, n_up = gpu.ibs_tile_grid()
    assert side == 4 and n_up == 10
    want = O.ibs(pop)
    for world in (1, 3):
        blocks = [gpu.ibs_tiles(first=r, stride=world) for r in range(world)]
        assert np.array_equal(shards.assemble_ibs(pop.n_genomes, blocks), want)
    # cells of padding genomes (200..255) read zero
    last = gpu.ibs_tiles(first=n_up - 1, stride=1, count=1)[0]
    assert np.all(last[200 - 192:, :, :] == 0) and np.all(last[:, 200 - 192:, :] == 0)


def test_ibs_blocks_dealt_to_ranks(gpu):
    """Whole 256 x 256 blocks of tiles per 'rank' (shards.block_tile_coords -> kgl_b200_run_ibs_tile_list): the unit of the
    tensor-core form; three ranks' tiles assemble into the oracle's matrix."""
    from kgl_gene_b200.shards import assemble_ibs_coords, block_tile_coords, n_upper_tiles
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(700, 2500, seed=23, missing_rate=0.01)
    gpu.upload_population(pop)
    want = O.ibs(pop)
    coords = [block_tile_coords(pop.n_genomes, r, 3) for r in range(3)]
    assert sum(c.shape[0] for c in coords) == n_upper_tiles(pop.n_genomes)
    tiles = [gpu.ibs_tile_list(c) for c in coords]
    assert gpu.ibs_used_tensor_cores()
    assert np.array_equal(assemble_ibs_coords(pop.n_genomes, coords, tiles), want)


def test_ibs_wide_population_on_tensor_cores(gpu):
    """More genomes than one launch's tile list (3,000 -> 1,128 tiles of 141 blocks): the Gram blocks are stored block by block, no
    N x N matrix; rows of a band use mirrored blocks below the diagonal."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(3000, 400, seed=29, missing_rate=0.004)
    gpu.upload_population(pop)
    want = O.ibs(pop)
    got = gpu.ibs()
    assert gpu.ibs_used_tensor_cores()
    assert np.array_equal(got, want)
    assert np.array_equal(gpu.ibs(2100, 2400), want[2100:2400])


def test_ibs_full_width_properties(gpu):
    """chr22-shaped width on device-generated data: symmetry through independent tiles, diagonal, row sums vs allele counts."""
    from kgl_gene_b200.synth import make_genomes, make_loci
    n, l = 2504, 40_000
    offsets, af = make_loci(l, 78)
    superpop, f = make_genomes(n, 78)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.synth_genotypes(78, n, l, f, missing_rate=0.001)
    _, gc = gpu.allele_count()
    band = gpu.ibs(1000, 1100)                       # band path: every tile of two tile rows, no mirroring
    full = gpu.ibs()                                 # upper triangle + mirrored
    assert np.array_equal(full[1000:1100], band)
    assert np.array_equal(full, full.transpose(1, 0, 2))
    d = np.arange(n)
    valid = (gc[:, 0] + gc[:, 1] + gc[:, 2]).astype(np.uint32)
    assert np.array_equal(full[d, d, 3], valid) and np.array_equal(full[d, d, 2], valid)
    assert np.all(full[d, d, 0] == 0) and np.all(full[d, d, 1] == 0)
    assert np.array_equal(full[..., :3].sum(-1), full[..., 3])


@pytest.mark.parametrize("n,l,miss", [(150, 3001, 0.03), (1, 77, 0.0), (257, 130, 0.0), (300, 20000, 0.03), (64, 33000, 0.001)])
def test_gram_tensor_core_matches_oracle(gpu, n, l, miss):
    """K5: int8 x int8 -> int32 on tcgen05; bit-exact, and tied to the popcount path when nothing is coded 3."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(n, l, seed=100 + n, missing_rate=miss)
    gpu.upload_population(pop)
    want, want_c = O.gram(pop, pop.af[5])
    got = gpu.gram()
    assert np.array_equal(got, want)
    got_c = gpu.grm(5)
    assert np.allclose(got_c, want_c, rtol=1e-9, atol=1e-7)
    if miss == 0.0:
        ibs = gpu.ibs().astype(np.int64)
        d = np.diag(got).astype(np.int64)
        assert np.array_equal(d[:, None] + d[None, :] - 2 * got.astype(np.int64), ibs[..., 1] + 4 * ibs[..., 0])


def test_gram_tiles_dealt_to_ranks(gpu):
    """The multi-GPU decomposition on one device: the tile subsets of three 'ranks' add up to the whole matrix."""
    import ctypes as C
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(600, 4000, seed=12, missing_rate=0.01)
    gpu.upload_population(pop)
    want, _ = O.gram(pop)
    total = np.zeros_like(want, dtype=np.int64)
    for r in range(3):
        gpu.enqueue_gram_tiles(r, 3)
        total += gpu.fetch_gram()          # symmetric read-out of a partial matrix: off-diagonal cells of missing tiles are 0
    assert np.array_equal(total, want.astype(np.int64))


def test_gram_full_width_identity(gpu):
    """chr22-shaped width on device-generated data without code-3 cells: the tensor-core and popcount paths must agree."""
    from kgl_gene_b200.synth import make_genomes, make_loci
    n, l = 2504, 50_000
    offsets, af = make_loci(l, 79)
    superpop, f = make_genomes(n, 79)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.synth_genotypes(79, n, l, f, missing_rate=0.0)
    g = gpu.gram().astype(np.int64)
    assert np.array_equal(g, g.T)
    _, gc = gpu.allele_count()
    assert np.array_equal(np.diag(g), (gc[:, 1] + 4 * gc[:, 2]).astype(np.int64))
    ibs = gpu.ibs().astype(np.int64)
    d = np.diag(g)
    assert np.array_equal(d[:, None] + d[None, :] - 2 * g, ibs[..., 1] + 4 * ibs[..., 0])


def test_golden_calc_fws(gpu, golden):
    """CalcFWS against the reference's own kga_analysis_PfEMP_FWS.cpp (compiled into oracle/_ref, golden ref_fws_*): per-genome
    AlleleSummmary in the eleven AF bins and the per-variant summaries, bit-exact; the alleles of multi-allelic loci are variants
    with their own AF (k_multi_bin_counts). Side cells with more than two variants (0xFF) do not say which alleles the genome
    carries: those genomes are compared with the oracle instead, those loci left out of the per-variant comparison."""
    from kgl_gene_b200 import fws
    name, pop, ref, _ = golden
    gpu.upload_population(pop)
    got = fws.calc_fws(gpu, pop=5, n_multi=pop.n_multi)
    known = np.ones(pop.n_genomes, dtype=bool)
    ordinary = np.ones(pop.n_loci, dtype=bool)
    if pop.n_multi:
        known = ~(pop.multi_cells == 0xFF).any(axis=0)
        ordinary[pop.multi_rows] = False
    bins = np.transpose(got["genome_bins"], (1, 0, 2))
    assert np.array_equal(bins[known], ref["fws_genome"][known])
    assert np.array_equal(got["bin_variants"], ref["fws_genome"].sum(axis=2)[0])
    want, want_rows = O.fws_bins(pop, 5, fws.FWS_BINS)
    assert np.array_equal(got["bin_variants"], want_rows)
    assert np.array_equal(got["genome_bins"][:, :, 1:], want[:, :, 1:3])
    assert np.array_equal(got["genome_bins"][:, :, 0], want[:, :, 0] + want[:, :, 3])
    m = (ref["fws_variant_present"] == 1) & ordinary
    assert np.array_equal(got["present"][ordinary], (ref["fws_variant_present"] == 1)[ordinary])
    assert np.array_equal(got["variant_summary"][m].astype(np.uint64), ref["fws_variant"][m])
    if pop.n_multi:
        has = ~np.isnan(pop.multi_af).all(axis=0)
        n_slots = np.where(has.any(axis=1), 3 - np.argmax(has[:, ::-1], axis=1), 0)
        sel = (np.arange(3)[None, :] < n_slots[:, None]) & ~(pop.multi_cells == 0xFF).any(axis=1)[:, None]
        present = ref["fws_multi_variant_present"] == 1
        assert np.array_equal(got["multi_present"][sel], present[sel])
        sel &= present
        assert np.array_equal(got["multi_variant_summary"][sel].astype(np.uint64), ref["fws_multi_variant"][sel])
        # all alleles, no presence filter: one bin over everything = every ordinary row and every listed allele that has an AF
        allc, rows = gpu.binned_genome_counts([0.0], [2.0], pop=5, present_only=False)
        assert int(rows[0]) == int((~np.isnan(pop.af[5][ordinary])).sum()) + int((~np.isnan(pop.multi_af[5])).sum())
        w2, _ = O.fws_bins(pop, 5, [(0.0, 2.0)], present_only=False)
        assert np.array_equal(allc, w2)
    # HeteroHomoZygous::updateVariantAnalysisType run by the harness over every offset of every genome
    want_hh = ref["hetero_homo"]       # total, snp, indel, homMinor, hetMinor, hetRefMinor, homRef
    assert np.array_equal(gpu.hetero_homo(), want_hh)
    if not pop.n_multi:
        _, gc = gpu.allele_count()
        hh = fws.hetero_homo_summary(gc)
        for j, key in enumerate(["total_variants", "snp_count", "indel_count", "homozygous_minor_alleles", "heterozygous_minor_alleles",
                                 "heterozygous_reference_minor_alleles", "homozygous_reference_alleles"]):
            assert np.array_equal(hh[key], want_hh[:, j]), key


@pytest.mark.parametrize("n,l,miss,spectrum", [(131, 5000, 0.01, "sfs"), (500, 3000, 0.0, "dense"), (2504, 20000, 0.001, "sfs")])
def test_fws_bins_match_oracle(gpu, n, l, miss, spectrum):
    """N1: CalcFWS per-genome AlleleSummmary in the eleven AF bins + per-variant summaries + HeteroHomoZygous / F_IS."""
    from kgl_gene_b200 import fws
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(n, l, seed=40 + n, missing_rate=miss, spectrum=spectrum, missing_af_rate=0.02)
    gpu.upload_population(pop)
    got = fws.calc_fws(gpu, pop=5)
    want, want_rows = O.fws_bins(pop, 5, fws.FWS_BINS)
    assert np.array_equal(got["bin_variants"], want_rows)
    assert np.array_equal(got["genome_bins"][:, :, 1:], want[:, :, 1:3])
    assert np.array_equal(got["genome_bins"][:, :, 0], want[:, :, 0] + want[:, :, 3])      # other-allele cells count as refHom
    olc, ogc = O.allele_count(pop)
    assert np.array_equal(got["variant_summary"][:, 1:], olc[:, 1:3])
    assert np.array_equal(got["variant_summary"][:, 0], olc[:, 0] + olc[:, 3])
    # all loci, no presence filter: the bins partition the loci that have an AF value
    allc, rows = gpu.binned_genome_counts([0.0], [2.0], pop=5, present_only=False)
    assert int(rows[0]) == int((~np.isnan(pop.af[5])).sum())
    w2, _ = O.fws_bins(pop, 5, [(0.0, 2.0)], present_only=False)
    assert np.array_equal(allc, w2)
    # HeteroHomoZygous bookkeeping on the raw per-genome counts
    _, gc = gpu.allele_count()
    hh = fws.hetero_homo_summary(gc)
    codes = pop.codes()
    assert np.array_equal(hh["total_variants"], ((codes == 1).sum(0) + 2 * (codes == 2).sum(0) + (codes == 3).sum(0)).astype(np.uint64))
    fis = fws.wrights_fis(hh, pop.superpop)
    for k in np.unique(pop.superpop):
        m = pop.superpop == k
        h_exp = hh["heterozygous_reference_minor_alleles"][m].sum() / hh["total_variants"][m].sum()
        h_obs = hh["heterozygous_reference_minor_alleles"][m] / hh["total_variants"][m]
        assert np.allclose(fis[m], (h_exp - h_obs) / h_exp, rtol=1e-12)


def test_vcf_ingest_to_device(gpu, tmp_path):
    """N2 end to end: VCF text -> packed matrix (host ingest, no PopulationDB) -> device pass, against the oracle on the source."""
    from kgl_gene_b200.synth import make_population
    from kgl_gene_b200.vcf import ingest_vcf, write_vcf
    pop, _ = make_population(200, 3000, seed=52, missing_rate=0.0)
    path = str(tmp_path / "chr.vcf.gz")
    write_vcf(pop, path)
    got, names, _, st = ingest_vcf(path, superpop=pop.superpop)
    assert st["kept"] == 3000 and len(names) == 200
    gpu.upload_population(got)
    gpu.select_loci()
    lc, res = gpu.count_and_inbreed()
    sel = O.select_all_pops(pop)
    want = O.inbreed(pop, sel, "Simple")
    assert np.array_equal(lc, O.allele_count(pop)[0])
    assert np.array_equal(results_matrix(res)[0], results_matrix(want)[0])
    assert rel_err(res["inbred_allele_sum"], want["inbred_allele_sum"]) < 1e-9


@pytest.mark.parametrize("algo,tol", [("Simple", 0.02), ("RitlandLocus", 0.03), ("HallME", 0.03), ("Loglikelihood", 0.02)])
def test_synthetic_self_check(gpu, tmp_path, algo, tol):
    """N4: the reference's Synthetic mode (101 genomes, planted F = -0.5 .. 0.5): every estimator recovers the planted
    coefficient (HallME estimates max(F, 0): an EM over a mixture weight)."""
    from kgl_gene_b200 import synthetic
    from kgl_gene_b200.synth import make_loci
    offsets, af = make_loci(60_000, 17, spectrum="dense")
    ids, syn, calc = synthetic.synthetic_self_check(gpu, af, offsets, algorithm=algo, seed=5)
    assert len(ids) == 101 and syn[0] == -0.5 and abs(syn[-1] - 0.5) < 1e-12
    # For F < 0 the class law leaves the simplex at small p (p^2 + F p q < 0 below p = -F q): the draw is clipped there, in the
    # reference's generator as well, so the planted value is only recovered approximately on the negative side.
    pos = syn >= 0.0 if algo != "HallME" else syn > 0.05
    assert np.max(np.abs(calc[pos] - syn[pos])) < tol, np.max(np.abs(calc[pos] - syn[pos]))
    if algo != "HallME":
        neg = syn < -0.02
        assert np.all(calc[neg] < 0.0) and np.all(calc[neg] >= syn[neg] - 0.03)       # clipped towards zero, never beyond the plant
        assert np.corrcoef(calc, syn)[0, 1] > 0.99
    synthetic.write_synthetic_csv(str(tmp_path / "syn.csv"), ids, syn, calc)
    assert open(tmp_path / "syn.csv").readline().strip() == "Sample,SynInbreed,CalcInbreed"


def test_device_generator_matches_numpy(gpu):
    from kgl_gene_b200.synth import make_genomes, make_loci, synth_codes
    from kgl_gene_b200.flatfile import pack_codes
    offsets, af = make_loci(700, 9)
    superpop, f = make_genomes(333, 9)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.synth_genotypes(1234, 333, 700, f, missing_rate=0.01, locus_base=5)
    assert np.array_equal(gpu.download_genotypes(), pack_codes(synth_codes(1234, af, superpop, f, 0.01, locus_base=5)))


def test_wide_population_multi_slice(gpu):
    """More than 16384 genomes: a locus row spans several CTA slices (global-atomic locus counts)."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(16384 + 777, 160, seed=31)
    sel = O.select_all_pops(pop)
    gpu.upload_population(pop)
    gpu.select_loci()
    lc, res = gpu.count_and_inbreed()
    olc, _ = O.allele_count(pop)
    assert np.array_equal(lc, olc)
    want = O.inbreed(pop, sel, "Simple")
    assert np.array_equal(results_matrix(res)[0], results_matrix(want)[0])


def test_full_width_properties_on_device_generated_population(gpu):
    """chr22-shaped width (2,504 genomes), generated on the device: size-independent invariants."""
    from kgl_gene_b200.synth import make_genomes, make_loci
    n, l = 2504, 200_000
    offsets, af = make_loci(l, 77)
    superpop, f = make_genomes(n, 77)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.synth_genotypes(77, n, l, f)
    gpu.select_loci()
    lc, gc = gpu.allele_count()
    assert np.all(lc.sum(axis=1) == n) and np.all(gc.sum(axis=1) == l)
    assert np.array_equal(lc.sum(axis=0).astype(np.uint64), gc.sum(axis=0))               # checksum of checksums
    lc2, res = gpu.count_and_inbreed()
    assert np.array_equal(lc, lc2)
    counts, freqs = results_matrix(res)
    # every locus is selected for every population here, so classified + dropped = all loci
    assert np.all(counts[:, 4] <= l) and np.all(counts[:, 1] == gc[:, 1]) and np.all(counts[:, 2] == gc[:, 2])
    assert np.allclose(freqs.sum(axis=1), counts[:, 4], rtol=1e-12)                       # Q8: class frequencies sum to n
    assert np.corrcoef(res["inbred_allele_sum"], f)[0, 1] > 0.99                          # recovers the planted F


@pytest.mark.parametrize("algo", ["Simple", "RitlandLocus", "HallME", "Loglikelihood"])
def test_locus_sharded_estimators_two_contexts(algo):
    """The split estimator protocol of the C ABI (inbreed_begin / accumulate / partials_buffer / update / fetch) with two locus
    shards: two contexts on one GPU play two ranks, their partial-sum buffers are summed on the device between accumulate and
    update exactly as the all-reduce does. The result must equal the unsharded run (and the oracle): covers the per-shard
    heterozygous counts, the per-shard feasibility limits and the list of unfinished genomes of the likelihood search."""
    import torch
    from kgl_gene_b200.capi import KglB200
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.shards import _RawCudaArray
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(200, 9000, seed=61, missing_rate=0.004)
    cut = 5000 - 32 * 3 + 7                                            # not a multiple of anything
    shards = [FlatPopulation(pop.offsets[a:b], np.ascontiguousarray(pop.af[:, a:b]), pop.superpop, np.ascontiguousarray(pop.packed[a:b]),
                             pop.n_genomes, pop.unphased) for a, b in ((0, cut), (cut, pop.n_loci))]
    dev = torch.device("cuda", 0)
    ctxs = [KglB200(0) for _ in shards]
    try:
        for c, sh in zip(ctxs, shards):
            c.upload_population(sh)
            c.select_loci()
        opts = dict(hall_start=np.linspace(0.05, 0.5, pop.n_genomes), hall_sweeps=50) if algo == "HallME" else {}
        for c in ctxs:
            c.inbreed_begin(algo, **opts)
        finished, passes = False, 0
        while not finished:
            for c in ctxs:
                c.inbreed_accumulate()
                c.synchronize()
            bufs = []
            for c in ctxs:
                ptr, cnt = c.inbreed_partials_buffer()
                bufs.append(torch.as_tensor(_RawCudaArray(ptr, cnt, "<f8"), device=dev))
            total = bufs[0] + bufs[1]
            for b in bufs:
                b.copy_(total)
            torch.cuda.synchronize()
            fin = [c.inbreed_update() for c in ctxs]
            assert fin[0] == fin[1]
            finished = fin[0]
            passes += 1
            assert passes < 400
        got = [c.inbreed_fetch() for c in ctxs]
    finally:
        for c in ctxs:
            c.close()
    sel = O.select_all_pops(pop)
    kw = dict(start=opts["hall_start"], sweeps=50) if algo == "HallME" else {}
    want = O.inbreed(pop, sel, algo, **kw)
    c_want, f_want = results_matrix(want)
    for g in got:
        c_got, f_got = results_matrix(g)
        assert np.array_equal(c_got, c_want)
        assert rel_err(f_got[:, :3], f_want[:, :3]) < TIGHT
        assert np.max(np.abs(g["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-9
    assert np.array_equal(got[0]["inbred_allele_sum"], got[1]["inbred_allele_sum"])      # both "ranks" hold the same bits


def test_peer_exchange_two_gpus():
    """Locus-sharded step with the exchange over NVLink peer memory (kgl_b200_enqueue_count_and_inbreed_peer): two ranks through
    bench.py, which asserts the fused exchange against the NCCL all-reduce path before timing. Needs two GPUs."""
    import json
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29531", os.path.join(root, "bench.py"), "--gpus", "2", "--steps", "3", "--warmup", "3", "--loci", "200000",
           "--no-kinship", "--no-estimators", "--no-e2e", "--no-cpu-baseline"]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert proc.returncode == 0, proc.stderr[-2000:]
    line = json.loads(proc.stdout.strip().splitlines()[-1])
    assert line["n_gpus"] == 2 and line["value"] > 0
    if line["config"]["exchange"] != "peer":
        pytest.skip("CUDA IPC peer mapping unavailable on this box: " + line["config"]["exchange"])


def test_bench_dump_outputs_two_gpus(tmp_path):
    """bench.py --dump-outputs with two locus-sharded ranks: rank 0's per-locus counts and the exchanged per-genome Simple results
    of the last timed step, against the oracle on rank 0's shard and on both shards together. Needs two GPUs."""
    import json
    import subprocess
    import sys
    import torch
    from bench import SEED
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n, l = 300, 50_000
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(root, "bench.py"), "--gpus", "2", "--steps", "3", "--warmup", "1",
           "--genomes", str(n), "--loci", str(l), "--no-kinship", "--no-estimators", "--no-e2e", "--no-cpu-baseline",
           "--dump-outputs", str(tmp_path)]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert proc.returncode == 0, proc.stderr[-2000:]
    assert json.loads(proc.stdout.strip().splitlines()[-1])["n_gpus"] == 2
    superpop, inbreeding = make_genomes(n, SEED)
    shards = []
    for rank in range(2):           # bench.py's shard of each rank
        offsets, af = make_loci(l, SEED + 1000 * rank)
        shards.append((offsets, af, O.synth_genotypes(SEED, n, l, af, superpop, inbreeding, locus_base=rank * l)))
    rank0 = FlatPopulation(shards[0][0], shards[0][1], superpop, shards[0][2], n, False)
    assert np.array_equal(np.load(tmp_path / "locus_counts.npy"), O.allele_count(rank0)[0])
    offsets = np.concatenate([shards[0][0], shards[1][0] + shards[0][0][-1] + 10])       # the two shards as one locus table
    both = FlatPopulation(offsets, np.concatenate([shards[0][1], shards[1][1]], axis=1), superpop,
                          np.concatenate([shards[0][2], shards[1][2]]), n, False)
    want = O.inbreed(both, O.select_all_pops(both), "Simple")
    for f in want.dtype.names:
        got = np.load(tmp_path / f"genome_{f}.npy")
        if f.endswith("_count"):
            assert np.array_equal(got, want[f]), f
        else:
            assert np.max(np.abs(got - want[f]) / np.maximum(np.abs(want[f]), 1e-3)) < 1e-6, f


@pytest.mark.parametrize("multi", [False, True], ids=["biallelic", "multi-allelic"])
def test_count_limited_selection_and_locus_filter(gpu, multi):
    """N3: RetrieveLociiVector::getLociiCount on the device (kgl_b200_count_loci: how the window loop of populationInbreeding finds
    a window's upper bound, kga_analysis_inbreed_diploid.cpp:48-51) against the oracle's count-mode walk, and the per-locus
    verdict of the variant-level filters (kgl_b200_set_locus_filter) against the oracle on the filtered locus table."""
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    pop, _ = make_population(96, 120_000, seed=55, missing_af_rate=0.05)
    if multi:
        add_multi_allelic(pop, 3000, seed=56)
    gpu.upload_population(pop)
    for k, kw in ((5, dict(lower=0, spacing=0, count=1000)), (5, dict(lower=400_000, spacing=1000, count=1000)),
                  (0, dict(lower=123_457, spacing=37, count=5000, min_af=0.01, max_af=0.6)), (2, dict(lower=900_000, spacing=500, count=10_000)),
                  (5, dict(lower=1_300_000, spacing=0, count=100)), (3, dict(lower=0, spacing=10**7, count=50))):
        want = O.select_all_pops(pop, mode=1, **kw)[k]
        offs = pop.offsets[want == 1]
        n, last = gpu.count_loci(pop=k, **kw)
        assert n == len(offs), (k, kw)
        if n:
            assert last == int(offs[-1]), (k, kw)
    # locus filter: a filtered locus is no candidate -- the spaced chain runs over the loci that are left
    rng = np.random.default_rng(5)
    keep = (rng.random(pop.n_loci) < 0.8).astype(np.uint8)
    gpu.set_locus_filter(keep)
    gpu.select_loci(spacing=40)
    from kgl_gene_b200.flatfile import FlatPopulation
    filtered = FlatPopulation(pop.offsets, pop.af.copy(), pop.superpop, pop.packed, pop.n_genomes, pop.unphased)
    filtered.af[:, keep == 0] = np.nan                   # the oracle's view of a filtered locus: no frequency, no candidate
    if multi:
        filtered.multi_rows, filtered.multi_cells = pop.multi_rows, pop.multi_cells
        filtered.multi_af = pop.multi_af.copy()
        filtered.multi_af[:, keep[pop.multi_rows] == 0, :] = np.nan
    want = O.select_all_pops(filtered, spacing=40)
    assert np.array_equal(gpu.get_locus_selection(), sel_bits(want))
    res = gpu.inbreed("Simple")
    assert np.array_equal(results_matrix(res)[0], results_matrix(O.inbreed(filtered, want, "Simple"))[0])
    gpu.set_locus_filter(None)
    gpu.select_loci(spacing=40)
    assert np.array_equal(gpu.get_locus_selection(), sel_bits(O.select_all_pops(pop, spacing=40)))


def test_hetero_homo_records_and_location_fis(gpu):
    """kgl_b200_run_hetero_homo against the per-offset rule of HeteroHomoZygous::updateVariantAnalysisType restated on the codes and
    side cells (pinned to the reference's translation unit by tests/test_plugin_dropin.py::test_pfemp_hetero_homo_csv_equals_reference_writer
    and the golden hetero_homo arrays), and kgl_b200_location_fis against the formula of UpdateSampleLocation."""
    from kgl_gene_b200.capi import location_fis
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    pop, _ = make_population(333, 6000, seed=44, missing_rate=0.01)
    add_multi_allelic(pop, 500, seed=45, three_rate=0.002)
    gpu.upload_population(pop)
    hh = gpu.hetero_homo()
    codes = pop.codes().astype(np.int64)
    plain = np.ones(pop.n_loci, dtype=bool); plain[pop.multi_rows] = False
    n1, n2, n3 = ((codes[plain] == c).sum(0) for c in (1, 2, 3))
    cells = pop.multi_cells.astype(np.int64)
    many = (cells == 0xFF).sum(0)
    single = ((cells != 0) & (cells != 0xFF) & (cells >> 4 == 0)).sum(0)
    same = ((cells != 0xFF) & (cells >> 4 != 0) & (cells >> 4 == (cells & 15))).sum(0)
    diff = ((cells != 0xFF) & (cells >> 4 != 0) & (cells >> 4 != (cells & 15))).sum(0)
    total = n1 + 2 * n2 + n3 + single + 2 * same + 2 * diff + 3 * many
    assert np.array_equal(hh[:, 0], total) and np.array_equal(hh[:, 1], total) and not hh[:, 2].any() and not hh[:, 6].any()
    assert np.array_equal(hh[:, 3], n2 + same + 2 * diff + 2 * many)
    assert np.array_equal(hh[:, 4], 2 * diff + many)
    assert np.array_equal(hh[:, 5], n1 + n3 + single)
    # locations: 9 cities in 3 countries; a city with fewer than 20 QC-pass samples takes its country's aggregate
    n = pop.n_genomes
    city = (np.arange(n) % 9).astype(np.uint32)
    city[:300] = (np.arange(300) % 8).astype(np.uint32)                   # city 8 is small
    country = (9 + city // 3).astype(np.uint32)
    qc = (np.arange(n) % 6 != 5).astype(np.uint8)
    members = [np.flatnonzero(city == c) for c in range(9)] + [np.flatnonzero(country == 9 + k) for k in range(3)]
    fis = location_fis(hh, members, city, country, qc, 20)
    het, tot = (hh[:, 4] + hh[:, 5]).astype(np.float64), hh[:, 0].astype(np.float64)
    for g in range(n):
        loc = city[g] if qc[members[city[g]]].sum() >= 20 else country[g]
        m = members[loc]
        want = 0.0
        if tot[m].sum() > 0 and tot[g] > 0:
            h_exp = het[m].sum() / tot[m].sum()
            want = (h_exp - het[g] / tot[g]) / h_exp
        assert fis[g] == want, g
    assert qc[members[8]].sum() < 20


def test_equivalent_implementations_on_random_shapes():
    """tools/fuzz_paths.py: moment tables (tensor-core and CUDA-core builders) against the every-cell sweeps, tensor-core IBS against
    the popcount kernel, on 25 random shapes / selections / frequency edge values (1 .. 1,500 genomes, 1 .. 60,000 loci)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "fuzz_paths.py"), "25", "11"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "all equal" in r.stdout
