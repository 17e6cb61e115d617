"""Pins the CPU oracle (oracle/kgl_oracle.c) against outputs of the reference's own code.

tests/golden/*.npz were produced by tests/golden/make_golden.py from oracle/_ref/kgl_ref_harness, i.e. the reference's
translation units compiled where they lie. Integer results must be bit-exact; here the double results are bit-exact
too, because the oracle performs the same IEEE operations in the same order.
"""
import numpy as np
import pytest

import oracle_py as O
from conftest import results_matrix

SUPER_POPS = ["AFR", "AMR", "EAS", "EUR", "SAS", "ALL"]


def test_locus_selection_matches_reference(golden):
    name, pop, ref, sel_kw = golden
    sel = O.select_all_pops(pop, **sel_kw)
    for k, sp in enumerate(SUPER_POPS):
        assert np.array_equal(pop.offsets[sel[k] == 1], ref["selected_offsets_" + sp]), (name, sp)


@pytest.mark.parametrize("algo", ["Simple", "RitlandLocus"])
def test_closed_form_estimators_bit_exact(golden, algo):
    name, pop, ref, sel_kw = golden
    sel = O.select_all_pops(pop, **sel_kw)
    counts, freqs = results_matrix(O.inbreed(pop, sel, algo))
    present = ref["genome_present"] == 1
    assert np.array_equal(counts[present], ref[algo + "_counts"][present])
    assert np.array_equal(freqs[present], ref[algo + "_freqs"][present])          # same ops, same order: bit-exact
    mine = O.inbreed(pop, sel, algo)["inbred_allele_sum"]
    assert np.array_equal(mine[present], ref[algo + "_coeff"][present], equal_nan=True)      # NaN: a genome without any term


def test_compensated_sums_agree_on_golden(golden):
    """oracle_py.inbreed(compensated=True), what the device's fixed-point sums are compared with at millions of loci, agrees
    with the reference's order to rounding on the golden cases."""
    name, pop, ref, sel_kw = golden
    sel = O.select_all_pops(pop, **sel_kw)
    for algo in ("Simple", "RitlandLocus"):
        a, b = O.inbreed(pop, sel, algo), O.inbreed(pop, sel, algo, compensated=True)
        assert np.array_equal(results_matrix(a)[0], results_matrix(b)[0]), (name, algo)
        assert np.allclose(results_matrix(b)[1], results_matrix(a)[1], rtol=1e-12, atol=0), (name, algo)
        assert np.allclose(b["inbred_allele_sum"], a["inbred_allele_sum"], rtol=1e-10, atol=1e-12, equal_nan=True), (name, algo)


def test_compensated_sums_are_exact():
    """Where one term repeats over 2 M loci (64 genomes heterozygous everywhere, one frequency) the compensated sums are
    exactly L times the term, while the reference's locus-by-locus double sum drifts (5e-11 relative; Simple's F, whose
    denominator cancels, moves by 3e-7)."""
    from fractions import Fraction
    from kgl_gene_b200.flatfile import FlatPopulation

    def repeated(n_loci):
        packed = np.zeros((n_loci, 16), np.uint8)
        packed[:, :8] = 0xFF                                                          # code 1 in every cell
        return FlatPopulation((1000 + 10 * np.arange(n_loci)).astype(np.uint32), np.full((6, n_loci), np.float32(1e-4)),
                              np.zeros(64, np.uint8), packed, 64, False)
    one = repeated(1)
    term = O.inbreed(one, O.select_all_pops(one), "Simple", compensated=True)[0]
    n_loci = 2_000_000
    many = repeated(n_loci)
    sel = O.select_all_pops(many)
    exact = O.inbreed(many, sel, "Simple", compensated=True)[0]
    drift = O.inbreed(many, sel, "Simple")[0]
    for f in ("major_homo_freq", "major_hetero_freq", "minor_homo_freq"):
        want = float(Fraction(float(term[f])) * n_loci)
        assert exact[f] == want, f
        assert drift[f] != want, f


def test_loglikelihood_grid_bit_exact(golden):
    name, pop, ref, sel_kw = golden
    sel = O.select_all_pops(pop, **sel_kw)
    ll = O.loglik_grid(pop, sel, ref["ll_grid"])
    present = ref["genome_present"] == 1
    assert np.array_equal(ll[present], ref["ll_grid_values"][present])


def test_loglikelihood_optimum_within_optimiser_tolerance(golden):
    """The reference stops Nelder-Mead at xtol_abs 1e-6 (calc.cpp:138) from random starts. The oracle returns the
    maximiser over the feasible region (no homozygous probability clamped), located with the derivative; for every genome
    of every fixture the reference's returned coefficient lies within the optimiser tolerance of it."""
    name, pop, ref, sel_kw = golden
    sel = O.select_all_pops(pop, **sel_kw)
    opt = O.inbreed(pop, sel, "Loglikelihood")["inbred_allele_sum"]
    present = ref["genome_present"] == 1
    close = np.abs(ref["Loglikelihood_coeff"][present] - opt[present]) < 2e-6
    if name == "multi_allelic_unphased":
        # Two of the 30 genomes carry a homozygous allele so rare that its term is clamped (calc.cpp:108) over a whole interval
        # of f; left of it the CLAMPED objective keeps growing with the heterozygous terms and Nelder-Mead ends at -0.618,
        # outside the feasible region the product (and this oracle) maximise over. Documented waiver (DESIGN 8); logLikelihood
        # itself is pinned bit for bit on this fixture by the grid test above.
        assert close.sum() >= close.size - 2
        return
    assert np.all(close)
    # dLL/df vanishes at the oracle optimum: the objective is flat to first order there (checked by symmetric differences)
    h = 1e-5
    for g in np.flatnonzero(present)[:8]:
        vals = O.loglik_grid(pop, sel, np.array([opt[g] - h, opt[g], opt[g] + h]))[g]
        assert vals[1] >= vals[0] and vals[1] >= vals[2]


def test_hallme_fifty_sweeps_bit_exact(golden):
    """Q1: the reference runs exactly 50 EM sweeps from its 5th random start; with std::random_device pinned in the
    harness the start is known, and the oracle's 50 sweeps reproduce the result bit for bit."""
    name, pop, ref, sel_kw = golden
    sel = O.select_all_pops(pop, **sel_kw)
    start = np.full(pop.n_genomes, ref["hall_start_sequence"][4])
    mine = O.inbreed(pop, sel, "HallME", start=start, sweeps=50)["inbred_allele_sum"]
    present = ref["genome_present"] == 1
    assert np.array_equal(mine[present], ref["HallME_coeff"][present], equal_nan=True)


def test_allele_summaries_match_variantdb(golden):
    """VariantDBVariant (kgl_variant_db_variant.cpp): het = cells == 1, minorHom = cells == 2 of the locus' A>G column.
    Dropped cells (code 3) carry a different allele in the harness, so they land in the column's refHom count."""
    name, pop, ref, sel_kw = golden
    lc, gc = O.allele_count(pop)
    m = ref["variant_present"] == 1
    sv = ref["summary_by_variant"]
    if pop.n_multi:
        # a multi-allelic locus has one VariantDBVariant column per allele; the harness reports the "A>G" one (slot 0): copies of
        # slot 0 in the side cells (0xFF = G, G, C). The matrix row itself only says hom-ref / not (codes 0 / 3).
        cells = pop.multi_cells.astype(np.int64)
        copies = ((cells & 15) == 1).astype(np.int64) + ((cells >> 4) == 1).astype(np.int64)
        copies[cells == 0xFF] = 2
        rows = pop.multi_rows
        on = m[rows]
        assert np.array_equal(sv[rows][on, 1], (copies == 1).sum(axis=1)[on]) and np.array_equal(sv[rows][on, 2], (copies == 2).sum(axis=1)[on])
        assert np.array_equal(lc[rows, 0], (cells == 0).sum(axis=1)) and np.array_equal(lc[rows, 3], (cells != 0).sum(axis=1))
        m = m.copy(); m[rows] = False
    assert np.array_equal(sv[m, 1], lc[m, 1]) and np.array_equal(sv[m, 2], lc[m, 2])
    assert np.array_equal(sv[m, 0], (lc[m, 0] + lc[m, 3]).astype(np.uint64))
    assert np.array_equal(lc.sum(axis=1), np.full(pop.n_loci, pop.n_genomes))
    assert np.array_equal(gc.sum(axis=1), np.full(pop.n_genomes, pop.n_loci))
    if pop.n_multi:
        return          # summaryByGenome runs over the per-allele columns of the multi-allelic loci as well
    # summaryByGenome runs over every distinct variant column, including the harness' "A>T" stand-in for a dropped cell
    # (one copy -> counted as heterozygous): het = n1 + n3, minorHom = n2, refHom = columns - het - minorHom.
    sg = ref["summary_by_genome"]
    present = ref["genome_present"] == 1
    n_columns = int(ref["variantdb_meta"][0])
    assert np.array_equal(sg[present, 1], gc[present, 1] + gc[present, 3]) and np.array_equal(sg[present, 2], gc[present, 2])
    assert np.array_equal(sg[present, 0], n_columns - sg[present, 1] - sg[present, 2])
    assert np.array_equal(ref["summary_population"], sg[present].sum(axis=0))


def _listed_slots(pop):
    """bool[M][3]: allele slots the multi-allelic locus lists (a slot is listed up to the last one that has a frequency anywhere)."""
    has = ~np.isnan(pop.multi_af).all(axis=0)
    n_slots = np.where(has.any(axis=1), 3 - np.argmax(has[:, ::-1], axis=1), 0)
    return np.arange(3)[None, :] < n_slots[:, None]


def test_calc_fws_restatement_matches_reference(golden):
    """oracle_py.fws_bins against the reference's CalcFWS::calcFwsStatistics (kga_PfEMP/kga_analysis_PfEMP_FWS.cpp:15-101,
    P7FrequencyFilter kgl_variant_filter_Pf7.cpp:20-66) run by the harness on a population whose variants carry INFO AF -- the
    alleles of the multi-allelic loci each with their own. Side cells with more than two variants (0xFF) do not record which
    alleles the genome carries: those genomes (and, for the per-variant map, those loci) are compared through the ordinary rows only."""
    from kgl_gene_b200.fws import FWS_BINS
    name, pop, ref, _ = golden
    want, rows = O.fws_bins(pop, 5, FWS_BINS)                       # [bin][genome][code]
    got = ref["fws_genome"]                                          # [genome][bin]{refHom, het, minorHom}
    w = np.transpose(want, (1, 0, 2))
    known = np.ones(pop.n_genomes, dtype=bool)
    if pop.n_multi:
        known = ~(pop.multi_cells == 0xFF).any(axis=0)
        assert known.sum() > pop.n_genomes // 2 or name.startswith("random")      # the fixtures keep most genomes
    # An allele that only genomes with a 0xFF cell carry is a variant of the reference population (the harness gives such a genome
    # slot 0 twice and slot 1 once) but not of the flat one, which does not know what the cell holds: one more column in its bin.
    extra = np.zeros(len(FWS_BINS), dtype=np.uint64)
    if pop.n_multi:
        copies = O.multi_allele_copies(pop)
        for m_i in np.flatnonzero((pop.multi_cells == 0xFF).any(axis=1)):
            for a in (0, 1):
                v = float(pop.multi_af[5, m_i, a])
                if not (copies[m_i, a] > 0).any() and not np.isnan(v):
                    for b, (lo, hi) in enumerate(FWS_BINS):
                        extra[b] += np.uint64(v >= lo and not v >= hi)
    assert np.array_equal(got[known, :, 1], w[known, :, 1]) and np.array_equal(got[known, :, 2], w[known, :, 2])
    assert np.array_equal(got[known, :, 0], w[known, :, 0] + w[known, :, 3] + extra[None, :])   # a cell with another allele has no copy of this variant
    assert np.array_equal(got.sum(axis=2), np.broadcast_to((rows + extra)[None, :], got.shape[:2]))   # every genome sees every column of its bin
    lc, _ = O.allele_count(pop)
    m = ref["fws_variant_present"] == 1
    ordinary = np.ones(pop.n_loci, dtype=bool)
    if pop.n_multi:
        ordinary[pop.multi_rows] = False
    assert np.array_equal(m[ordinary], ((lc[:, 1] + lc[:, 2]) > 0)[ordinary])
    m = m & ordinary
    fv = ref["fws_variant"]
    assert np.array_equal(fv[m, 1], lc[m, 1]) and np.array_equal(fv[m, 2], lc[m, 2]) and np.array_equal(fv[m, 0], lc[m, 0] + lc[m, 3])
    if pop.n_multi:
        copies = O.multi_allele_copies(pop)                                        # [M][3][N]
        sel = _listed_slots(pop) & ~(pop.multi_cells == 0xFF).any(axis=1)[:, None]
        present = ref["fws_multi_variant_present"] == 1
        assert (sel.sum() > pop.n_multi or name.startswith("random")) and np.array_equal((copies > 0).any(axis=2)[sel], present[sel])
        sel &= present
        for c in range(3):
            assert np.array_equal((copies == c).sum(axis=2)[sel], ref["fws_multi_variant"][:, :, c][sel]), (name, c)


def test_hetero_homo_rule_matches_reference(golden):
    """kgl_gene_b200.fws.hetero_homo_summary (host mirror of HeteroHomoZygous::updateVariantAnalysisType,
    kga_PfEMP/kga_analysis_PfEMP_heterozygous.cpp:61-105) and the oracle's restatement with multi-allelic loci against the
    reference TU run over every offset of every genome."""
    from kgl_gene_b200.fws import hetero_homo_summary
    name, pop, ref, _ = golden
    want = ref["hetero_homo"]
    assert np.array_equal(O.hetero_homo(pop), want), name
    if pop.n_multi:
        return
    _, gc = O.allele_count(pop)
    hh = hetero_homo_summary(gc)
    for j, key in enumerate(["total_variants", "snp_count", "indel_count", "homozygous_minor_alleles", "heterozygous_minor_alleles",
                             "heterozygous_reference_minor_alleles", "homozygous_reference_alleles"]):
        assert np.array_equal(hh[key], want[:, j]), (name, key)


def test_synthetic_generator_matches_numpy():
    from kgl_gene_b200.synth import make_population
    pop, f = make_population(77, 300, seed=5)
    packed = O.synth_genotypes(5, 77, 300, pop.af, pop.superpop, f)
    assert np.array_equal(packed, pop.packed)


def test_ibs_oracle_basic_properties():
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(19, 257, seed=9, missing_rate=0.05)
    ibs = O.ibs(pop)
    assert np.array_equal(ibs, ibs.transpose(1, 0, 2))
    assert np.array_equal(ibs[..., :3].sum(-1), ibs[..., 3])
    codes = pop.codes()
    valid = (codes != 3).sum(axis=0)
    d = np.arange(19)
    assert np.array_equal(ibs[d, d, 2], valid) and np.all(ibs[d, d, 0] == 0)


@pytest.mark.skipif(not O.have_reference_harness(), reason="oracle/_ref not built (needs /root/reference)")
def test_live_reference_run_matches_oracle():
    """Fresh (non-golden) population through the live reference harness, when it exists."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(16, 400, seed=777, spectrum="dense")
    ref = O.run_reference(pop, algos=("Simple", "RitlandLocus"), spacing=15, variantdb=False)
    sel = O.select_all_pops(pop, spacing=15)
    for algo in ("Simple", "RitlandLocus"):
        assert np.array_equal(O.inbreed(pop, sel, algo)["inbred_allele_sum"], ref[algo + "_coeff"])


# ---------------------------------------------------------------------------------------------- scale checkers ----------
@pytest.mark.parametrize("n,l,miss", [(150, 3001, 0.03), (70, 999, 0.0), (1, 40, 0.1), (130, 64, 0.5), (65, 129, 0.2)])
def test_popcount_ibs_restatement_equals_naive_loop(n, l, miss):
    """SURVEY 8c: "plus a popcount CPU restatement for scale" -- thermometer bit-planes + popcount against the naive O(N^2 L) loop."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(n, l, seed=21 + n, missing_rate=miss)
    want = O.ibs(pop)
    assert np.array_equal(O.ibs_band_popcount(pop, 0, n), want)
    if n > 100:
        assert np.array_equal(O.ibs_band_popcount(pop, 64, 130), want[64:130])


def test_inbreed_subset_equals_full_run():
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(90, 4000, seed=14)
    sel = O.select_all_pops(pop, spacing=15)
    some = np.array([3, 89, 40, 0], dtype=np.uint32)
    start = np.linspace(0.05, 0.5, pop.n_genomes)
    for algo, kw in (("Simple", {}), ("RitlandLocus", {}), ("HallME", dict(start=start, sweeps=50)), ("Loglikelihood", {})):
        assert O.inbreed(pop, sel, algo, genomes=some, **kw).tobytes() == O.inbreed(pop, sel, algo, **kw)[some].tobytes()


def test_parallel_allele_count_is_exact():
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(333, 5000, seed=15, missing_rate=0.02)
    lc, gc = O.allele_count(pop)
    codes = pop.codes()
    for c in range(4):
        assert np.array_equal(lc[:, c], (codes == c).sum(1)) and np.array_equal(gc[:, c], (codes == c).sum(0))


@pytest.mark.skipif(not O.have_reference_harness(), reason="oracle/_ref/kgl_ref_harness not built (make -C oracle ref)")
@pytest.mark.parametrize("seed", [int(x) for x in __import__("os").environ.get("KGL_ORACLE_FUZZ_SEEDS", "1,2,3,4,5,6").split(",")])
def test_oracle_pinned_on_random_populations(seed):
    """The pins above, on populations and selections drawn at random and run through the reference's translation units on the
    spot (oracle/_ref/kgl_ref_harness) instead of the committed fixtures: locus selection, Simple / RitlandLocus (counts, sums and
    coefficients), logLikelihood on a grid and 50 HallME sweeps -- all bit for bit -- the VariantDBVariant summaries, CalcFWS and
    the hetero/homo records."""
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    rng = np.random.default_rng(seed)
    n, l = int(rng.choice([3, 20, 45, 70])), int(rng.choice([60, 400, 1500]))
    pop, _ = make_population(n, l, seed=int(rng.integers(1, 10**6)), spectrum=str(rng.choice(["sfs", "dense"])),
                             missing_rate=float(rng.choice([0.0, 0.02])), missing_af_rate=float(rng.choice([0.0, 0.05])),
                             grouped=bool(rng.integers(0, 2)), unphased=bool(rng.integers(0, 3) == 0))
    poke = int(rng.integers(0, 3))
    if poke == 1:
        pop.af[:, ::7] = np.float32(rng.choice([0.995, 1.0, 0.5]))
    elif poke == 2:
        pop.af[:, 3::11] = np.float32(rng.choice([0.0005, 0.0, 1e-7]))
    if l >= 400 and rng.integers(0, 2):
        add_multi_allelic(pop, int(rng.choice([10, l // 8])), seed=int(rng.integers(1, 10**6)))
    sel_kw = dict(spacing=int(rng.choice([0, 0, 15, 200])), min_af=float(rng.choice([0.0, 0.01, 0.1])), max_af=float(rng.choice([1.0, 0.45])))
    if rng.integers(0, 2):
        lo, hi = sorted(rng.integers(0, l, size=2).tolist())
        sel_kw.update(lower=int(pop.offsets[lo]), upper=int(pop.offsets[hi]))
    count = int(rng.choice([1, 7, 100, 5000]))
    ref = O.run_reference(pop, grid=9, fws=True, seed=int(rng.integers(1, 100)), count=count, **sel_kw)
    ref.pop("_stderr", None)
    sel_kw.setdefault("lower", 0); sel_kw.setdefault("upper", 10**9)
    # the count-limited walk of the window loop (RetrieveLociiVector::getLociiCount, kga_analysis_inbreed_locus.cpp:159-183)
    counted = O.select_all_pops(pop, count=count, mode=1, **sel_kw)
    for k, sp in enumerate(SUPER_POPS):
        assert np.array_equal(pop.offsets[counted[k] == 1], ref["counted_offsets_" + sp]), (seed, sp, count)
    case = (f"random-{seed}", pop, ref, sel_kw)
    test_locus_selection_matches_reference(case)
    for algo in ("Simple", "RitlandLocus"):
        test_closed_form_estimators_bit_exact(case, algo)
    test_loglikelihood_grid_bit_exact(case)
    test_hallme_fifty_sweeps_bit_exact(case)
    test_allele_summaries_match_variantdb(case)
    test_calc_fws_restatement_matches_reference(case)
    test_hetero_homo_rule_matches_reference(case)


@pytest.mark.skipif(not O.have_reference_harness(), reason="oracle/_ref/kgl_ref_harness not built (make -C oracle ref)")
def test_loglikelihood_maximiser_against_the_reference_optimiser_on_random_populations():
    """Loglikelihood is parity-unpinned (nlopt's Nelder-Mead from random starts, SURVEY 8c). What can be pinned: on random
    populations the coefficient the reference returns lies within its own tolerance (xtol_abs 1e-6) of the oracle's maximiser for
    almost every genome; where it does not, the oracle's point has the higher likelihood -- except for a few genomes of UNPHASED
    populations, where the reference's simplex leaves the feasible region and finds a higher value of the clamped objective
    (calc.cpp:108; the waiver of DESIGN 8). A campaign of 60 populations (KGL_ORACLE_FUZZ_SEEDS=1..60): 2,825 genomes, 2,790
    within 2e-6, 29 with the oracle strictly better, 6 (all unphased) with the clamped objective higher at the reference's point."""
    import os
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    total = close = better = outside = 0
    for seed in [int(x) for x in os.environ.get("KGL_ORACLE_FUZZ_SEEDS", "1,2,3,4,5,6,7,8").split(",")]:
        rng = np.random.default_rng(1000 + seed)
        n, l = int(rng.choice([20, 45, 70])), int(rng.choice([400, 1500]))
        unphased = bool(rng.integers(0, 3) == 0)
        pop, _ = make_population(n, l, seed=int(rng.integers(1, 10**6)), spectrum=str(rng.choice(["sfs", "dense"])),
                                 missing_rate=float(rng.choice([0.0, 0.02])), missing_af_rate=float(rng.choice([0.0, 0.05])),
                                 grouped=bool(rng.integers(0, 2)), unphased=unphased)
        if rng.integers(0, 2):
            add_multi_allelic(pop, int(rng.choice([10, l // 8])), seed=int(rng.integers(1, 10**6)))
        sel_kw = dict(spacing=int(rng.choice([0, 15])), min_af=float(rng.choice([0.0, 0.01])))
        ref = O.run_reference(pop, algos=("Loglikelihood",), seed=int(rng.integers(1, 100)), variantdb=False, **sel_kw)
        sel = O.select_all_pops(pop, **sel_kw)
        opt = O.inbreed(pop, sel, "Loglikelihood")["inbred_allele_sum"]
        got = ref["Loglikelihood_coeff"]
        for g in np.flatnonzero(ref["genome_present"] == 1):
            if not (np.isfinite(got[g]) and np.isfinite(opt[g])):
                continue
            total += 1
            if abs(got[g] - opt[g]) < 2e-6:
                close += 1
                continue
            ll = O.loglik_grid(pop, sel, np.array([opt[g], got[g]]))[g]
            if ll[0] >= ll[1] - 1e-9 * max(1.0, abs(ll[1])):
                better += 1
            else:
                outside += 1
                assert unphased, (seed, int(g), opt[g], got[g], ll)
    assert total > 200 and close >= 0.97 * total and outside <= 0.01 * total, (total, close, better, outside)
