"""Population differentiation on the device (kgl_b200_run_group_counts / kgl_b200_run_fst): per-group counts equal to numpy's,
exactly, over population widths with and without padding genomes, contiguous, interleaved and random labellings, excluded
genomes, empty groups, 1 to 64 groups, code-3 cells and multi-allelic rows; F_ST, its per-locus terms and its windows bit-equal to
the host restatement (tests/fst_oracle.py) for both estimators; determinism, every error code, and no interference with the
other passes of the context."""
import ctypes as C

import numpy as np
import pytest

import fst_oracle as FO
from kgl_gene_b200.flatfile import FlatPopulation, pack_codes
from kgl_gene_b200.synth import add_multi_allelic, make_population

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.close()


def random_codes(n, l, seed, missing=0.0, groups=None, n_groups=1):
    """Codes with a frequency per (locus, group), so that groups differ; `missing` of the cells coded 3."""
    rng = np.random.default_rng(seed)
    p = rng.beta(0.4, 0.6, size=(l, max(n_groups, 1)))
    lab = np.zeros(n, dtype=np.int64) if groups is None else np.where(groups == 0xFF, 0, groups).astype(np.int64)
    codes = rng.binomial(2, p[:, lab]).astype(np.uint8)
    if missing:
        codes[rng.random((l, n)) < missing] = 3
    return codes


def labels(n, n_groups, layout, seed, excluded=0.0):
    rng = np.random.default_rng(seed)
    if layout == "contiguous":
        g = (np.arange(n) * n_groups // max(n, 1)).astype(np.uint8)
    elif layout == "interleaved":
        g = (np.arange(n) % n_groups).astype(np.uint8)
    else:
        g = rng.integers(0, n_groups, size=n).astype(np.uint8)
    if excluded:
        g[rng.random(n) < excluded] = 0xFF
    return g


def upload(gpu, codes, superpop=None, offsets=None):
    l, n = codes.shape
    off = np.arange(1000, 1000 + 10 * l, 10, dtype=np.uint32) if offsets is None else np.asarray(offsets, dtype=np.uint32)
    sp = np.zeros(n, dtype=np.uint8) if superpop is None else superpop
    pop = FlatPopulation(off, np.full((6, l), 0.1, dtype=np.float32), sp, pack_codes(codes), n, False)
    gpu.upload_population(pop)
    return pop


def check_counts(gpu, codes, group, n_groups):
    got = gpu.group_counts(group, n_groups)
    want = FO.group_counts(codes, group, n_groups)
    assert got.dtype == np.uint32 and got.shape == want.shape
    assert np.array_equal(got, want)
    lc, _ = gpu.allele_count(want_genomes=False)
    excluded = FO.group_counts(codes, np.where(group == 0xFF, 0, 1), 1)[:, 0]
    assert np.array_equal(got.sum(axis=1, dtype=np.uint64) + excluded, lc)        # the groups and the excluded make up run_allele_count
    return got


@pytest.mark.parametrize("n,l,layout,n_groups,miss,excl", [
    (1, 500, "contiguous", 1, 0.0, 0.0),
    (1, 300, "random", 6, 0.05, 0.0),            # five empty groups
    (63, 700, "random", 6, 0.0, 0.1),
    (64, 513, "interleaved", 6, 0.01, 0.0),
    (65, 300, "random", 64, 0.01, 0.1),          # most groups hold one genome or none
    (65, 257, "contiguous", 64, 0.0, 0.0),
    (2504, 1200, "interleaved", 6, 0.002, 0.05),
    (2504, 600, "contiguous", 6, 0.0, 0.0),
    (2504, 400, "random", 64, 0.01, 0.0),
    (2504, 300, "interleaved", 1, 0.0, 0.3),
    (20000, 150, "contiguous", 6, 0.001, 0.0),
    (20000, 100, "random", 64, 0.0, 0.02),
    (20000, 90, "interleaved", 6, 0.02, 0.0),
])
def test_group_counts_exact(gpu, n, l, layout, n_groups, miss, excl):
    g = labels(n, n_groups, layout, seed=n + l, excluded=excl)
    if n_groups == 6 and n > 6:
        g[g == 4] = 0xFF                          # an empty group in the middle
    codes = random_codes(n, l, seed=n * 7 + l, missing=miss, groups=g, n_groups=n_groups)
    upload(gpu, codes)
    check_counts(gpu, codes, g, n_groups)


def many_tiles_per_cta_loci():
    """Loci for which every CTA of k_group_counts takes at least three tiles of 32 rows, the last one partial: its grid is at most
    8 CTAs (2,048 threads of 256) per SM, so at most 8 x SMs tiles run in the first round."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return sms * 8 * 32 * 3 + 17


@pytest.mark.parametrize("n,n_groups,layout", [(65, 6, "interleaved"), (65, 64, "random"), (130, 6, "contiguous")])
def test_many_tiles_per_cta(gpu, n, n_groups, layout):
    """The grid-stride loop over tiles: the barrier at the top of a tile, the counters cleared again, written out per tile."""
    l = many_tiles_per_cta_loci()
    assert l % 32 != 0
    g = labels(n, n_groups, layout, seed=l + n_groups, excluded=0.05)
    codes = random_codes(n, l, seed=n_groups, missing=0.01, groups=g, n_groups=n_groups)
    pop = upload(gpu, codes)
    check_counts(gpu, codes, g, n_groups)
    pairs = None if n_groups == 6 else [(0, 63), (7, 30), (12, 13)]
    for method in ("hudson", "weir_cockerham"):
        check_fst(gpu, codes, g, n_groups, method, pairs=pairs, offsets=pop.offsets, window_bp=100_000, step_bp=40_000)


def test_group_counts_superpop_labels_and_multi_allelic(gpu):
    pop, _ = make_population(700, 2000, seed=3, missing_rate=0.004)
    pop = add_multi_allelic(pop, 60, seed=3)
    gpu.upload_population(pop)
    codes = pop.codes()
    assert (codes[pop.multi_rows] == 3).any()
    got = gpu.group_counts()
    assert got.shape == (2000, 6, 4)
    assert np.array_equal(got, FO.group_counts(codes, pop.superpop, 6))
    # interleave the super-populations: the cached superpop tables must follow a new labelling
    sp = (np.arange(700) % 5).astype(np.uint8)
    gpu.set_genome_superpop(sp)
    assert np.array_equal(gpu.group_counts(), FO.group_counts(codes, sp, 6))
    g = labels(700, 9, "random", seed=1, excluded=0.1)
    check_counts(gpu, codes, g, 9)
    assert np.array_equal(gpu.group_counts(), FO.group_counts(codes, sp, 6))   # explicit labels in between


def assert_bits(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))


def check_fst(gpu, codes, group, n_groups, method, pairs=None, keep=None, offsets=None, window_bp=0, step_bp=0):
    res = gpu.fst(group, n_groups, method, pairs, keep, per_locus=True, window_bp=window_bp, step_bp=step_bp)
    counts = FO.group_counts(codes, group, n_groups)
    pr = FO.all_pairs(n_groups) if pairs is None else np.asarray(pairs, dtype=np.uint32).reshape(-1, 2)
    assert np.array_equal(res["pairs"], pr)
    assert_bits(res["fst"], FO.fst(counts, pr, method, keep))
    assert_bits(res["per_locus"], FO.per_locus(counts, pr, method, keep))
    if window_bp:
        assert_bits(res["windows"], FO.windows(counts, pr, method, offsets, window_bp, step_bp, keep))
    return res


@pytest.mark.parametrize("method", ["hudson", "weir_cockerham"])
def test_fst_bit_equal(gpu, method):
    n, l = 1000, 3000
    g = labels(n, 6, "interleaved", seed=2, excluded=0.05)
    g[17] = 5                                     # group 5: one genome
    g[g == 5] = 0xFF
    g[17] = 5
    codes = random_codes(n, l, seed=11, missing=0.01, groups=g, n_groups=6)
    codes[100:140] = 3                            # all-missing loci
    codes[200:260] = 0                            # monomorphic loci
    codes[300:320] = 2
    rng = np.random.default_rng(5)
    off = np.cumsum(rng.integers(1, 40, size=l)) + 500
    off[2000:2100] += 20000                       # a gap: windows without loci
    off[2100:] += 20000
    pop = upload(gpu, codes, offsets=off)
    off = pop.offsets
    keep = (rng.random(l) < 0.8).astype(np.uint8)
    res = check_fst(gpu, codes, g, 6, method)
    assert np.isfinite(res["fst"]).all()
    check_fst(gpu, codes, g, 6, method, pairs=[(0, 5), (2, 3), (1, 4)], keep=keep)
    res = check_fst(gpu, codes, g, 6, method, keep=keep, offsets=off, window_bp=5000, step_bp=2500)
    assert (res["windows"][:, :, 2] == 0).any() and (res["windows"][:, :, 2] > 0).any()
    check_fst(gpu, codes, g, 6, method, offsets=off, window_bp=777)
    check_fst(gpu, codes, g, 6, method, offsets=off, window_bp=4000, step_bp=7000)     # step > window: gaps between windows
    # NaN: no locus kept
    res = gpu.fst(g, 6, method, keep=np.zeros(l, dtype=np.uint8))
    assert np.isnan(res["fst"]).all()
    # an empty group: its pairs use no locus
    g2 = g.copy()
    g2[g2 == 3] = 0xFF
    res = check_fst(gpu, codes, g2, 6, method)
    assert np.isnan(res["fst"][[i for i, (a, b) in enumerate(res["pairs"]) if 3 in (a, b)]]).all()


def test_fst_window_boundaries(gpu):
    """Offsets on a grid of 10: many loci sit exactly at w step + window (outside window w) and at w step (inside it)."""
    n, l = 300, 700
    g = labels(n, 3, "random", seed=6, excluded=0.05)
    codes = random_codes(n, l, seed=6, missing=0.01, groups=g, n_groups=3)
    off = np.arange(1000, 1000 + 10 * l, 10, dtype=np.uint32)
    upload(gpu, codes, offsets=off)
    for window, step in ((100, 50), (100, 0), (30, 20), (10, 10), (25, 40)):
        for method in ("hudson", "weir_cockerham"):
            res = check_fst(gpu, codes, g, 3, method, offsets=off, window_bp=window, step_bp=step)
            assert res["windows"].shape[1] == 7990 // (step or window) + 1


@pytest.mark.parametrize("method", ["hudson", "weir_cockerham"])
def test_fst_superpop_labels_many_groups_and_padding(gpu, method):
    pop, _ = make_population(2504, 2600, seed=8, missing_rate=0.002)
    pop = add_multi_allelic(pop, 30, seed=8)
    gpu.upload_population(pop)
    codes = pop.codes()
    res = gpu.fst(method=method, per_locus=True)
    counts = FO.group_counts(codes, pop.superpop, 6)
    assert_bits(res["fst"], FO.fst(counts, FO.all_pairs(6), method))
    assert_bits(res["per_locus"], FO.per_locus(counts, FO.all_pairs(6), method))
    g = labels(2504, 40, "random", seed=4, excluded=0.01)
    check_fst(gpu, codes, g, 40, method, pairs=[(0, 39), (5, 6), (12, 30)])


def test_fst_deterministic(gpu):
    codes = random_codes(3000, 5000, seed=12, missing=0.003, groups=labels(3000, 6, "random", 1), n_groups=6)
    pop = upload(gpu, codes)
    g = labels(3000, 6, "random", 1)
    for method in ("hudson", "weir_cockerham"):
        a = gpu.fst(g, 6, method, per_locus=True, window_bp=5000)
        b = gpu.fst(g, 6, method, per_locus=True, window_bp=5000)
        for k in ("fst", "per_locus", "windows"):
            assert_bits(a[k], b[k])
    assert pop.n_genomes == 3000


def test_errors(gpu):
    from kgl_gene_b200.capi import FstOptions, KglB200, KglError
    fresh = KglB200(0)
    fresh.n_loci, fresh.n_genomes = 10, 5
    with pytest.raises(KglError, match=r"run_group_counts failed \[2\]"):
        fresh.group_counts(np.zeros(5, dtype=np.uint8), 1)
    with pytest.raises(KglError, match=r"run_fst failed \[2\]"):
        fresh.fst(np.zeros(5, dtype=np.uint8), 2)
    codes = random_codes(40, 300, seed=3)
    pop = FlatPopulation(np.arange(300, dtype=np.uint32) * 5, np.full((6, 300), 0.1, dtype=np.float32), np.zeros(40, dtype=np.uint8),
                         pack_codes(codes), 40, False)
    fresh.upload_genotypes(pop.packed, 40)
    with pytest.raises(KglError, match=r"run_group_counts failed \[2\]"):      # group NULL without super-population labels
        fresh.group_counts()
    with pytest.raises(KglError, match=r"run_fst failed \[2\]"):
        fresh.fst()
    fresh.upload_loci(pop.af, None)
    g = labels(40, 3, "random", 1)
    with pytest.raises(KglError, match=r"run_fst failed \[2\]"):               # windows without offsets
        fresh.fst(g, 3, window_bp=100)
    fresh.upload_loci(pop.af, pop.offsets[::-1].copy())
    with pytest.raises(KglError, match=r"run_fst failed \[1\]"):               # decreasing offsets
        fresh.fst(g, 3, window_bp=100)
    fresh.upload_loci(pop.af, pop.offsets)
    fresh.set_genome_superpop(pop.superpop)
    bad = g.copy()
    bad[7] = 3
    for args in ((bad, 3), (g, 0), (g, 65)):
        with pytest.raises(KglError, match=r"run_group_counts failed \[1\]"):
            fresh.group_counts(*args)
    with pytest.raises(KglError, match=r"run_fst failed \[1\]"):
        fresh.fst(bad, 3)
    for pairs in ([(1, 1)], [(2, 1)], [(0, 3)]):
        with pytest.raises(KglError, match=r"run_fst failed \[1\]"):
            fresh.fst(g, 3, pairs=pairs)
    with pytest.raises(KglError, match=r"run_fst failed \[1\]"):               # one group: no pair
        fresh.fst(np.zeros(40, dtype=np.uint8), 1)
    with pytest.raises(ValueError, match="pairs is empty"):                  # an empty list is not "every pair"
        fresh.fst(g, 3, pairs=[])
    # a refused call leaves *n_windows as it was
    n_win = C.c_uint64(12345)
    opt = FstOptions(group=bad.ctypes.data, n_groups=3, window_bp=100)
    assert fresh.lib.kgl_b200_run_fst(fresh.h, C.byref(opt), C.c_void_p(np.zeros(3).ctypes.data), None, None, C.byref(n_win)) == 1
    assert n_win.value == 12345
    opt = FstOptions(group=g.ctypes.data, n_groups=3, method=2)
    assert fresh.lib.kgl_b200_run_fst(fresh.h, C.byref(opt), C.c_void_p(np.zeros(3).ctypes.data), None, None, None) == 1
    opt.method = 0
    assert fresh.lib.kgl_b200_run_fst(fresh.h, C.byref(opt), None, None, None, None) == 1
    assert fresh.lib.kgl_b200_run_fst(fresh.h, None, C.c_void_p(np.zeros(3).ctypes.data), None, None, None) == 1
    assert fresh.lib.kgl_b200_run_group_counts(fresh.h, C.c_uint32(3), C.c_void_p(g.ctypes.data), None) == 1
    # the context still works after every refusal
    assert np.array_equal(fresh.group_counts(g, 3), FO.group_counts(codes, g, 3))
    fresh.close()


def test_no_interference(gpu):
    pop, _ = make_population(400, 3000, seed=21, missing_rate=0.003)
    gpu.upload_population(pop)
    codes = pop.codes()
    gpu.select_loci(spacing=0)
    gpu.count_and_inbreed()
    lc_pass = gpu.fetch_locus_counts()
    before = (gpu.allele_count(), gpu.pca(k=4, seed=3), gpu.ld_prune(0.2, 200))
    g = labels(400, 6, "random", 2, excluded=0.1)
    gpu.group_counts(g, 6)
    gpu.fst(g, 6, "weir_cockerham", per_locus=True, window_bp=3000)
    gpu.fst(method="hudson")
    after = (gpu.allele_count(), gpu.pca(k=4, seed=3), gpu.ld_prune(0.2, 200))
    assert np.array_equal(gpu.fetch_locus_counts(), lc_pass)
    for x, y in zip(before[0], after[0]):
        assert np.array_equal(x, y)
    for k in ("eigenvalues", "scores"):
        assert np.array_equal(before[1][k], after[1][k])
    assert np.array_equal(before[2][0], after[2][0]) and before[2][1] == after[2][1]
    assert np.array_equal(gpu.group_counts(), FO.group_counts(codes, pop.superpop, 6))
