"""Hardy-Weinberg equilibrium and variant QC on the device (kgl_b200_run_hardy / kgl_b200_run_variant_qc): p, mid-p and F bit-equal
to the host restatement (tests/hwe_oracle.py, every term, no early stop) over population widths, 1 to 64 groups, contiguous,
interleaved and random labels, excluded genomes, code-3 cells, multi-allelic rows, one group of 100,000 genomes with rows built for
long walks, far tails and underflow, and more cells than one launch wave; the QC mask equal to the numpy rule; the chain
variant_qc -> ld_prune -> pca; determinism, no interference with the other passes, and every error code."""
import ctypes as C

import numpy as np
import pytest

import fst_oracle as FO
import hwe_oracle as HO
from kgl_gene_b200.flatfile import FlatPopulation, pack_codes
from kgl_gene_b200.synth import add_multi_allelic, make_population

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.close()


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


def random_codes(n, l, seed, missing=0.0, groups=None, n_groups=1, inbreeding=0.0):
    """Codes from a frequency per (locus, group), part of the loci with a heterozygote deficit or excess, `missing` coded 3."""
    rng = np.random.default_rng(seed)
    p = rng.beta(0.4, 0.6, size=(l, max(n_groups, 1)))
    lab = np.zeros(n, dtype=np.int64) if groups is None else np.where(groups == 0xFF, 0, groups).astype(np.int64)
    q = p[:, lab]
    codes = rng.binomial(2, q).astype(np.uint8)
    if inbreeding:
        ibd = rng.random((l, n)) < inbreeding                       # both copies of one draw: heterozygote deficit
        codes[ibd] = (2 * (rng.random((l, n)) < q))[ibd].astype(np.uint8)
        het = (rng.random((l, 1)) < 0.1) & (rng.random((l, n)) < 0.3)   # some loci with an excess
        codes[het] = 1
    if missing:
        codes[rng.random((l, n)) < missing] = 3
    return codes


def upload(gpu, codes, superpop=None):
    l, n = codes.shape
    sp = np.zeros(n, dtype=np.uint8) if superpop is None else superpop
    pop = FlatPopulation(np.arange(1000, 1000 + 10 * l, 10, dtype=np.uint32), np.full((6, l), 0.1, dtype=np.float32), sp,
                         pack_codes(codes), n, False)
    gpu.upload_population(pop)
    return pop


def assert_bits(got, want):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    bad = np.flatnonzero(got.view(np.uint64) != want.view(np.uint64))
    assert bad.size == 0, (bad[:8], got.ravel()[bad[:8]], want.ravel()[bad[:8]])


def check_hardy(gpu, codes, group, n_groups, multi_rows=None):
    """Device p, mid-p and F bit-equal to the oracle; returns the oracle's p."""
    counts = FO.group_counts(codes, group, n_groups)
    p, f = HO.hardy(counts, multi_rows)
    pm, _ = HO.hardy(counts, multi_rows, midp=True)
    got = gpu.hardy(group, n_groups, f=True)
    assert_bits(got["p"], p)
    assert_bits(got["f"], f)
    assert_bits(gpu.hardy(group, n_groups, midp=True)["p"], pm)
    assert not (got["p"] > 1.0).any()
    return p


@pytest.mark.parametrize("n,l,layout,n_groups,miss,excl", [
    (1, 300, "contiguous", 1, 0.05, 0.0),
    (63, 700, "random", 6, 0.01, 0.1),
    (64, 513, "interleaved", 6, 0.01, 0.0),
    (65, 300, "random", 64, 0.01, 0.1),          # most groups hold one genome or none
    (65, 257, "contiguous", 1, 0.0, 0.0),
    (2504, 900, "contiguous", 6, 0.002, 0.0),
    (2504, 400, "interleaved", 1, 0.0, 0.3),
    (2504, 300, "random", 64, 0.01, 0.0),
    (20000, 60, "contiguous", 6, 0.001, 0.0),
    (20000, 40, "random", 64, 0.0, 0.02),
    (20000, 30, "interleaved", 1, 0.02, 0.0),
])
def test_hardy_bit_equal(gpu, n, l, layout, n_groups, miss, excl):
    g = labels(n, n_groups, layout, seed=n + l, excluded=excl)
    codes = random_codes(n, l, seed=n * 3 + l, missing=miss, groups=g, n_groups=n_groups, inbreeding=0.1)
    upload(gpu, codes)
    check_hardy(gpu, codes, g, n_groups)


def row(n, n0, n1, n2, rng):
    r = np.array([0] * n0 + [1] * n1 + [2] * n2 + [3] * (n - n0 - n1 - n2), dtype=np.uint8)
    rng.shuffle(r)
    return r


def built_rows(n, rng):
    """Rows aimed at the edges of the walk for one group of n genomes."""
    h, a = n // 2, int(n * 0.25925)
    specs = [
        (0, n, 0),                                    # all heterozygous: P(obs) underflows at large n, p = 0
        (h, 0, n - h),                                # all homozygous, no heterozygote
        (n // 4, n // 2, n - n // 4 - n // 2),        # exact HWE proportions at p = 1/2
        (n, 0, 0), (0, 0, n),                         # monomorphic
        (0, 0, 0),                                    # v = 0: NaN
        (n - 1, 1, 0), (n - 2, 0, 2), (n - 3, 2, 1),  # a handful of rare copies
        (int(n * 0.81), int(n * 0.18), n - int(n * 0.81) - int(n * 0.18)),
        (a, n - 2 * a, a),                            # far below the mode: P(obs) ~ 1.8e-30 at 100,000 genomes
        (int(n * 0.245), int(n * 0.51), n - int(n * 0.245) - int(n * 0.51)),                # above the mode
        (int(n * 0.3), int(n * 0.3), n - int(n * 0.6)),
        (int(n * 0.49), int(n * 0.02), n - int(n * 0.49) - int(n * 0.02)),
        (int(n * 0.9), int(n * 0.05), int(n * 0.02)),  # with code-3 cells
    ]
    return np.stack([row(n, *s, rng) for s in specs])


def test_one_group_of_100k_genomes(gpu):
    """Long walks: up to 50,001 support values; the far tails where the early stop must look at N as well as S."""
    n = 100_000
    rng = np.random.default_rng(7)
    codes = np.concatenate([built_rows(n, rng), random_codes(n, 8, seed=5, missing=0.001, inbreeding=0.02)])
    upload(gpu, codes)
    g = np.zeros(n, dtype=np.uint8)
    p = check_hardy(gpu, codes, g, 1)
    assert p[0, 0] == 0.0 and p[3, 0] == 1.0 and np.isnan(p[5, 0])
    assert 0.0 < p[10, 0] < 1e-25
    full = int(HO.walk_terms(*(FO.group_counts(codes, g, 1)[:, 0, c] for c in range(3))).sum())
    assert 0 < gpu.last_hardy_terms() < full


def test_every_count_of_small_groups(gpu):
    """Every (n0, n1, n2) of a group of 40 genomes (code 3 for the rest), and the counts at 188 genomes where an exact tie rounds
    just above P(obs) and only the 2^-40 margin keeps it in N."""
    n = 188
    rng = np.random.default_rng(17)
    specs = [(n0, n1, n2) for v in range(41) for n1 in range(v + 1) for n2 in range(v - n1 + 1) for n0 in (v - n1 - n2,)]
    specs += [(155, 30, 3), (3, 30, 155)]
    codes = np.stack([row(n, *s, rng) for s in specs])
    upload(gpu, codes)
    p = check_hardy(gpu, codes, np.zeros(n, dtype=np.uint8), 1)
    assert p[-1, 0] == p[-2, 0] == HO.exact(155, 30, 3)


def test_built_rows_across_groups(gpu):
    """The built rows in 6 contiguous groups of 2,504 with excluded genomes, and in 64 interleaved groups."""
    n = 2504
    rng = np.random.default_rng(9)
    codes = np.concatenate([built_rows(n, rng), random_codes(n, 100, seed=4, missing=0.01, inbreeding=0.1)])
    upload(gpu, codes)
    check_hardy(gpu, codes, labels(n, 6, "contiguous", 1, excluded=0.05), 6)
    check_hardy(gpu, codes, labels(n, 64, "interleaved", 1), 64)


def test_superpop_labels_and_multi_allelic(gpu):
    pop, _ = make_population(700, 2000, seed=3, missing_rate=0.004)
    pop = add_multi_allelic(pop, 60, seed=3)
    gpu.upload_population(pop)
    codes = pop.codes()
    counts = FO.group_counts(codes, pop.superpop, 6)
    p, f = HO.hardy(counts, pop.multi_rows)
    got = gpu.hardy(f=True)
    assert got["p"].shape == (2000, 6)
    assert_bits(got["p"], p)
    assert_bits(got["f"], f)
    assert np.isnan(got["p"][pop.multi_rows]).all() and np.isnan(got["f"][pop.multi_rows]).all()
    pooled = np.zeros(700, dtype=np.uint8)
    assert_bits(gpu.hardy(pooled, 1)["p"], HO.hardy(FO.group_counts(codes, pooled, 1), pop.multi_rows)[0])


def waves_cells(gpu):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return sms * 16 * 128       # k_hwe: 128 threads a block, at most 16 blocks (2,048 threads) an SM


def test_more_cells_than_one_wave(gpu):
    """k_hwe over more cells than one launch wave, with a partial last block; the sort over several tiles of cub's radix pass."""
    G = 6
    l = waves_cells(gpu) * 3 // (2 * G) + 13
    assert (l * G) % 128 != 0
    n = 65
    g = labels(n, G, "random", 3, excluded=0.05)
    codes = random_codes(n, l, seed=8, missing=0.01, groups=g, n_groups=G, inbreeding=0.2)
    upload(gpu, codes)
    check_hardy(gpu, codes, g, G)


def qc_reference(gpu, codes, pop, g, G, multi_rows=None, keep=None, **thr):
    counts = FO.group_counts(codes, g, G) if thr.get("min_hwe_p") else None
    p = HO.hardy(counts, multi_rows, midp=thr.pop("midp", False))[0] if counts is not None else None
    pooled = FO.group_counts(codes, np.zeros(codes.shape[1], dtype=np.uint8), 1)[:, 0, :]
    return HO.variant_qc(pooled, codes.shape[1], p, keep, multi_rows, **thr)


def test_variant_qc_rule(gpu):
    pop, _ = make_population(1500, 4000, seed=12, missing_rate=0.02)
    pop = add_multi_allelic(pop, 40, seed=12)
    gpu.upload_population(pop)
    codes = pop.codes()
    rng = np.random.default_rng(2)
    gpu_keep = (rng.random(4000) < 0.9).astype(np.uint8)
    g = pop.superpop
    cases = [dict(min_call_rate=0.985), dict(min_maf=0.05), dict(min_hwe_p=1e-6), dict(min_hwe_p=0.05, midp=True),
             dict(min_call_rate=0.98, min_maf=0.01, min_hwe_p=1e-4), dict(min_call_rate=1.0), dict(min_maf=0.5), dict(min_hwe_p=1.0)]
    k0, n0 = gpu.variant_qc()                     # no filter: every locus but the multi-allelic rows
    assert n0 == 4000 - 40 and int(k0.sum()) == n0 and not k0[pop.multi_rows].any()
    for thr in cases:
        for keep in (None, gpu_keep):
            want, n_want = qc_reference(gpu, codes, pop, g, 6, pop.multi_rows, keep, **dict(thr))
            got, n_got = gpu.variant_qc(keep=keep, **thr)
            assert np.array_equal(got, want), thr
            assert n_got == n_want
    # explicit labels: one pooled group, and 9 random groups
    for lab, G in ((np.zeros(1500, dtype=np.uint8), 1), (labels(1500, 9, "random", 4, excluded=0.1), 9)):
        want, n_want = qc_reference(gpu, codes, pop, lab, G, pop.multi_rows, None, min_hwe_p=1e-3, min_maf=0.02)
        got, n_got = gpu.variant_qc(min_hwe_p=1e-3, min_maf=0.02, group=lab, n_groups=G)
        assert np.array_equal(got, want) and n_got == n_want


def test_qc_chain_ld_prune_pca(gpu):
    pop, _ = make_population(800, 3000, seed=31, missing_rate=0.01)
    gpu.upload_population(pop)
    codes = pop.codes()
    keep, n_kept = gpu.variant_qc(min_call_rate=0.98, min_maf=0.01, min_hwe_p=1e-6)
    assert 0 < n_kept < 3000
    pooled = FO.group_counts(codes, np.zeros(800, dtype=np.uint8), 1)[:, 0, :].astype(np.int64)
    s, v = pooled[:, 1] + 2 * pooled[:, 2], pooled[:, 0] + pooled[:, 1] + pooled[:, 2]
    poly = (keep != 0) & (s > 0) & (s < 2 * v)
    pr, n_pr = gpu.ld_prune(0.2, 100, keep=keep)
    assert not (pr & ~keep).any()
    res = gpu.pca(k=4, seed=1, keep=keep)
    assert res["n_loci_used"] == int(poly.sum()) == n_kept   # MAF >= 0.01 leaves only polymorphic loci
    res2 = gpu.pca(k=4, seed=1, keep=pr)
    assert res2["n_loci_used"] == n_pr


def test_second_call_bit_identical(gpu):
    n, l = 2504, 700
    g = labels(n, 6, "random", 5, excluded=0.02)
    codes = random_codes(n, l, seed=13, missing=0.01, groups=g, n_groups=6, inbreeding=0.1)
    upload(gpu, codes)
    a = gpu.hardy(g, 6, f=True)
    gpu.hardy(labels(n, 64, "interleaved", 2), 64, midp=True)       # other labels and shapes in between
    qa = gpu.variant_qc(min_hwe_p=1e-3, group=g, n_groups=6)
    b = gpu.hardy(g, 6, f=True)
    qb = gpu.variant_qc(min_hwe_p=1e-3, group=g, n_groups=6)
    assert_bits(a["p"], b["p"])
    assert_bits(a["f"], b["f"])
    assert np.array_equal(qa[0], qb[0]) and qa[1] == qb[1]
    t = gpu.last_hardy_terms()
    gpu.variant_qc(min_hwe_p=1e-3, group=g, n_groups=6)
    assert gpu.last_hardy_terms() == t > 0


def test_no_interference(gpu):
    pop, _ = make_population(400, 3000, seed=21, missing_rate=0.003)
    gpu.upload_population(pop)
    codes = pop.codes()
    gpu.select_loci(spacing=0)
    gpu.count_and_inbreed()
    lc_pass = gpu.fetch_locus_counts()
    g = labels(400, 6, "random", 2, excluded=0.1)
    before = (gpu.allele_count(), gpu.group_counts(g, 6), gpu.fst(g, 6, "hudson", per_locus=True), gpu.group_counts())
    gpu.hardy(g, 6, f=True)
    gpu.variant_qc(min_call_rate=0.99, min_maf=0.01, min_hwe_p=1e-4)
    gpu.hardy(midp=True)
    after = (gpu.allele_count(), gpu.group_counts(g, 6), gpu.fst(g, 6, "hudson", per_locus=True), gpu.group_counts())
    assert np.array_equal(gpu.fetch_locus_counts(), lc_pass)
    for x, y in zip(before[0], after[0]):
        assert np.array_equal(x, y)
    assert np.array_equal(before[1], after[1]) and np.array_equal(before[3], after[3])
    assert np.array_equal(before[3], FO.group_counts(codes, pop.superpop, 6))
    assert_bits(before[2]["fst"], after[2]["fst"])
    assert_bits(before[2]["per_locus"], after[2]["per_locus"])


def test_errors(gpu):
    from kgl_gene_b200.capi import HardyOptions, KglB200, KglError, QcOptions
    fresh = KglB200(0)
    fresh.n_loci, fresh.n_genomes = 300, 40
    z = np.zeros(40, dtype=np.uint8)
    with pytest.raises(KglError, match=r"run_hardy failed \[2\]"):
        fresh.hardy(z, 1)
    with pytest.raises(KglError, match=r"run_variant_qc failed \[2\]"):
        fresh.variant_qc()
    codes = random_codes(40, 300, seed=3)
    fresh.upload_genotypes(pack_codes(codes), 40)
    with pytest.raises(KglError, match=r"run_hardy failed \[2\]"):             # group NULL without super-population labels
        fresh.hardy()
    with pytest.raises(KglError, match=r"run_variant_qc failed \[2\]"):
        fresh.variant_qc(min_hwe_p=1e-6)
    fresh.variant_qc(min_maf=0.01)                                             # no test: no labels needed
    bad = labels(40, 3, "random", 1)
    bad[7] = 3
    for args in ((bad, 3), (z, 0), (z, 65)):
        with pytest.raises(KglError, match=r"run_hardy failed \[1\]"):
            fresh.hardy(*args)
        with pytest.raises(KglError, match=r"run_variant_qc failed \[1\]"):
            fresh.variant_qc(min_hwe_p=1e-6, group=args[0], n_groups=args[1])
    for thr in (dict(min_call_rate=-0.1), dict(min_call_rate=1.5), dict(min_call_rate=float("nan")), dict(min_maf=0.51),
                dict(min_maf=-1e-9), dict(min_maf=float("nan")), dict(min_hwe_p=1.01), dict(min_hwe_p=-0.5), dict(min_hwe_p=float("nan"))):
        with pytest.raises(KglError, match=r"run_variant_qc failed \[1\]"):
            fresh.variant_qc(**thr)
    p = np.zeros((300, 1))
    opt = HardyOptions(group=z.ctypes.data, n_groups=1, midp=2)
    assert fresh.lib.kgl_b200_run_hardy(fresh.h, C.byref(opt), C.c_void_p(p.ctypes.data), None) == 1
    opt.midp = 0
    assert fresh.lib.kgl_b200_run_hardy(fresh.h, C.byref(opt), None, None) == 1
    assert fresh.lib.kgl_b200_run_hardy(fresh.h, None, C.c_void_p(p.ctypes.data), None) == 1
    out, n = np.zeros(300, dtype=np.uint8), C.c_uint64(0)
    q = QcOptions(midp=2)
    assert fresh.lib.kgl_b200_run_variant_qc(fresh.h, C.byref(q), C.c_void_p(out.ctypes.data), C.byref(n)) == 1
    q.midp = 0
    assert fresh.lib.kgl_b200_run_variant_qc(fresh.h, C.byref(q), None, C.byref(n)) == 1
    assert fresh.lib.kgl_b200_run_variant_qc(fresh.h, C.byref(q), C.c_void_p(out.ctypes.data), None) == 1
    assert fresh.lib.kgl_b200_run_variant_qc(fresh.h, None, C.c_void_p(out.ctypes.data), C.byref(n)) == 1
    # the context still works after every refusal, and a zero-initialised struct filters nothing
    assert fresh.lib.kgl_b200_run_variant_qc(fresh.h, C.byref(q), C.c_void_p(out.ctypes.data), C.byref(n)) == 0
    assert n.value == 300 and out.all()
    assert_bits(fresh.hardy(z, 1)["p"], HO.hardy(FO.group_counts(codes, z, 1))[0])
    fresh.close()
