"""Genotype PCA on the device (kgl_b200_run_grm_product / kgl_b200_run_pca): the operator bit-equal to the host restatement
(tests/pca_oracle.py), the components against a dense eigendecomposition of Psi, planted ancestry, loadings, determinism, misuse
and no interference with the other Gram users of the context."""
import numpy as np
import pytest

import pca_oracle as P
from kgl_gene_b200.flatfile import pack_codes
from kgl_gene_b200.synth import add_multi_allelic, make_loci, make_population, synth_codes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.close()


def bit_equal(x, y):
    x, y = np.ascontiguousarray(x, dtype=np.float64), np.ascontiguousarray(y, dtype=np.float64)
    return x.shape == y.shape and np.array_equal(x.view(np.uint64), y.view(np.uint64))


def with_monomorphic(pop, every=17):
    """Rows l % every == 0 become monomorphic (all hom-ref or all hom-alt, code-3 cells kept)."""
    codes = pop.codes()
    rows = np.arange(0, pop.n_loci, every)
    codes[rows] = np.where(codes[rows] == 3, 3, np.where(rows[:, None] % 2 == 0, 0, 2))
    pop.packed = pack_codes(codes)
    return pop


def check_product(gpu, pop, cols, seed, keep=None):
    gpu.upload_population(pop)
    x = np.random.default_rng(seed).standard_normal((pop.n_genomes, cols))
    y, m = gpu.grm_product(x, keep=keep)
    want, want_m = P.grm_product(pop.codes(), x, keep)
    assert m == want_m
    assert bit_equal(y, want)


@pytest.mark.parametrize("n,l,miss,cols", [(257, 1001, 0.0, 16),      # no code-3 cell
                                           (63, 3333, 0.002, 17),     # few code-3 cells (indexed)
                                           (1000, 777, 0.03, 48),     # 3 % code-3 cells, still indexed: N L / 64 < 2^16
                                           (1000, 5001, 0.03, 48),    # more than 1.5 % code-3 cells and N L / 64 > 2^16: not indexed
                                           (2, 130, 0.05, 1),
                                           # 20,000 genomes: pass 1 (K = genomes, 157 stages) split in two chunks, red.add into
                                           # the cleared slab; pass 2 237 units, two per CTA at 148 SMs (tests/test_gram_plan.py)
                                           (20_000, 700, 0.0, 48),
                                           (20_000, 700, 0.002, 48)])
def test_product_bit_equal(gpu, n, l, miss, cols):
    pop, _ = make_population(n, l, seed=100 + n, missing_rate=miss)
    if l == 5001:      # the premise: more code-3 cells than the index takes (kgl_b200_upload_genotypes: max(2^16, N L / 64))
        assert (pop.codes() == 3).sum() > max(1 << 16, n * l // 64)
    check_product(gpu, with_monomorphic(pop), cols, n)


def test_product_multi_allelic_and_keep(gpu):
    pop, _ = make_population(300, 2500, seed=9, missing_rate=0.004)
    pop = add_multi_allelic(with_monomorphic(pop), 40, seed=9)
    keep = (np.random.default_rng(1).random(pop.n_loci) < 0.7).astype(np.uint8)
    check_product(gpu, pop, 17, 1, keep)
    check_product(gpu, pop, 48, 2)


def test_product_wide_population(gpu):
    """> 56 units of 64 genomes: the device rows are padded to a wider pitch."""
    pop, _ = make_population(3700, 300, seed=4, missing_rate=0.002)
    check_product(gpu, pop, 16, 3)


def test_product_several_slabs(gpu):
    """48 columns with code-3 cells: a pass-1 slab holds 174,592 loci, so 180,001 loci take two."""
    pop, _ = make_population(40, 180001, seed=6, missing_rate=0.01)
    check_product(gpu, pop, 48, 4)


def structured(n=500, l=6000, seed=31):
    """Five super-populations of unequal sizes, each drawing from its own AF column: Psi has four separated top eigenvalues."""
    offsets, af = make_loci(l, seed, "dense")
    frac = np.array([0.36, 0.26, 0.18, 0.12, 0.08])
    sp = np.repeat(np.arange(5), np.round(frac * n).astype(int))[:n].astype(np.uint8)
    codes = synth_codes(seed, af, sp, np.zeros(n), 0.002)
    from kgl_gene_b200.flatfile import FlatPopulation
    return FlatPopulation(offsets, af, sp, pack_codes(codes), n, False), codes


def test_pca_against_dense_eigh(gpu):
    """Both the operator (quantised to 2^-29 of each column's maximum, so perturbed by ~1e-8 of lambda_1) and the convergence
    factor (lambda_17 / lambda_4)^(2q) = 0.17^100 sit far below 1e-7 at q = 50, with relative gaps >= 10 % between the top five
    eigenvalues (asserted): eigenvalues to 1e-7 relative, 1 - |cos| to 1e-7. With the defaults (k = 10, q = 10, b = 16) the top
    four converge as 0.17^20 ~ 4e-16 and the bulk eigenvalues 5..10 not at all, so only the top four are checked, to 1e-5."""
    pop, codes = structured()
    w, u = np.linalg.eigh(P.psi(codes))
    w, u = w[::-1], u[:, ::-1]
    assert np.all(w[1:5] / w[:4] <= 0.9)
    gpu.upload_population(pop)
    r = gpu.pca(k=4, iterations=50, seed=3)
    assert r["n_loci_used"] == int(P.locus_stats(codes)[2].sum())
    assert np.all(np.abs(r["eigenvalues"] - w[:4]) <= 1e-7 * w[:4])
    cos = np.abs(np.sum(r["scores"] * u[:, :4], axis=0))
    assert np.all(1.0 - cos <= 1e-7)
    sc = r["scores"]
    top = np.argmax(np.abs(sc), axis=0)
    assert np.all(sc[top, np.arange(4)] > 0)                       # sign convention
    assert np.allclose(sc.T @ sc, np.eye(4), atol=1e-12)
    d = gpu.pca()
    assert d["eigenvalues"].shape == (10,) and d["scores"].shape == (500, 10)
    assert np.all(np.abs(d["eigenvalues"][:4] - w[:4]) <= 1e-5 * w[:4])


def test_start_block_is_the_oracles(gpu):
    """run_pca's start block (pca_start_entry) is pca_oracle.start_block: with q = 1 the Ritz values of span(Psi orth(Omega))
    depend on the start block (another seed moves them by >= 3e-4 relative here) and on the operator only through its
    quantisation (~1e-8), so they agree with a numpy Rayleigh-Ritz on the oracle's block to 1e-6. k = 10: b = 16."""
    pop, codes = structured(300, 3000, 5)
    psi = P.psi(codes)

    def ritz(seed):
        q = np.linalg.qr(psi @ np.linalg.qr(P.start_block(seed, 300, 16))[0])[0]
        return np.linalg.eigvalsh(q.T @ psi @ q)[::-1][:10]

    want = ritz(11)
    assert np.min(np.abs(ritz(12) - want) / want) > 1e-4
    gpu.upload_population(pop)
    got = gpu.pca(k=10, iterations=1, seed=11)["eigenvalues"]
    assert np.all(np.abs(got - want) <= 1e-6 * want)


def test_planted_superpopulations(gpu):
    pop, _ = make_population(2000, 50000, seed=12)
    gpu.upload_population(pop)
    sc = gpu.pca(k=4)["scores"]
    labels = pop.superpop.astype(int)
    centroids = np.stack([sc[labels == s].mean(axis=0) for s in range(5)])
    nearest = np.argmin(((sc[:, None, :] - centroids[None]) ** 2).sum(axis=2), axis=1)
    assert np.array_equal(nearest, labels)


def test_loadings(gpu):
    """u_i = Z v_i / sqrt(M lambda_i): unit norm and Z^T u_i = sqrt(M lambda_i) v_i up to the eigen-residual of v_i (q = 50:
    ~1e-8 of lambda_1 from the quantised operator), 0 at unused loci."""
    pop, codes = structured(300, 4000, 8)
    keep = (np.random.default_rng(2).random(pop.n_loci) < 0.8).astype(np.uint8)
    gpu.upload_population(pop)
    r = gpu.pca(k=4, iterations=50, keep=keep, loadings=True)
    lo, v, lam, m = r["loadings"], r["scores"], r["eigenvalues"], r["n_loci_used"]
    used = P.locus_stats(codes, keep)[2]
    assert not lo[~used].any()
    assert np.allclose(np.linalg.norm(lo, axis=0), 1.0, atol=1e-7)
    zt_u = P.z_matrix(codes, keep).T @ lo
    assert np.allclose(zt_u, np.sqrt(m * lam)[None, :] * v, atol=1e-6 * np.sqrt(m * lam[0]))


def test_deterministic(gpu):
    pop, _ = structured(300, 3000, 5)
    gpu.upload_population(pop)
    a = gpu.pca(k=6, seed=1, loadings=True)
    b = gpu.pca(k=6, seed=1, loadings=True)
    for key in ("eigenvalues", "scores", "loadings"):
        assert bit_equal(a[key], b[key]), key
    x = np.random.default_rng(0).standard_normal((300, 20))
    assert bit_equal(gpu.grm_product(x)[0], gpu.grm_product(x)[0])


def test_misuse(gpu):
    from kgl_gene_b200.capi import KglB200, KglError
    fresh = KglB200(0)
    fresh.n_genomes = 10
    with pytest.raises(KglError, match=r"run_pca failed \[2\]"):
        fresh.pca(k=2)
    with pytest.raises(KglError, match=r"run_grm_product failed \[2\]"):
        fresh.grm_product(np.zeros((10, 2)))
    fresh.close()
    pop, _ = make_population(30, 500, seed=2)
    gpu.upload_population(pop)
    for bad in (dict(k=41), dict(k=30), dict(k=5, keep=np.isin(np.arange(500), [1, 2, 3]).astype(np.uint8)),
                dict(k=2, keep=np.zeros(500, dtype=np.uint8))):
        with pytest.raises(KglError, match=r"run_pca failed \[1\]"):
            gpu.pca(**bad)
    for cols in (0, 49):
        with pytest.raises(KglError, match=r"run_grm_product failed \[1\]"):
            gpu.grm_product(np.zeros((30, cols)))
    with pytest.raises(KglError, match=r"run_grm_product failed \[1\]"):
        gpu.grm_product(np.ones((30, 1)), keep=np.zeros(500, dtype=np.uint8))


def test_misuse_too_many_loci(gpu):
    """n_loci >= 2^28 would overflow the int32 digit accumulators: refused before any work (device-generated matrix)."""
    from kgl_gene_b200.capi import KglB200, KglError
    ctx = KglB200(0)
    l = 1 << 28
    ctx.upload_loci(np.zeros((1, l), dtype=np.float32))
    ctx.set_genome_superpop(np.zeros(4, dtype=np.uint8))
    ctx.synth_genotypes(1, 4, l, np.zeros(4), missing_rate=0.0)
    with pytest.raises(KglError, match=r"run_pca failed \[1\]"):
        ctx.pca(k=2)
    with pytest.raises(KglError, match=r"run_grm_product failed \[1\]"):
        ctx.grm_product(np.ones((4, 1)))
    ctx.close()


def test_no_interference(gpu):
    pop, _ = make_population(300, 3000, seed=21, missing_rate=0.003)
    gpu.upload_population(pop)
    gpu.select_loci(spacing=0)
    gpu.count_and_inbreed()
    before = (gpu.ibs(), gpu.king(), gpu.gram(), gpu.grm(0), gpu.fetch_locus_counts())
    gpu.pca(k=3, loadings=True)
    gpu.grm_product(np.ones((300, 5)))
    assert np.array_equal(gpu.fetch_locus_counts(), before[4])          # PCA counts into a buffer of its own
    after = (gpu.ibs(), gpu.king(), gpu.gram(), gpu.grm(0))
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[2], after[2])
    assert bit_equal(np.nan_to_num(before[1], nan=7.0), np.nan_to_num(after[1], nan=7.0)) and bit_equal(before[3], after[3])
