"""CPU checks of the genotype PCA restatement (tests/pca_oracle.py) and of the C ABI's options struct."""
import ctypes as C

import numpy as np
import pytest

import pca_oracle as P
from kgl_gene_b200.synth import make_population


def _codes(n, l, seed, missing):
    pop, _ = make_population(n, l, seed=seed, missing_rate=missing)
    codes = pop.codes()
    codes[: l // 20] = np.where(codes[: l // 20] == 3, 3, 0)            # monomorphic loci (p = 0) drop out
    return codes


@pytest.mark.parametrize("n,l,missing,cols", [(50, 700, 0.0, 3), (120, 2000, 0.03, 17), (9, 300, 0.2, 1)])
def test_oracle_product_within_quantisation_bound(n, l, missing, cols):
    """|y - Z^T Z x| <= 2^-28 (|Z|^T |Z| 1 max|x_j| + (sum_l G_lg) max|W_j| + (loci valid for g) max|V_j|) + rounding: the block is
    quantised to 2^-s_j <= 2^-28 max|x_j| (rint, or the clamp at 2^29 - 1), W and V to 2^-28 of their column maxima; the double
    operations after the exact contractions add a relative 2^-50 of the magnitudes they combine."""
    codes = _codes(n, l, 11 + n, missing)
    rng = np.random.default_rng(n)
    x = rng.standard_normal((n, cols))
    keep = (rng.random(l) < 0.9).astype(np.uint8)
    y, m = P.grm_product(codes, x, keep)
    z = P.z_matrix(codes, keep)
    want = z.T @ (z @ x)
    p, d, used = P.locus_stats(codes, keep)
    w = d[:, None] * (z @ x)
    v = (2.0 * p)[:, None] * w
    G = np.where(codes == 3, 0, codes).astype(np.float64) * used[:, None]
    valid = ((codes != 3) & used[:, None]).astype(np.float64)
    az = np.abs(z)
    bound = 2.0**-28 * (az.T @ (az @ np.ones(n)))[:, None] * np.abs(x).max(axis=0)[None, :]
    bound += 2.0**-28 * G.sum(axis=0)[:, None] * np.abs(w).max(axis=0)[None, :]
    bound += 2.0**-28 * valid.sum(axis=0)[:, None] * np.abs(v).max(axis=0)[None, :]
    bound += 2.0**-50 * (az.T @ (az @ np.abs(x)) + G.T @ np.abs(w) + valid.T @ np.abs(v))
    assert m == int(used.sum()) > 0
    assert np.all(np.abs(y - want) <= bound)


def test_digit_round_trip_and_quantisation():
    rng = np.random.default_rng(5)
    F = np.concatenate([rng.standard_normal((200, 3)) * [1e-12, 1.0, 3e7], np.zeros((200, 1))], axis=1)
    F[7, 1] = np.nextafter(1.0, 0.0) * 2.0**np.frexp(np.abs(F[:, 1]).max())[1]    # rounds to 2^29: clamped to 2^29 - 1
    s = P.shifts(F)
    scaled = np.abs(np.ldexp(F, s[None, :].astype(np.int32))).max(axis=0)
    assert np.all((scaled[:3] >= 2.0**28) & (scaled[:3] < 2.0**29)) and s[3] == 0
    q = P.quantise(F, s)
    assert q.min() >= -(2**29) and q.max() <= 2**29 - 1 and q[7, 1] == 2**29 - 1
    fq = q + P.OFFSET
    dg = P.digits(fq)
    assert dg.shape == (15,) + F.shape and dg.max() <= 3
    assert np.array_equal(sum(dg[d].astype(np.int64) << (2 * d) for d in range(15)), fq)
    assert np.array_equal(P.digits(np.array([0, 2**30 - 1]))[:, 1], np.full(15, 3)) and not P.digits(np.array([0])).any()


def test_start_block_is_a_pure_gaussian_function_of_seed_genome_column():
    a = P.start_block(7, 3000, 32)
    assert np.array_equal(P.start_block(7, 40, 16), a[:40, :16])            # independent of the population size and block width
    assert not np.array_equal(P.start_block(8, 40, 16), a[:40, :16])
    assert abs(a.mean()) < 0.01 and abs(a.std() - 1.0) < 0.01
    assert abs(np.mean(a**4) - 3.0) < 0.1                                     # Gaussian kurtosis
    assert np.all(np.isfinite(a))


def test_options_struct_layout():
    from kgl_gene_b200 import capi
    assert C.sizeof(capi.PcaOptions) == 24
    assert [getattr(capi.PcaOptions, f).offset for f in ("keep", "n_components", "iterations", "seed")] == [0, 8, 12, 16]


def test_pca_binding_sizes_its_buffers_for_the_default_k():
    """k = 0 means the C ABI's default of 10 components: the binding passes 10 and allocates for 10 (a stand-in library
    records what it is handed)."""
    from kgl_gene_b200.capi import KglB200
    seen = {}

    class Lib:
        def kgl_b200_run_pca(self, h, opt, ev, sc, ld, m):
            seen["k"] = opt._obj.n_components
            return 0

    ctx = KglB200.__new__(KglB200)
    ctx.lib, ctx.h, ctx.n_genomes, ctx.n_loci = Lib(), None, 7, 5
    r = ctx.pca(k=0, loadings=True)
    assert seen["k"] == 10
    assert r["eigenvalues"].shape == (10,) and r["scores"].shape == (7, 10) and r["loadings"].shape == (5, 10)
    assert ctx.pca(k=3)["scores"].shape == (7, 3) and seen["k"] == 3
    with pytest.raises(ValueError):
        ctx.pca(k=-1)
