"""KING-robust kinship on the device (kgl_b200_run_king / kgl_b200_run_king_pairs) against the oracle's matrix-product
restatement: counts equal, kinship bit-equal, in every missing-cell mode of the IBS path and with its dense part on the tensor
cores and on the popcount kernel."""
import ctypes as C
import os

import numpy as np
import pytest

import king_oracle as K
import oracle_py as O
from kgl_gene_b200.kinship import SECOND, THIRD, king_degree

pytestmark = pytest.mark.gpu

COUNTS = ("n_valid", "ibs0", "ibs1", "het_het", "het_a", "het_b")


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.set_ibs_tensor_cores(True)
    ctx.close()


def bit_equal(x, y):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    nx, ny = np.isnan(x), np.isnan(y)
    return x.shape == y.shape and np.array_equal(nx, ny) and np.array_equal(x[~nx].view(np.uint64), y[~ny].view(np.uint64))


def oracle_pairs(want, min_kinship, coords=None):
    """The oracle's pair list: every a < b with kinship >= min_kinship (inside the tiles `coords`), sorted by (a, b)."""
    from kgl_gene_b200.capi import KING_PAIR_DTYPE
    n = want["kinship"].shape[0]
    a, b = np.triu_indices(n, 1)
    if coords is not None:
        tiles = {(int(i), int(j)) for i, j in np.asarray(coords).reshape(-1, 2)}
        keep = np.array([(x // 64, y // 64) in tiles for x, y in zip(a, b)], dtype=bool)
        a, b = a[keep], b[keep]
    with np.errstate(invalid="ignore"):
        sel = want["kinship"][a, b] >= min_kinship
    a, b = a[sel], b[sel]
    out = np.zeros(a.shape[0], dtype=KING_PAIR_DTYPE)
    out["a"], out["b"] = a, b
    for k in COUNTS:
        out[k] = want[k][a, b]
    out["kinship"] = want["kinship"][a, b]
    return out


def same_pairs(got, want):
    return got.shape == want.shape and all(np.array_equal(got[k], want[k]) for k in ("a", "b") + COUNTS) and bit_equal(got["kinship"], want["kinship"])


def check_dense(gpu, pop, want, band):
    for tensor in (True, False):
        gpu.set_ibs_tensor_cores(tensor)
        got = gpu.king()
        assert bit_equal(got, want["kinship"]), f"tensor={tensor}"
        assert bit_equal(gpu.king(*band), want["kinship"][band[0]:band[1]]), f"tensor={tensor} band={band}"
    gpu.set_ibs_tensor_cores(True)


@pytest.mark.parametrize("n,l,miss", [(70, 999, 0.0),        # no code-3 cell
                                      (300, 20000, 0.03),    # too many code-3 cells to index: in-kernel validity plane
                                      (64, 64, 0.5),         # exactly one tile, half the cells dropped
                                      (1, 40, 0.1),          # a single genome
                                      (129, 33000, 0.002),   # several word chunks per tile
                                      (600, 20000, 0.002)])  # 6 blocks x 157 stages: the HH and M Gram runs split in two chunks
def test_king_modes_and_edges(gpu, n, l, miss):
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(n, l, seed=3 + n, missing_rate=miss)
    gpu.upload_population(pop)
    want = K.king(pop)
    check_dense(gpu, pop, want, (n // 3, max(n // 3 + 1, 2 * n // 3)))


def test_king_wide_population(gpu):
    """3,000 genomes: the tile list spans several blocks per side, band rows 2100:2400 read mirrored blocks below the diagonal
    (where the stored M value belongs to the partner)."""
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(3000, 400, seed=29, missing_rate=0.004)
    gpu.upload_population(pop)
    want = K.king(pop)
    got = gpu.king()
    assert gpu.ibs_used_tensor_cores()
    assert bit_equal(got, want["kinship"])
    assert bit_equal(gpu.king(2100, 2400), want["kinship"][2100:2400])


@pytest.mark.parametrize("multi", [False, True])
def test_king_pair_lists(gpu, multi):
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    pop, _ = make_population(700, 2500, seed=41, missing_rate=0.01)
    if multi:
        add_multi_allelic(pop, 200, seed=42)
    gpu.upload_population(pop)
    want = K.king(pop)
    for tensor in (True, False):
        gpu.set_ibs_tensor_cores(tensor)
        for t in (-np.inf, 0.0, 0.0442):
            assert same_pairs(gpu.king_pairs(t), oracle_pairs(want, t)), (tensor, t)
    gpu.set_ibs_tensor_cores(True)


def test_king_pairs_dealt_to_ranks(gpu):
    """Three ranks' shards.block_tile_coords lists give the whole list; each rank's list is the oracle's pairs of its tiles."""
    from kgl_gene_b200.shards import block_tile_coords
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(700, 2500, seed=23, missing_rate=0.01)
    gpu.upload_population(pop)
    want = K.king(pop)
    parts = []
    for r in range(3):
        coords = block_tile_coords(pop.n_genomes, r, 3)
        mine = gpu.king_pairs(-np.inf, coords)
        assert same_pairs(mine, oracle_pairs(want, -np.inf, coords))
        parts.append(mine)
    joined = np.concatenate(parts)
    joined = joined[np.lexsort((joined["b"], joined["a"]))]
    assert same_pairs(joined, oracle_pairs(want, -np.inf))


def test_king_pairs_capacity(gpu):
    from kgl_gene_b200.capi import KGL_B200_ERR_NOMEM, KING_PAIR_DTYPE
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(150, 3000, seed=43, missing_rate=0.01)
    gpu.upload_population(pop)
    want = oracle_pairs(K.king(pop), 0.0)
    assert want.shape[0] > 10
    out = np.zeros(10, dtype=KING_PAIR_DTYPE)
    n = C.c_uint64(0)
    rc = gpu.lib.kgl_b200_run_king_pairs(gpu.h, C.c_uint64(0), None, C.c_double(0.0), C.c_uint64(10), C.c_void_p(out.ctypes.data), C.byref(n))
    assert rc == KGL_B200_ERR_NOMEM and n.value == want.shape[0]
    assert same_pairs(gpu.king_pairs(0.0, capacity=10), want)                  # the binding's retry with the exact capacity
    assert same_pairs(gpu.king_pairs(0.0, capacity=want.shape[0]), want)


def _transmit(parent, rng):
    """One allele of each locus from an unphased genotype: 0 -> 0, 2 -> 1, 1 -> 0 or 1 at random."""
    return np.where(parent == 1, rng.integers(0, 2, parent.shape), parent // 2)


def test_king_planted_relatives(gpu):
    """One super-population, F = 0, 0.5 % missing cells; duplicates, parent-offspring, full and half siblings planted by Mendelian
    transmission. Every planted pair is found at 0.0442 with its degree; no unplanted pair reaches 2^-3.5."""
    from kgl_gene_b200.flatfile import FlatPopulation, pack_codes
    from kgl_gene_b200.synth import make_loci, synth_codes
    rng = np.random.default_rng(44)
    n_found, l = 200, 20000
    offsets, af = make_loci(l, 44)
    founders = synth_codes(44, af, np.zeros(n_found + 6, np.uint8), np.zeros(n_found + 6), missing_rate=0.0).T.astype(np.int64)
    outside = founders[n_found:]                   # parents that are not part of the population
    genomes = list(founders[:n_found])
    planted = {}                                   # (a, b) -> (degree, kind)

    def add(g):
        genomes.append(g)
        return len(genomes) - 1

    def child(p, q):
        return _transmit(p, rng) + _transmit(q, rng)

    f = iter(range(n_found))
    for _ in range(3):                             # duplicates
        a = next(f)
        planted[(a, add(genomes[a].copy()))] = (0, "duplicate")
    for _ in range(3):                             # parent-offspring trios
        p, q = next(f), next(f)
        c = add(child(genomes[p], genomes[q]))
        planted[(p, c)] = planted[(q, c)] = (1, "parent-offspring")
    for _ in range(3):                             # full siblings and their parents
        p, q = next(f), next(f)
        s1, s2 = add(child(genomes[p], genomes[q])), add(child(genomes[p], genomes[q]))
        planted[(s1, s2)] = (1, "full siblings")
        for par in (p, q):
            planted[(par, s1)] = planted[(par, s2)] = (1, "parent-offspring")
    for i in range(3):                             # half siblings: one shared parent, the others from outside the population
        p = next(f)
        h1, h2 = add(child(genomes[p], outside[2 * i])), add(child(genomes[p], outside[2 * i + 1]))
        planted[(h1, h2)] = (2, "half siblings")
        planted[(p, h1)] = planted[(p, h2)] = (1, "parent-offspring")
    codes = np.stack(genomes).T.astype(np.uint8)   # [L][N]
    codes[rng.random(codes.shape) < 0.005] = 3
    n = codes.shape[1]
    pop = FlatPopulation(offsets, af, np.zeros(n, np.uint8), pack_codes(codes), n, False)
    gpu.upload_population(pop)
    pairs = gpu.king_pairs(THIRD)
    assert same_pairs(pairs, oracle_pairs(K.king(pop), THIRD))
    found = {(int(a), int(b)): (float(k), int(i0)) for a, b, k, i0 in zip(pairs["a"], pairs["b"], pairs["kinship"], pairs["ibs0"])}
    for (a, b), (deg, kind) in planted.items():
        assert (a, b) in found, (a, b, kind)
        k, ibs0 = found[(a, b)]
        assert king_degree(k) == deg, (a, b, k, kind)
        if kind == "duplicate":
            assert k == 0.5
        if kind == "parent-offspring":
            assert ibs0 == 0                       # no opposite homozygotes
    for (a, b), (k, ibs0) in found.items():
        if (a, b) not in planted:
            assert k < SECOND, (a, b, k)


def test_king_random_shapes(gpu):
    """Seeded random shapes; KGL_KING_RANDOM_CASES sets the campaign size."""
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    rng = np.random.default_rng(int(os.environ.get("KGL_KING_RANDOM_SEED", "45")))
    for case in range(int(os.environ.get("KGL_KING_RANDOM_CASES", "4"))):
        n, l = int(rng.integers(1, 420)), int(rng.integers(1, 6000))
        miss = float(rng.choice([0.0, 0.001, 0.02, 0.2]))
        pop, _ = make_population(n, l, seed=1000 + case, missing_rate=miss, spectrum=str(rng.choice(["sfs", "dense"])))
        if rng.random() < 0.3 and l > 10:
            add_multi_allelic(pop, int(rng.integers(1, l // 4 + 2)), seed=2000 + case)
        gpu.upload_population(pop)
        want = K.king(pop)
        tensor = bool(rng.random() < 0.5)
        gpu.set_ibs_tensor_cores(tensor)
        info = (case, n, l, miss, tensor)
        assert bit_equal(gpu.king(), want["kinship"]), info
        r0 = int(rng.integers(0, n)); r1 = int(rng.integers(r0 + 1, n + 1))
        assert bit_equal(gpu.king(r0, r1), want["kinship"][r0:r1]), info + (r0, r1)
        t = float(rng.choice([-np.inf, 0.0, THIRD, rng.uniform(-0.5, 0.5)]))
        assert same_pairs(gpu.king_pairs(t), oracle_pairs(want, t)), info + (t,)
    gpu.set_ibs_tensor_cores(True)


def test_king_misuse():
    from kgl_gene_b200.capi import KING_PAIR_DTYPE, KglB200
    from kgl_gene_b200.synth import make_population
    ERR_INVALID, ERR_STATE = 1, 2
    ctx = KglB200(0)
    try:
        lib, h = ctx.lib, ctx.h
        out = np.zeros(64 * 64, dtype=np.float64)
        pairs = np.zeros(16, dtype=KING_PAIR_DTYPE)
        n = C.c_uint64(0)
        pp, op = C.c_void_p(pairs.ctypes.data), C.c_void_p(out.ctypes.data)
        # before a genotype upload
        assert lib.kgl_b200_run_king(h, C.c_uint64(0), C.c_uint64(1), op) == ERR_STATE
        assert lib.kgl_b200_run_king_pairs(h, C.c_uint64(0), None, C.c_double(0.0), C.c_uint64(16), pp, C.byref(n)) == ERR_STATE
        pop, _ = make_population(100, 500, seed=46, missing_rate=0.01)
        ctx.upload_population(pop)
        # null outputs, bad bands
        assert lib.kgl_b200_run_king(h, C.c_uint64(0), C.c_uint64(1), None) == ERR_INVALID
        assert lib.kgl_b200_run_king(h, C.c_uint64(5), C.c_uint64(5), op) == ERR_INVALID
        assert lib.kgl_b200_run_king(h, C.c_uint64(0), C.c_uint64(101), op) == ERR_INVALID
        assert lib.kgl_b200_run_king_pairs(h, C.c_uint64(0), None, C.c_double(0.0), C.c_uint64(16), None, C.byref(n)) == ERR_INVALID
        assert lib.kgl_b200_run_king_pairs(h, C.c_uint64(0), None, C.c_double(0.0), C.c_uint64(16), pp, None) == ERR_INVALID
        # tiles outside the grid (2 x 2 tiles) or below the diagonal
        for bad in ([[0, 2]], [[2, 2]], [[1, 0]], [[0, 0], [1, 0]]):
            c = np.ascontiguousarray(bad, dtype=np.uint32)
            assert lib.kgl_b200_run_king_pairs(h, C.c_uint64(c.shape[0]), C.c_void_p(c.ctypes.data), C.c_double(0.0), C.c_uint64(16), pp,
                                               C.byref(n)) == ERR_INVALID, bad
        # the context still computes afterwards
        assert bit_equal(ctx.king(), K.king(pop)["kinship"])
    finally:
        ctx.close()


@pytest.mark.parametrize("tensor", [True, False])
def test_king_leaves_ibs_and_gram_alone(gpu, tensor):
    from kgl_gene_b200.shards import block_tile_coords
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(600, 3000, seed=47, missing_rate=0.01)
    gpu.upload_population(pop)
    gpu.set_ibs_tensor_cores(tensor)
    coords = block_tile_coords(pop.n_genomes, 1, 3)
    before = (gpu.ibs(), gpu.ibs(100, 300), gpu.ibs_tile_list(coords), gpu.gram())
    gpu.king(); gpu.king(100, 300); gpu.king_pairs(0.0, coords); gpu.king_pairs(0.0)
    after = (gpu.ibs(), gpu.ibs(100, 300), gpu.ibs_tile_list(coords), gpu.gram())
    for x, y in zip(before, after):
        assert np.array_equal(x, y)
    assert np.array_equal(after[0], O.ibs(pop))
    gpu.set_ibs_tensor_cores(True)


def test_king_full_width_properties(gpu):
    """chr22-shaped width on device-generated data: symmetric, diagonal 0.5, band rows equal to whole-matrix rows."""
    from kgl_gene_b200.synth import make_genomes, make_loci
    n, l = 2504, 40_000
    offsets, af = make_loci(l, 78)
    superpop, f = make_genomes(n, 78)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.synth_genotypes(78, n, l, f, missing_rate=0.001)
    full = gpu.king()
    assert bit_equal(full, full.T)
    assert np.all(np.diag(full) == 0.5)
    assert bit_equal(gpu.king(1000, 1100), full[1000:1100])
    assert np.all(full[~np.eye(n, dtype=bool)] < 0.5)
