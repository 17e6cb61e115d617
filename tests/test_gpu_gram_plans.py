"""The tensor-core Gram kernel (k_gram_i8, kgl_gene_b200/csrc/gram_i8.cuh) at the launch plans its callers reach.

k_gram_i8 runs units of (256 x 256 tile, chunk of K) round-robin over its CTAs. Its hard paths run only on some plans: a CTA
that runs several units carries the phases of its 3-deep stage ring and of its single TMEM accumulator set from one unit to
the next; units of one CTA can differ in length (the short last chunk); a split-K run adds its chunks with red.add into an
output the caller cleared, a one-chunk run stores; and the output is written as compact blocks (IBS, KING), into the pitched
ld x ld matrix (run_gram) or as a rectangular product (PCA). Each case here sizes its loci or its tile list with the planner
(tests/gram_plan_probe.cu) on this device's SM count, asserts the plan it names, prints it, and compares bit for bit:
  * a split whose last chunk is 1 stage, and one whose last chunk is 2 stages (shorter than the stage ring): run_gram, the IBS
    tile list on the tensor cores (tiles below the diagonal included), KING with its dense part on the popcount kernel (the
    HH Gram run and the M = H C^T run) and on the tensor cores, against float64 products of indicator matrices and the
    popcount oracle;
  * exactly SMs + 1 units in one chunk (enqueue_gram_tiles), so one CTA runs two units and stores both;
  * run_gram with three or more multi-stage units per CTA, split-K, chunks of unequal length, on saturated content;
  * KING over a band of rows, king(row_begin, row_end), whose tiles below the diagonal read mirrored blocks: two units per
    CTA, split-K, chunks of unequal length, both of KING's Gram runs, on saturated content.
Saturated content: genome g's code at locus l is (g + floor(l / 128)) mod m, so every 128-locus k-stage holds one code per
genome and the results follow from the number of loci per residue of the stage index. A stage that is lost, duplicated or
read from the wrong chunk changes the result. With m = 4 the code-3 cells are too many to index, so IBS takes the popcount
kernel and KING runs both HH and M on the tensor cores.
PCA pass 1 split-K and pass 2 with several units per CTA are rows of tests/test_gpu_pca.py::test_product_bit_equal, KING's M
run split in two is a row of tests/test_gpu_king.py::test_king_modes_and_edges; tests/test_gram_plan.py pins all these plans
at 148 SMs."""
import numpy as np
import pytest

import gram_plan_probe as GP
import king_oracle as K
import oracle_py as O

pytestmark = pytest.mark.gpu

SEED = 20261021


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.set_ibs_tensor_cores(True)
    ctx.close()


def first_plan(requests, ok):
    """The plan of the first request the predicate accepts (the probe evaluates them all in one call)."""
    _, cols = GP.plans(requests)
    for i in range(cols["n_tiles"].size):
        p = {f: int(v[i]) for f, v in cols.items()}
        if ok(p):
            return p
    raise AssertionError("no request reaches the plan")


def show(name, p):
    print(GP.describe(name, p))


def bit_equal(x, y):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    nx, ny = np.isnan(x), np.isnan(y)
    return x.shape == y.shape and np.array_equal(nx, ny) and np.array_equal(x[~nx].view(np.uint64), y[~ny].view(np.uint64))


def gram_ref(codes, rows=slice(None), cols=slice(None), weights=None, chunk=1 << 16):
    """sum_l w_l g_il g_jl for genomes i in rows, j in cols; codes uint8 [L][N], g the dosage (code 3 -> 0): int64, exact
    float64 products (every partial sum < 2^53)."""
    w = np.ones(codes.shape[0]) if weights is None else np.asarray(weights, dtype=np.float64)
    acc = 0.0
    for l0 in range(0, codes.shape[0], chunk):
        g = codes[l0:l0 + chunk].astype(np.float64)
        g[g == 3] = 0.0
        acc = acc + (g[:, rows] * w[l0:l0 + chunk, None]).T @ g[:, cols]
    return np.asarray(acc).astype(np.int64)


def device_population(gpu, n, n_loci, missing_rate):
    """Generated on the device, downloaded: the references' input."""
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    offsets, af = make_loci(n_loci, SEED)
    superpop, f = make_genomes(n, SEED)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.set_unphased(False)
    gpu.synth_genotypes(SEED, n, n_loci, f, missing_rate=missing_rate)
    return FlatPopulation(offsets, af, superpop, gpu.download_genotypes(), n, False)


def saturated(gpu, n, n_loci, m):
    """Uploads the saturated population (g + floor(l / 128)) mod m. Returns (pop, patterns uint8 [m][N], loci per pattern):
    every locus of a stage s carries pattern s mod m."""
    from kgl_gene_b200.flatfile import FlatPopulation, pack_codes
    from kgl_gene_b200.synth import make_genomes
    patterns = ((np.arange(n)[None, :] + np.arange(m)[:, None]) % m).astype(np.uint8)
    which = (np.arange(n_loci) // 128) % m
    offsets = (1000 + 10 * np.arange(n_loci)).astype(np.uint32)
    af = np.full((6, n_loci), 0.25, dtype=np.float32)
    superpop, _ = make_genomes(n, SEED)
    pop = FlatPopulation(offsets, af, superpop, pack_codes(patterns)[which], n, False)
    gpu.upload_population(pop)
    return pop, patterns, np.bincount(which, minlength=m)


# ---- a last chunk of 1 or 2 stages ------------------------------------------------------------------------------------------
SHORT_GENOMES = 130          # one 256 x 256 block, rows in both M = 128 halves of the tile


@pytest.mark.parametrize("last", [1, 2])
def test_last_chunk_shorter_than_the_ring(gpu, sms, last):
    """One tile / one block, split-K, the last chunk `last` stages (a partial last stage of 77 loci): run_gram, the IBS tile
    list on the tensor cores and KING both ways. The loci are the fewest that reach this split on this device."""
    p = first_plan([(1, k, sms) for k in range(128, 20_000)], lambda p: p["n_chunks"] > 1 and p["last_stages"] == last)
    n_loci = (p["k_stages"] - 1) * 128 + 77
    show(f"last chunk {last} ({SHORT_GENOMES} x {n_loci})", p)
    assert p["stages_per_chunk"] >= 64 and p["last_stages"] < 3
    pop = device_population(gpu, SHORT_GENOMES, n_loci, 0.002)
    codes = pop.codes()
    assert 0 < (codes == 3).sum() < (SHORT_GENOMES * n_loci) // 64      # indexed code-3 cells: the tensor-core IBS form, and an M run

    assert np.array_equal(gpu.gram(), gram_ref(codes))

    want_ibs = O.ibs(pop)
    coords = np.array([(0, 0), (1, 0), (2, 1), (0, 2), (2, 2)], dtype=np.uint32)
    got = gpu.ibs_tile_list(coords)
    assert gpu.ibs_used_tensor_cores()
    padded = np.zeros((192, 192, 4), dtype=np.uint32)
    padded[:SHORT_GENOMES, :SHORT_GENOMES] = want_ibs
    for t, (ti, tj) in enumerate(coords):
        assert np.array_equal(got[t], padded[64 * ti:64 * ti + 64, 64 * tj:64 * tj + 64]), (ti, tj)

    want = K.king_codes(codes)["kinship"]
    for tensor in (False, True):
        gpu.set_ibs_tensor_cores(tensor)
        assert bit_equal(gpu.king(), want), f"tensor={tensor}"
        assert gpu.ibs_used_tensor_cores() == tensor
    gpu.set_ibs_tensor_cores(True)


# ---- SMs + 1 units, one chunk -----------------------------------------------------------------------------------------------
def test_one_more_unit_than_sms(gpu, sms):
    """enqueue_gram_tiles(first, stride) over the fewest 256-genome blocks that give exactly SMs + 1 tiles: one chunk (3,000
    loci), CTA 0 runs two units and stores both; the other tiles of the matrix stay zero."""
    pick = None
    for nb in range(1, 200):
        total = nb * (nb + 1) // 2
        for stride in range(1, 16):
            for first in range(stride):
                if len(range(first, total, stride)) == sms + 1:
                    pick = (nb, first, stride)
                    break
            if pick: break
        if pick: break
    nb, first, stride = pick
    n, n_loci = nb * 256 - 19, 3_000
    p = GP.plan(sms + 1, GP.k_stages(n_loci), sms)
    show(f"SMs + 1 units ({n} x {n_loci}, tiles {first}::{stride} of {nb * (nb + 1) // 2})", p)
    assert p["n_chunks"] == 1 and p["units"] == sms + 1 and p["grid"] == sms and p["max_units_per_cta"] == 2
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(n, n_loci, seed=SEED, missing_rate=0.001)
    gpu.upload_population(pop)
    gpu.enqueue_gram_tiles(first, stride)
    got = gpu.fetch_gram()
    g = pop.codes().astype(np.float64)
    g[g == 3] = 0.0
    tiles = [(ti, tj) for ti in range(nb) for tj in range(ti, nb)][first::stride]
    assert len(tiles) == sms + 1
    for ti, tj in tiles:
        r, c = slice(256 * ti, min(n, 256 * ti + 256)), slice(256 * tj, min(n, 256 * tj + 256))
        want = (g[:, r].T @ g[:, c]).astype(np.int64)
        assert np.array_equal(got[r, c], want), (ti, tj)
        assert np.array_equal(got[c, r], want.T), (ti, tj)
        got[r, c] = 0
        got[c, r] = 0
    assert not got.any()


# ---- run_gram: >= 3 multi-stage units per CTA, saturated ------------------------------------------------------------------
GRAM_SAT_GENOMES = 4_315     # 17 x 17 blocks, the last one partial: 153 tiles


def test_gram_several_units_per_cta_saturated(gpu, sms):
    """run_gram into the pitched ld x ld matrix with at least three multi-stage units per CTA, split-K, a last chunk shorter
    than the others; saturated content with m = 3 (40,000 loci on a B200)."""
    tiles = GP.upper_tiles(GRAM_SAT_GENOMES)
    p = first_plan([(tiles, GP.k_stages(l), sms) for l in range(40_000, 400_000, 1_000)],
                   lambda p: p["n_chunks"] > 1 and p["max_units_per_cta"] >= 3 and p["last_stages"] < p["stages_per_chunk"])
    n_loci = p["k_stages"] * 128 - 51
    show(f"run_gram saturated ({GRAM_SAT_GENOMES} x {n_loci})", p)
    _, patterns, per = saturated(gpu, GRAM_SAT_GENOMES, n_loci, 3)
    want = gram_ref(patterns, weights=per)
    assert np.array_equal(gpu.gram(), want)


# ---- KING over a band with mirrored blocks, saturated ----------------------------------------------------------------------
KING_BAND_LOCI = 30_000


def test_king_band_mirrored_blocks_saturated(gpu, sms):
    """king(row_begin, row_end) over 100 rows of a middle block row: the band's tiles touch every block of that row, those
    left of the diagonal mirrored. The fewest blocks per side that give two units per CTA with split-K at 30,000 loci;
    saturated content with m = 4 (the popcount kernel for IBS, HH and M on the tensor cores)."""
    ks = GP.k_stages(KING_BAND_LOCI)
    p = first_plan([(nb, ks, sms) for nb in range(2, 400)],
                   lambda p: p["n_chunks"] > 1 and p["max_units_per_cta"] >= 2 and p["last_stages"] < p["stages_per_chunk"])
    nb = p["n_tiles"]
    n = nb * 256 - 40
    r0 = 256 * (nb // 2) + 70
    r1 = r0 + 100                                      # two 64-genome tile rows of block row nb // 2
    show(f"KING band saturated ({n} x {KING_BAND_LOCI}, rows {r0}:{r1}, {nb} blocks, {nb // 2} mirrored)", p)
    _, patterns, per = saturated(gpu, n, KING_BAND_LOCI, 4)
    got = gpu.king(r0, r1)
    assert not gpu.ibs_used_tensor_cores()
    want = K.king_codes(patterns, weights=per, rows=slice(r0, r1))["kinship"]
    assert np.isfinite(want).any()
    assert bit_equal(got, want)
