"""Pairwise IBS on the popcount kernel (k_ibs_tiles, kgl_gene_b200/csrc/ibs_tile.cuh), the sparse repair of indexed code-3 cells
(k_ibs_missing_fix) and the slab drivers of kgl_b200_api.cu at the launch plans they reach.

k_ibs_tiles runs units of (64 x 64 tile, chunk of words) round-robin over one persistent CTA per SM, through a six-slot stage
ring whose barrier phases carry from one unit to the next; a split plan adds its chunks atomically into a cleared accumulator, a
one-chunk plan stores. It is the only dense IBS / KING path for a population whose code-3 cells are too many to index (more than
1/64 of the cells: the validity plane), and it runs on pre-masked planes, followed by the repair, with the tensor cores off.
The repair cuts every genome's dropped rows into segments: with more than one, J (plane 2) is added atomically into a plane the
caller cleared (by a 2-D memset when the dense plan has one chunk), otherwise stored by the first counter pass and added by the
next, one pass per 32,760 rows. The C ABI runs at most 8,192 tiles per launch and cuts larger calls into launches and slabs.

Each case sizes its input with the planner (tests/ibs_plan_probe.cu) on this device's SM count, asserts the plan it names, prints
it, and runs twice on one context: both results must equal the reference, so a missing clear shows as stale counts. IBS is
compared cell for cell, KING bit for bit. tests/test_ibs_plan.py pins these plans at 148 SMs."""
import numpy as np
import pytest

import ibs_plan_probe as IP
import king_oracle as K
import oracle_py as O

pytestmark = pytest.mark.gpu

SEED = 20261022
FORMS = ("no code 3", "indexed", "validity plane")
MISSING = {"no code 3": 0.0, "indexed": 0.005, "validity plane": 0.05}


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
    _, cols = IP.plans(requests)
    for i in range(cols["n_tiles"].size):
        p = {f: int(v[i]) for f, v in cols.items()}
        if ok(p):
            return p
    raise AssertionError("no request reaches the plan")


def show(name, p):
    print(IP.describe(name, p))


def bit_equal(x, y):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    nx, ny = np.isnan(x), np.isnan(y)
    return x.shape == y.shape and np.array_equal(nx, ny) and np.array_equal(x[~nx].view(np.uint64), y[~ny].view(np.uint64))


def upload_codes(gpu, codes):
    """Uploads the code matrix uint8 [L][N]; returns the population."""
    from kgl_gene_b200.flatfile import FlatPopulation, pack_codes
    from kgl_gene_b200.synth import make_genomes
    n_loci, n = codes.shape
    offsets = (1000 + 10 * np.arange(n_loci)).astype(np.uint32)
    af = np.full((6, n_loci), 0.25, dtype=np.float32)
    superpop, _ = make_genomes(n, SEED)
    pop = FlatPopulation(offsets, af, superpop, pack_codes(codes), n, False)
    gpu.upload_population(pop)
    return pop


def random_codes(n, n_loci, form, seed):
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(n, n_loci, seed=seed, missing_rate=MISSING[form])
    return pop.codes()


def assert_form(codes, form):
    """The plane form the population takes: indexed iff 0 < code-3 cells <= max(2^16, N L / 64) (dropped_index_limit)."""
    n3 = int((codes == 3).sum())
    limit = max(1 << 16, codes.size // 64)
    assert {"no code 3": n3 == 0, "indexed": 0 < n3 <= limit, "validity plane": n3 > limit}[form], (form, n3, limit)


def ibs_ref(codes, rows=slice(None), weights=None):
    """uint32 [rows][N][4] = {IBS0, IBS1, IBS2, valid} from king_oracle's indicator products, IBS2 = n_valid - ibs0 - ibs1."""
    k = K.king_codes(codes, weights=weights, rows=rows)
    return np.stack([k["ibs0"], k["ibs1"], k["n_valid"] - k["ibs0"] - k["ibs1"], k["n_valid"]], axis=-1).astype(np.uint32)


def tiles_of(matrix, coords):
    """The 64 x 64 tiles `coords` of an [N][N][4] matrix, padding genomes 0: uint32 [len(coords)][64][64][4]."""
    n = matrix.shape[0]
    side = IP.side(n)
    padded = np.zeros((side * 64, side * 64, 4), dtype=np.uint32)
    padded[:n, :n] = matrix
    blocks = padded.reshape(side, 64, side, 64, 4)
    coords = np.asarray(coords)
    return blocks[coords[:, 0], :, coords[:, 1]]


def upper_coords(side):
    return np.array([(i, j) for i in range(side) for j in range(i, side)], dtype=np.uint32)


# ---- >= 3 multi-stage units per CTA, split, saturated -------------------------------------------------------------------------
SAT_GENOMES = 1_100
SAT_PATTERNS = 5
SAT_STAGE_LOCI = 512         # one 16-word stage


@pytest.mark.parametrize("form", FORMS)
def test_several_split_units_per_cta_saturated(gpu, sms, form):
    """ibs() of the whole matrix with at least three multi-stage units per CTA, split, stages per chunk not a multiple of the
    ring, an unequal last chunk and a partial last stage (1,100 x 25,000 on a B200: 3 chunks of 17 stages, the last 238 words, 4
    units per CTA). Genome g's code at locus l is P[(l // 512) mod 5][g], so every stage holds one pattern and the result is
    sum_r n_r ibs(P_r): a stage lost, duplicated or read from the wrong chunk changes it. Indexed: a few genomes coded 3 in one
    pattern; validity plane: code 3 dense."""
    tiles = IP.upper_tiles(SAT_GENOMES)
    p = first_plan([(tiles, l, sms, 0, SAT_GENOMES) for l in range(25_000, 400_000, 500)],
                   lambda p: p["n_chunks"] > 1 and p["max_units_per_cta"] >= 3 and p["stages_per_chunk"] % 6 != 0
                   and p["last_chunk_words"] < p["words_per_chunk"] and p["last_stage_words"] < 16)
    n_loci = p["n_loci"]
    show(f"saturated {SAT_GENOMES} x {n_loci}, {form}", p)
    rng = np.random.default_rng(SEED)
    patterns = rng.integers(0, 4 if form == "validity plane" else 3, size=(SAT_PATTERNS, SAT_GENOMES)).astype(np.uint8)
    if form == "indexed":
        patterns[2, [5, 64, 77, 700, 1_099]] = 3
    which = (np.arange(n_loci) // SAT_STAGE_LOCI) % SAT_PATTERNS
    codes = patterns[which]
    assert_form(codes, form)
    upload_codes(gpu, codes)
    want = ibs_ref(patterns, weights=np.bincount(which, minlength=SAT_PATTERNS))
    gpu.set_ibs_tensor_cores(False)
    for run in (1, 2):
        assert np.array_equal(gpu.ibs(), want), f"run {run}"
        assert not gpu.ibs_used_tensor_cores()


# ---- SMs + 1 units, one chunk ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("form", FORMS)
def test_one_more_unit_than_sms(gpu, sms, form):
    """ibs_tiles(0, 1, SMs + 1) with one chunk of several stages: CTA 0 runs two units and stores both."""
    side = next(s for s in range(1, 1000) if s * (s + 1) // 2 >= sms + 1)
    n, n_loci = side * 64 - 21, 3_000
    codes = random_codes(n, n_loci, form, SEED + 1)
    p = IP.plan(sms + 1, n_loci, sms, int((codes == 3).sum()), n)
    show(f"SMs + 1 units ({n} x {n_loci}, {form})", p)
    assert p["n_chunks"] == 1 and p["units"] == sms + 1 and p["grid"] == sms and p["max_units_per_cta"] == 2
    assert p["stages_per_chunk"] > 1 and p["segs"] == 1
    assert_form(codes, form)
    upload_codes(gpu, codes)
    want = tiles_of(ibs_ref(codes), upper_coords(side)[:sms + 1])
    gpu.set_ibs_tensor_cores(False)
    for run in (1, 2):
        assert np.array_equal(gpu.ibs_tiles(0, 1, sms + 1), want), f"run {run}"
        assert not gpu.ibs_used_tensor_cores()


# ---- a split whose last stage holds 2 words -------------------------------------------------------------------------------------
LAST2_GENOMES = 250


@pytest.mark.parametrize("form", FORMS)
def test_split_last_stage_of_two_words(gpu, sms, form):
    """ibs() of 250 genomes (10 tiles), split, words_used = 2 mod 16: the last stage of the last chunk holds 2 words."""
    tiles = IP.upper_tiles(LAST2_GENOMES)
    p = first_plan([(tiles, 32 * (16 * k + 2) - 5, sms, 0, LAST2_GENOMES) for k in range(16, 2_000)],
                   lambda p: p["n_chunks"] > 1 and p["last_stage_words"] == 2)
    n_loci = p["n_loci"]
    show(f"last stage 2 words ({LAST2_GENOMES} x {n_loci}, {form})", p)
    codes = random_codes(LAST2_GENOMES, n_loci, form, SEED + 2)
    assert_form(codes, form)
    upload_codes(gpu, codes)
    want = ibs_ref(codes)
    gpu.set_ibs_tensor_cores(False)
    for run in (1, 2):
        assert np.array_equal(gpu.ibs(), want), f"run {run}"
        assert not gpu.ibs_used_tensor_cores()


# ---- the repair at each of its plans --------------------------------------------------------------------------------------------
def heavy_codes(n, n_loci, heavy, seed):
    """Random codes 0..2 with code 3 only in the genomes of `heavy` ({genome: dropped rows}), at rows drawn without replacement."""
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, 3, size=(n_loci, n)).astype(np.uint8)
    for g, rows in heavy.items():
        codes[rng.choice(n_loci, size=rows, replace=False), g] = 3
    return codes


def listed_tiles(side, count, seed):
    """count tile coordinates cycling through every cell of the side x side grid (below the diagonal too), shuffled."""
    grid = np.array([(i, j) for i in range(side) for j in range(side)], dtype=np.uint32)
    coords = grid[np.arange(count) % len(grid)]
    return coords[np.random.default_rng(seed).permutation(count)]


def check_repair(gpu, pop, codes, coords):
    """ibs_tile_list(coords) with the dense part on the popcount kernel and on the tensor cores, twice each, against oracle_py.ibs."""
    assert_form(codes, "indexed")
    want = tiles_of(O.ibs(pop), coords)
    for tensor in (False, True):
        gpu.set_ibs_tensor_cores(tensor)
        for run in (1, 2):
            assert np.array_equal(gpu.ibs_tile_list(coords), want), f"tensor={tensor}, run {run}"
            assert gpu.ibs_used_tensor_cores() == tensor
    gpu.set_ibs_tensor_cores(True)


REPAIR_A = (256, 40_000, {g: 4_400 for g in range(3, 256, 8)})          # 140,800 dropped rows, 550 per genome on average
REPAIR_B = (128, 70_000, {7: 66_000, 20: 2_000, 64: 2_000, 65: 2_000, 100: 2_000, 127: 2_000})   # 76,000, one genome > 65,520


@pytest.fixture(scope="module")
def repair_a():
    n, n_loci, heavy = REPAIR_A
    codes = heavy_codes(n, n_loci, heavy, SEED + 3)
    return codes, sum(heavy.values()), max(heavy.values())


@pytest.fixture(scope="module")
def repair_b():
    n, n_loci, heavy = REPAIR_B
    codes = heavy_codes(n, n_loci, heavy, SEED + 4)
    return codes, sum(heavy.values()), max(heavy.values())


@pytest.mark.parametrize("split", [False, True], ids=["one chunk", "split"])
def test_repair_segments(gpu, sms, repair_a, split):
    """256 x 40,000 with the dropped rows concentrated in 32 genomes (550 per genome on average): the fewest listed tiles from
    4 x SMs on with segs > 1 and a one-chunk dense plan (J cleared by the 2-D memset; 592 tiles on a B200), or a split plan
    (the whole accumulator cleared; 593)."""
    codes, n_dropped, max_rows = repair_a
    n, n_loci = codes.shape[1], codes.shape[0]
    p = first_plan([(t, n_loci, sms, n_dropped, n, max_rows) for t in range(4 * sms, 8 * sms)],
                   lambda p: p["segs"] > 1 and (p["n_chunks"] > 1) == split)
    show(f"repair {n} x {n_loci}, {'split' if split else 'one chunk'}", p)
    pop = upload_codes(gpu, codes)
    check_repair(gpu, pop, codes, listed_tiles(IP.side(n), p["n_tiles"], SEED + 5))


@pytest.mark.parametrize("segments", [2, 1])
def test_repair_counter_flush(gpu, sms, repair_b, segments):
    """128 x 70,000 with one genome of 66,000 dropped rows. segs = 2: the four tiles of the grid, so each segment walks 33,000
    rows and flushes its counters once (J added atomically). segs = 1: 8 x SMs listed tiles, so one thread walks all 66,000
    rows in three counter passes (J stored by the first, added by the others)."""
    codes, n_dropped, max_rows = repair_b
    n, n_loci = codes.shape[1], codes.shape[0]
    n_tiles = 4 if segments == 2 else 8 * sms
    p = IP.plan(n_tiles, n_loci, sms, n_dropped, n, max_rows)
    show(f"repair flush {n} x {n_loci}, {segments} segment(s)", p)
    assert p["segs"] == segments and p["walk_passes"] == (2 if segments == 2 else 3)
    pop = upload_codes(gpu, codes)
    check_repair(gpu, pop, codes, listed_tiles(IP.side(n), n_tiles, SEED + 6))


# ---- slab drivers ---------------------------------------------------------------------------------------------------------------
SLAB_GENOMES, SLAB_LOCI = 8_200, 300           # 8,385 upper tiles: more than one launch
ROW_BLOCK = 1_024


@pytest.fixture(scope="module", params=["indexed", "validity plane"])
def slab_population(request):
    """8,200 x 300 with 40 genomes duplicated (KING kinship 0.5), and its references, built in row blocks: IBS uint32 [N][N][4]
    and KING float64 [N][N]."""
    form = request.param
    codes = random_codes(SLAB_GENOMES, SLAB_LOCI, form, SEED + 7)
    codes[:, 8_000:8_040] = codes[:, 100:140]
    assert_form(codes, form)
    ibs = np.empty((SLAB_GENOMES, SLAB_GENOMES, 4), dtype=np.uint32)
    kin = np.empty((SLAB_GENOMES, SLAB_GENOMES))
    for r0 in range(0, SLAB_GENOMES, ROW_BLOCK):
        rows = slice(r0, min(SLAB_GENOMES, r0 + ROW_BLOCK))
        k = K.king_codes(codes, rows=rows)
        ibs[rows] = np.stack([k["ibs0"], k["ibs1"], k["n_valid"] - k["ibs0"] - k["ibs1"], k["n_valid"]], axis=-1)
        kin[rows] = k["kinship"]
    return form, codes, ibs, kin


def king_pairs_ref(kin, t):
    a, b = np.nonzero(np.triu(kin >= t, 1))
    return a, b, kin[a, b]


@pytest.mark.parametrize("tensor", [False, True], ids=["popcount", "tensor cores"])
def test_slab_drivers(gpu, sms, slab_population, tensor):
    """8,200 x 300: ibs() of the whole matrix in two launches, ibs(1, N) in three band slabs, ibs_tile_list and ibs_tiles of
    8,200 tiles in two launches, king() whole and as a band, king_pairs at 0.0442 and at a threshold that lists ~100,000
    pairs. The one-chunk popcount plan runs 56 one-stage units per CTA on a B200."""
    form, codes, want_ibs, want_kin = slab_population
    if tensor and form != "indexed":
        pytest.skip("code 3 too dense to index: the popcount kernel only")
    n = SLAB_GENOMES
    side, n_upper = IP.side(n), IP.upper_tiles(n)
    n_dropped = int((codes == 3).sum())
    for t in sorted(set(IP.pairwise_launches(n, 0, n, 16) + IP.pairwise_launches(n, 1, n, 16))):
        show(f"slab driver {n} x {SLAB_LOCI} ({form}), a launch of {t} tiles", IP.plan(t, SLAB_LOCI, sms, n_dropped, n))
    upload_codes(gpu, codes)
    gpu.set_ibs_tensor_cores(tensor)

    def runs(call, want_launches, check, what):
        for run in (1, 2):
            gpu.ibs_timer_reset()
            got = call()
            assert len(gpu.ibs_timer_read()) == want_launches, what
            assert check(got), f"{what}, run {run}"
            assert gpu.ibs_used_tensor_cores() == tensor
            del got

    runs(gpu.ibs, 2, lambda g: np.array_equal(g, want_ibs), "ibs()")
    runs(lambda: gpu.ibs(1, n), len(IP.pairwise_launches(n, 1, n, 16)), lambda g: np.array_equal(g, want_ibs[1:]), "ibs(1, N)")
    assert len(IP.pairwise_launches(n, 1, n, 16)) >= 2

    coords = listed_tiles(side, 8_200, SEED + 8)
    want = tiles_of(want_ibs, coords)
    runs(lambda: gpu.ibs_tile_list(coords), 2, lambda g: np.array_equal(g, want), "ibs_tile_list")
    first = n_upper - 8_200
    want = tiles_of(want_ibs, upper_coords(side)[first:])
    runs(lambda: gpu.ibs_tiles(first, 1, 8_200), 2, lambda g: np.array_equal(g, want), "ibs_tiles")
    del want

    runs(gpu.king, 2, lambda g: bit_equal(g, want_kin), "king()")
    band = IP.pairwise_launches(n, 1, n, 8)
    assert len(band) >= 2
    runs(lambda: gpu.king(1, n), len(band), lambda g: bit_equal(g, want_kin[1:]), "king(1, N)")

    upper = want_kin[np.triu_indices(n, 1)]
    many = np.sort(upper[~np.isnan(upper)])[-100_000]
    for t in (0.0442, many):
        a, b, k = king_pairs_ref(want_kin, t)
        assert a.size >= (40 if t == 0.0442 else 100_000)

        def same(got):
            return np.array_equal(got["a"], a) and np.array_equal(got["b"], b) and bit_equal(got["kinship"], k)

        runs(lambda: gpu.king_pairs(t), 2, same, f"king_pairs({t})")
    gpu.set_ibs_tensor_cores(True)
