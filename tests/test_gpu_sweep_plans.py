"""The estimator sweeps (k_terms_fast, kgl_gene_b200/csrc/terms_fast.cuh; k_genome_terms, sample_major.cuh) and the moment tables
(terms_moments.cuh, terms_moments_mma.cuh) at the launch plans and unit splits they reach.

k_terms_fast is the only path for RitlandLocus, for the unphased root search and for the exact sweeps of HallME and the phased
root search. Each sweep case sizes its population with the planner (tests/terms_plan_probe.cu) on this device's SM count and
shared-memory limit, asserts the plan it names, prints it, and runs twice on one context, so stale shared or chunk state shows;
both runs must agree bit for bit and with oracle_py.inbreed (class counts equal, F and the estimator's value to 1e-9).

The moment-table cases restate the tensor-core builder's unit rule in numpy (a unit ends at every 4,096 sorted items of a
population and wherever the (bins, codes) of the frequency-sorted loci change) so that each can assert the split it relies on.
HallME with one sweep is f (n_hom + (1 - f) S1) / n, which checks every genome's S1 from the tables against the oracle directly.
tests/test_terms_plan.py pins these plans at 148 SMs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_py as O
import terms_plan_probe as TP
from conftest import results_matrix

pytestmark = pytest.mark.gpu

SEED = 20261022
TOL = 1e-9
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


@pytest.fixture(scope="module")
def device():
    """(SM count, opt-in shared memory per block) of device 0."""
    import torch
    prop = torch.cuda.get_device_properties(0)
    return prop.multi_processor_count, prop.shared_memory_per_block_optin


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.close()


def new_context():
    from kgl_gene_b200.capi import KglB200
    return KglB200(0)


def sweep_plan(device, name, mode, n_genomes, n_loci, rows=(0, TP.NO_WINDOW)):
    sms, smem = device
    p = TP.plan(mode, TP.gblocks_of(n_genomes), TP.term_words(n_loci), sms, rows[0], rows[1], smem)
    print(TP.describe(name, p))
    assert p["ok"] == 1, TP.describe(name, p)
    return p


def device_population(gpu, n, n_loci, unphased=False, af=None, superpop=None):
    """Generated on the device, downloaded: the oracle's input."""
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    offsets, af0 = make_loci(n_loci, SEED)
    sp, f = make_genomes(n, SEED)
    af = af0 if af is None else af
    sp = sp if superpop is None else superpop
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(sp)
    gpu.set_unphased(unphased)
    gpu.synth_genotypes(SEED, n, n_loci, f, missing_rate=0.002)
    return FlatPopulation(offsets, af, sp, gpu.download_genotypes(), n, unphased)


def log_uniform_af(n_loci, seed, lo=1e-12, hi=0.5):
    """Frequencies log-uniform over [lo, hi] in every population: every bin of the moment tables is used."""
    rng = np.random.default_rng(seed)
    return np.exp(rng.uniform(np.log(lo), np.log(hi), size=(6, n_loci))).astype(np.float32)


def subset(n):
    """One genome of every 32-genome block (a different lane in each), and the last genome: every warp and slot of a plan."""
    g = np.arange((n + 31) // 32) * 32 + np.arange((n + 31) // 32) % 32
    return np.unique(np.append(g[g < n], n - 1)).astype(np.uint32)


def bit_equal(a, b):
    for f in a.dtype.names:
        x, y = np.ascontiguousarray(a[f]), np.ascontiguousarray(b[f])
        if x.tobytes() != y.tobytes():
            return False
    return True


def rel_err(a, b, floor=0.0):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), max(floor, 1e-300))) if a.size else 0.0


def assert_matches(got, want, tag, tol=TOL):
    c_got, f_got = results_matrix(got)
    c_want, f_want = results_matrix(want)
    assert np.array_equal(c_got, c_want), tag
    assert rel_err(f_got, f_want, floor=1e-6) < tol, tag
    a, b = got["inbred_allele_sum"], want["inbred_allele_sum"]
    assert np.array_equal(np.isfinite(a), np.isfinite(b)), tag
    fin = np.isfinite(b)
    err = np.abs(a[fin] - b[fin]) / np.maximum(np.abs(b[fin]), 1.0)
    assert err.size == 0 or err.max() < tol, (tag, float(err.max()))


ESTIMATORS = {   # name -> (GPU call kwargs, oracle kwargs); HallME and the phased root search on the exact sweeps
    "RitlandLocus": ({}, {}),
    "HallME": (dict(exact_sweeps=True, hall_sweeps=50), dict(sweeps=50)),
    "Loglikelihood": (dict(exact_sweeps=True), {}),
}


def run_and_check(gpu, pop, sel, algo, kwargs, okw, genomes, tag):
    kw, okw = dict(kwargs), dict(okw)
    if algo == "HallME":
        start = np.random.default_rng(SEED).uniform(0.05, 1.0, size=pop.n_genomes)
        kw["hall_start"], okw["start"] = start, start
    first = gpu.inbreed(algo, **kw)
    second = gpu.inbreed(algo, **kw)
    assert bit_equal(first, second), (tag, "second run differs")
    want = O.inbreed(pop, sel, algo, genomes=genomes, **okw)
    assert_matches(first[genomes], want, tag)
    return first


# ---- k_terms_fast: CTA shapes ----------------------------------------------------------------------------------------------------
SHAPES = [  # name, genomes, loci, warps, slots
    ("4 warps", 100, 20_000, 4, 1),
    ("8 warps", 230, 20_000, 8, 1),
    ("24 x 8", 6_144, 20_000, 24, 8),
    ("22 x 8, partial row", 5_408, 20_000, 22, 8),
]
MODE_OF = {"RitlandLocus": "RITLAND", "HallME": "HALL", "Loglikelihood": "NEWTON"}


@pytest.mark.parametrize("name,n,n_loci,warps,slots", SHAPES, ids=[s[0] for s in SHAPES])
def test_sweep_shapes(gpu, device, name, n, n_loci, warps, slots):
    """RitlandLocus, HallME (exact sweeps) and the phased root search (exact sweeps: LIMITS, then NEWTON) at the small CTAs, 24
    warps x 8 slots and 22 x 8 = 176 slots for 169 genome blocks."""
    pop = device_population(gpu, n, n_loci)
    sel = O.select_all_pops(pop)
    gpu.select_loci()
    genomes = subset(n)
    for algo, (kw, okw) in ESTIMATORS.items():
        modes = ("LIMITS", "NEWTON") if algo == "Loglikelihood" else (MODE_OF[algo],)
        for m in modes:
            p = sweep_plan(device, f"{name} {algo}", m, n, n_loci)
            assert (p["warps"], p["slots"]) == (warps, slots)
        run_and_check(gpu, pop, sel, algo, kw, okw, genomes, (name, algo))


@pytest.mark.parametrize("n", [5_408, 6_144])
def test_unphased_root_search_fits(gpu, device, n):
    """The unphased root search (LIMITS, then NEWTON_U with three accumulators per slot) at the sizes whose 8-slot plan of 22 and
    24 warps would need 234,240 and 246,528 B of shared memory: the planner takes 16 x 8 in two rows of CTAs instead. Before
    that, kgl_b200_run_inbreed returned an error here."""
    n_loci = 20_000
    p = sweep_plan(device, f"unphased {n}", "NEWTON_U", n, n_loci)
    assert p["smem"] <= device[1] and p["slots"] == 8 and p["gy"] >= 2
    pop = device_population(gpu, n, n_loci, unphased=True)
    sel = O.select_all_pops(pop)
    gpu.select_loci()
    run_and_check(gpu, pop, sel, "Loglikelihood", {}, {}, subset(n), ("unphased", n))


# ---- k_terms_fast: selection windows ---------------------------------------------------------------------------------------------
def window_loci(sms):
    """Loci whose sample-major copy has sms + 9 tiles of 8 words, the last of 4: more tiles than one per CTA (two per chunk,
    the last chunk short) at 24 x 8 slots (40,000 loci on a B200)."""
    return ((sms + 9) * 8 - 4) * 32 - 64


WINDOWS = ["inside one tile", "one row past a tile", "to a 4-word last tile", "every tile"]


@pytest.mark.parametrize("window", WINDOWS)
def test_sweep_windows(gpu, device, window):
    """Selection windows over 6,144 genomes: only the tiles holding a selectable row are swept, in chunks of tile_begin +
    blockIdx.x * tiles_per_chunk."""
    n, n_loci = 6_144, window_loci(device[0])
    rows = {"inside one tile": (300, 480), "one row past a tile": (100, 513), "to a 4-word last tile": (n_loci - 1_000, n_loci),
            "every tile": (0, n_loci)}[window]
    p = sweep_plan(device, f"window {window}", "NEWTON", n, n_loci, rows)
    tiles = {"inside one tile": (1, 2), "one row past a tile": (0, 3)}.get(window)
    if tiles:
        assert (p["tile_begin"], p["tile_end"]) == tiles
    else:
        assert p["tile_end"] == (TP.term_words(n_loci) + 7) // 8 and TP.term_words(n_loci) % 8 == 4
    if window == "every tile":
        assert p["tiles_per_chunk"] > 1 and p["last_chunk_tiles"] < p["tiles_per_chunk"]
    pop = device_population(gpu, n, n_loci)
    sel_kw = dict(lower=int(pop.offsets[rows[0]]), upper=int(pop.offsets[rows[1] - 1]))
    sel = O.select_all_pops(pop, **sel_kw)
    gpu.select_loci(**sel_kw)
    genomes = subset(n)
    for algo, (kw, okw) in ESTIMATORS.items():
        run_and_check(gpu, pop, sel, algo, kw, okw, genomes, (window, algo))


def test_loglik_grid_short_last_chunk(gpu, device):
    """loglik_grid on k_genome_terms with a last chunk of fewer words than the others (2,048 x 32,128 on a B200: 126 chunks of
    8 words, the last of 4)."""
    sms, smem = device
    n, n_loci = 2_048, 32_128
    p = TP.plan("RITLAND", TP.device_gblocks(n), TP.term_words(n_loci), sms, 0, TP.NO_WINDOW, smem)
    print(TP.describe("loglik_grid", p))
    assert p["term_n_chunks"] > 1 and p["term_last_chunk_words"] < p["term_words_per_chunk"]
    pop = device_population(gpu, n, n_loci)
    sel = O.select_all_pops(pop)
    gpu.select_loci()
    grid = np.array([-0.3, 0.0, 0.11, 0.6])
    for _ in range(2):
        got, want = gpu.loglik_grid(grid), O.loglik_grid(pop, sel, grid)
        fin = np.isfinite(want)
        assert np.array_equal(np.isfinite(got), fin)
        assert rel_err(got[fin], want[fin]) < 1e-11


# ---- moment tables ---------------------------------------------------------------------------------------------------------------
MOM_CHUNK, BINS_MAX = 4096, 2560


def mom_bin(r):
    bits = np.ascontiguousarray(r, dtype=np.float64).view(np.int64)
    e = ((bits >> 52) & 0x7FF) - 1023
    b = np.where((e < -40) | (e >= 40), -1, (e + 40) * 32 + ((bits >> 47) & 31))
    return np.where(e == 1024, np.where(((bits & 0xFFFFFFFFFFFFF) == 0) & (bits > 0), BINS_MAX, -1), b)


def mom_classify(af, unphased):
    """mom_classify of terms_moments.cuh: (common code, rare code, r_common, r_rare) per locus."""
    p = np.clip(np.nan_to_num(af.astype(np.float64), nan=0.0), 0.0, 1.0)
    q = np.clip(1.0 - p, 0.0, 1.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        r0 = np.where(1.0 - q > 0, q / (1.0 - q), np.inf)
        r2 = np.where(1.0 - p > 0, p / (1.0 - p), np.inf)
    ref_in, alt = q > 0.01, -1 if unphased else 2
    ref_common = q >= p
    cc = np.where(ref_common, np.where(ref_in, 0, -1), alt)
    rc = np.where(ref_common, alt, np.where(ref_in, 0, -1))
    return cc, rc, np.where(ref_common, r0, r2), np.where(ref_common, r2, r0)


def moment_units(pop, sel):
    """The tensor-core builder's units as k_mom_keys / k_mom_bounds / k_mom_units form them, restated: per population the
    selected loci sorted by the float bits of p (stable: rows ascending), a boundary at every 4,096th item and at every change of
    (common bin, rare bin, codes). Returns ([unit sizes of each population], nbt = bins spanned + the a == 1 class)."""
    sizes, lo, hi = [], BINS_MAX, -1
    for k in range(pop.af.shape[0]):
        a = pop.af[k, np.flatnonzero(sel[k])]
        a = a[np.argsort(np.clip(np.nan_to_num(a, nan=0.0), 0, 1).astype(np.float32).view(np.uint32), kind="stable")]
        if a.size == 0:
            sizes.append([])
            continue
        cc, rc, r_c, r_r = mom_classify(a, pop.unphased)
        cb, rb = np.where(cc >= 0, mom_bin(r_c), 0xFFFF), np.where(rc >= 0, mom_bin(r_r), 0xFFFF)
        seg = np.stack([cb, rb, cc, rc], axis=1)
        bound = np.arange(a.size) % MOM_CHUNK == 0
        bound[1:] |= (seg[1:] != seg[:-1]).any(axis=1)
        sizes.append(np.diff(np.append(np.flatnonzero(bound), a.size)).tolist())
        used = np.concatenate([cb[(cc >= 0) & (cb < BINS_MAX)], rb[rc >= 0]])
        assert (used >= 0).all() and (used < BINS_MAX).all(), "a class outside the bins: the run would use the exact kernels"
        lo, hi = min(lo, int(used.min())), max(hi, int(used.max()))
    return sizes, hi - lo + 2


def check_tables(gpu, pop, sel, tag, genomes=None):
    """HallME with one sweep (the tables' S1 for every genome) at 1e-10, 50 sweeps and the root search at 1e-9, each on the
    tensor-core builder; the CUDA-core builder bit for bit. The tables belong to the selection, so every run selects again and
    builds them afresh."""
    genomes = np.arange(pop.n_genomes, dtype=np.uint32) if genomes is None else genomes
    start = np.random.default_rng(SEED + 1).uniform(0.05, 1.0, size=pop.n_genomes)
    out = {}
    for algo, kw, okw, tol in (("HallME", dict(hall_start=start, hall_sweeps=1), dict(start=start, sweeps=1), 1e-10),
                               ("HallME", dict(hall_start=start, hall_sweeps=50), dict(start=start, sweeps=50), TOL),
                               ("Loglikelihood", {}, {}, TOL)):
        gpu.select_loci()
        got = gpu.inbreed(algo, **kw)
        assert gpu.used_moment_tables() == 2, (tag, algo)
        assert_matches(got[genomes], O.inbreed(pop, sel, algo, genomes=genomes, **okw), (tag, algo, kw.get("hall_sweeps")), tol)
        gpu.select_loci()
        cuda_cores = gpu.inbreed(algo, moments_on_cuda_cores=True, **kw)
        assert gpu.used_moment_tables() == 1, (tag, algo)
        assert bit_equal(got, cuda_cores), (tag, algo, "tensor-core and CUDA-core tables differ")
        out[(algo, kw.get("hall_sweeps"))] = got
    return out


def test_moment_units_split_at_4096(gpu):
    """One frequency on 8,193 loci: every population's loci form units of 4,096 + 4,096 + 1 items with the same bins, so the
    tensor-core builder restarts its accumulation at the same (bins, codes) twice."""
    n, n_loci = 300, 8_193
    pop = device_population(gpu, n, n_loci, af=np.full((6, n_loci), 0.3, dtype=np.float32))
    sel = O.select_all_pops(pop)
    gpu.select_loci()
    sizes, _ = moment_units(pop, sel)
    assert all(s == [4096, 4096, 1] for s in sizes), sizes
    check_tables(gpu, pop, sel, "4,096 split")


def test_moment_tables_every_bin(gpu):
    """Frequencies log-uniform over [1e-12, 0.5]: nbt is close to its maximum of 2,561, and k_mom_run holds nbt x 64 B of
    shared memory (about 164 KB)."""
    n, n_loci = 300, 30_000
    pop = device_population(gpu, n, n_loci, af=log_uniform_af(n_loci, SEED))
    sel = O.select_all_pops(pop)
    gpu.select_loci()
    sizes, nbt = moment_units(pop, sel)
    print(f"every bin: nbt {nbt} ({nbt * 64} B of k_mom_run shared memory), {sum(map(len, sizes))} units")
    assert 2_500 <= nbt <= 2_561
    check_tables(gpu, pop, sel, "every bin")


def lists_after_hall(gpu_a, gpu_b, pop, sel, genomes, tag):
    """HallME on the tables, then the root search on the same selection (context a), against the root search after an exact
    HallME (context b: the tables are built for the first time). Returns the launches of each root search; both results must be
    equal bit for bit and match the oracle."""
    start = np.random.default_rng(SEED + 2).uniform(0.05, 1.0, size=pop.n_genomes)
    deltas, res = [], []
    for ctx, exact in ((gpu_a, False), (gpu_b, True)):
        ctx.select_loci()
        ctx.inbreed("HallME", hall_start=start, hall_sweeps=3, exact_sweeps=exact)
        assert ctx.used_moment_tables() == (0 if exact else 2), tag
        before = ctx.launch_count()
        res.append(ctx.inbreed("Loglikelihood"))
        deltas.append(ctx.launch_count() - before)
        assert ctx.used_moment_tables() == 2, tag
    assert bit_equal(res[0], res[1]), (tag, "root search after HallME differs from a fresh build")
    assert_matches(res[0][genomes], O.inbreed(pop, sel, "Loglikelihood", genomes=genomes), tag)
    print(f"{tag}: root-search launches after HallME's tables {deltas[0]}, after a fresh build {deltas[1]}")
    return deltas


def test_moment_counts_kept_then_lists(gpu):
    """HallME keeps the tensor-core builder's per-unit counts; the root search after it builds only its lists (fewer launches
    than a fresh build) and equals a fresh build bit for bit."""
    from kgl_gene_b200.flatfile import FlatPopulation
    n, n_loci = 600, 20_000
    pop = device_population(gpu, n, n_loci, af=log_uniform_af(n_loci, SEED + 3, lo=1e-6))
    sel = O.select_all_pops(pop)
    sizes, _ = moment_units(pop, sel)
    npad = (n + 63) // 64 * 64
    assert sum(map(len, sizes)) * npad * 8 <= 2 << 30
    other = new_context()
    try:
        other.upload_population(FlatPopulation(pop.offsets, pop.af, pop.superpop, pop.packed, n, False))
        kept, fresh = lists_after_hall(gpu, other, pop, sel, subset(n), "counts kept")
    finally:
        other.close()
    assert kept < fresh


def test_moment_counts_dropped_at_24000_genomes(gpu):
    """24,000 genomes with every bin in every population: n_units x Npad x 8 B exceeds 2 GiB, so HallME does not keep the
    per-unit counts and the root search after it rebuilds its tables in full on the tensor cores (as many launches as a fresh
    build, the same result bit for bit)."""
    from kgl_gene_b200.flatfile import FlatPopulation
    n, n_loci = 24_000, 30_000
    pop = device_population(gpu, n, n_loci, af=log_uniform_af(n_loci, SEED + 4))
    sel = O.select_all_pops(pop)
    sizes, nbt = moment_units(pop, sel)
    n_units, npad = sum(map(len, sizes)), (n + 63) // 64 * 64
    print(f"24,000 genomes: {n_units} units, nbt {nbt}; counts would take {n_units * npad * 8 / 2**30:.2f} GiB")
    assert n_units > 1.2 * (2 << 30) / (npad * 8)
    other = new_context()
    try:
        other.upload_population(FlatPopulation(pop.offsets, pop.af, pop.superpop, pop.packed, n, False))
        after_hall, fresh = lists_after_hall(gpu, other, pop, sel, subset(n)[::4], "counts dropped")
    finally:
        other.close()
    assert after_hall == fresh


def labels_splitting_tiles(n):
    """Populations that split the 256-genome fill tile and the 128-genome MMA tile: genomes 128..255 are population 1, the last
    genome alone is population 3, population 5 is empty, the rest interleave populations 0, 2 and 4."""
    sp = np.array([0, 2, 4], dtype=np.uint8)[np.arange(n) % 3]
    sp[128:256] = 1
    if n > 1:
        sp[n - 1] = 3
    return sp


@pytest.mark.parametrize("n", [1, 63, 65, 127, 129, 257])
def test_moment_tables_split_tiles(gpu, n):
    """Population tile ranges of k_mom_mma (128 genomes) and k_mom_unit_fill (256) that start and end inside a tile, a population
    of one genome and one of none, at genome counts around both tile sizes."""
    n_loci = 3_000
    pop = device_population(gpu, n, n_loci, superpop=labels_splitting_tiles(n))
    sel = O.select_all_pops(pop)
    gpu.select_loci()
    check_tables(gpu, pop, sel, f"split tiles, {n} genomes")


_FALLBACK = r"""
import json, sys
import numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
from kgl_gene_b200.capi import KglB200
from kgl_gene_b200.synth import make_population
pop, _ = make_population(300, 5_000, seed={seed})
ctx = KglB200(0)
ctx.upload_population(pop)
ctx.select_loci()
start = np.random.default_rng({seed}).uniform(0.05, 1.0, size=pop.n_genomes)
out = {{}}
for algo, kw in (("HallME", dict(hall_start=start, hall_sweeps=20)), ("Loglikelihood", {{}})):
    a = ctx.inbreed(algo, **kw)
    used = ctx.used_moment_tables()
    b = ctx.inbreed(algo, exact_sweeps=True, **kw)
    out[algo] = [used, a.tobytes() == b.tobytes()]
ctx.close()
print(json.dumps(out))
"""


def test_moment_bytes_limit_sends_the_run_to_the_exact_sweeps():
    """KGL_B200_MOMENT_BYTES=1 (read once per process, so in a process of its own): no moment tables, and HallME and the root
    search equal their exact sweeps bit for bit."""
    env = dict(os.environ, KGL_B200_MOMENT_BYTES="1")
    code = _FALLBACK.format(root=ROOT, tests=HERE, seed=SEED)
    proc = subprocess.run([sys.executable, "-s", "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr
    out = json.loads(proc.stdout.strip().splitlines()[-1])
    assert out == {"HallME": [0, True], "Loglikelihood": [0, True]}, out
