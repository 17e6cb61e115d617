"""Linkage disequilibrium on the device (kgl_b200_run_ld_pairs / kgl_b200_run_ld_prune): pair lists bit-equal to the host
restatement (tests/ld_oracle.py) -- n_valid, the bits of r^2 and the order -- over the code-3 regimes, padding genomes, split-K Gram
runs, window shapes and their boundaries; the greedy prune equal to the oracle's scan, also across slabs; determinism, every error
code, and no interference with the other Gram users of the context."""
import ctypes as C

import numpy as np
import pytest

import gram_plan_probe as GP
import ld_oracle as LD
from kgl_gene_b200.flatfile import FlatPopulation, pack_codes
from kgl_gene_b200.synth import add_multi_allelic, make_population

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    from kgl_gene_b200.capi import KglB200
    ctx = KglB200(0)
    yield ctx
    ctx.close()


def population(codes, offsets=None):
    l, n = codes.shape
    offsets = np.arange(1000, 1000 + 10 * l, 10, dtype=np.uint32) if offsets is None else np.asarray(offsets, dtype=np.uint32)
    return FlatPopulation(offsets, np.full((6, l), 0.1, dtype=np.float32), np.zeros(n, dtype=np.uint8), pack_codes(codes), n, False)


def upload(gpu, codes, offsets=None):
    pop = population(codes, offsets)
    gpu.upload_population(pop)
    return pop.offsets


def assert_same_pairs(got, want):
    assert len(got) == len(want)
    for f in ("a", "b", "n_valid"):
        assert np.array_equal(got[f], want[f]), f
    assert not got["reserved"].any()
    assert np.array_equal(got["r2"].view(np.uint64), want["r2"].view(np.uint64))


def check_pairs(gpu, codes, offsets, min_r2, wl=0, wb=0, keep=None):
    got = gpu.ld_pairs(min_r2, wl, wb, keep)
    want = LD.ld_pairs(codes, min_r2, offsets, wl, wb, keep)
    assert_same_pairs(got, want)
    return got


def with_monomorphic(codes, every=17):
    rows = np.arange(0, codes.shape[0], every)
    codes[rows] = np.where(codes[rows] == 3, 3, np.where(rows[:, None] % 2 == 0, 0, 2))
    return codes


@pytest.mark.parametrize("n,l,miss,wl,min_r2", [
    (257, 3000, 0.0, 300, 0.1),          # no code-3 cell: one Gram run
    (300, 2000, 0.002, 256, 0.05),       # few code-3 cells (indexed): four runs, mirrors
    (1000, 5001, 0.03, 3, 0.0),          # more than 1.5 % code-3 cells: not indexed; N = 1000 pads K to 1,024
    (2, 500, 0.05, 10, 0.0),             # two genomes: mostly NaN
    (129, 1500, 0.01, 2, 0.0),           # window of 2 loci
    (90, 2600, 0.004, 800, 0.3),         # a window spanning >= 3 tiles
])
def test_pairs_bit_equal(gpu, n, l, miss, wl, min_r2):
    codes = with_monomorphic(LD.planted(n, l, seed=n + l, missing=miss))
    if l == 5001:      # the premise: more code-3 cells than the index takes (kgl_b200_upload_genotypes: max(2^16, N L / 64))
        assert (codes == 3).sum() > max(1 << 16, n * l // 64)
    off = upload(gpu, codes)
    check_pairs(gpu, codes, off, min_r2, wl)


def test_pairs_multi_allelic_monomorphic_and_keep(gpu):
    pop, _ = make_population(300, 2500, seed=9, missing_rate=0.004)
    pop = add_multi_allelic(pop, 40, seed=9)
    codes = with_monomorphic(pop.codes())
    pop.packed = pack_codes(codes)
    gpu.upload_population(pop)
    keep = (np.random.default_rng(1).random(pop.n_loci) < 0.7).astype(np.uint8)
    elig = LD.eligible(codes, keep)
    assert not elig[pop.multi_rows].any() and not elig[::17].any()
    got = check_pairs(gpu, codes, pop.offsets, 0.0, 100, 0, keep)
    assert len(got) > 10000 and not np.isin(got["a"], np.flatnonzero(~elig)).any() and not np.isin(got["b"], np.flatnonzero(~elig)).any()
    check_pairs(gpu, codes, pop.offsets, 0.0, 100)


@pytest.mark.parametrize("miss", [0.0, 0.002])
def test_pairs_split_k(gpu, miss):
    """20,000 genomes: 157 k-stages; the five band tiles (three diagonal, two off) and the seven of the mirrored runs are split in
    two chunks at 148 SMs, so every run adds into cleared compact blocks."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    codes = LD.planted(20_000, 600, seed=5, missing=miss)
    a, b = LD.window_pairs(LD.eligible(codes), None, 10, 0)
    tiles = set(zip((a // 256).tolist(), (b // 256).tolist()))
    nb, nl = len(tiles), len(tiles) + sum(i != j for i, j in tiles)
    for t in (nb, nl):
        p = GP.plan(t, GP.k_stages(20_000), sms)
        print(GP.describe(f"LD band ({t} tiles)", p))
        assert p["n_chunks"] > 1
    off = upload(gpu, codes)
    check_pairs(gpu, codes, off, 0.0, 10)


def test_windows_by_bp_and_both_and_their_boundaries(gpu):
    """Offsets with small gaps, so that many pairs sit exactly at the bp limit: limits W - 1, W, W + 1 (rank, `<`) and B - 1, B,
    B + 1 (bp, `<=`) each give the oracle's list."""
    rng = np.random.default_rng(4)
    codes = LD.planted(200, 1800, seed=4, missing=0.003)
    off = np.cumsum(rng.integers(0, 4, size=1800)) + 100
    off = upload(gpu, codes, off)
    for wl in (99, 100, 101):
        check_pairs(gpu, codes, off, 0.0, wl)
    for wb in (59, 60, 61):
        check_pairs(gpu, codes, off, 0.0, 0, wb)
    check_pairs(gpu, codes, off, 0.0, 30, 90)
    check_pairs(gpu, codes, off, 0.2, 300, 40)


def test_planted_blocks_and_min_r2_zero(gpu):
    codes = LD.planted(500, 1200, seed=2, block=60, founders=2, mutation=0.002)
    off = upload(gpu, codes)
    got = check_pairs(gpu, codes, off, 0.9, 120)
    assert len(got) > 1000 and (got["r2"] == 1.0).any()
    _, _, _, r = LD.all_window_r2(codes, off, 120)
    allp = check_pairs(gpu, codes, off, 0.0, 120)
    assert len(allp) == int((~np.isnan(r)).sum())                     # min_r2 = 0: every non-NaN in-window pair


def test_nomem_then_retry(gpu):
    from kgl_gene_b200.capi import KGL_B200_ERR_NOMEM, LD_PAIR_DTYPE, LdOptions
    codes = LD.planted(100, 1000, seed=7, missing=0.002)
    off = upload(gpu, codes)
    want = LD.ld_pairs(codes, 0.3, off, 50)
    opt = LdOptions(window_loci=50)
    out = np.zeros(10, dtype=LD_PAIR_DTYPE)
    n = C.c_uint64(0)
    rc = gpu.lib.kgl_b200_run_ld_pairs(gpu.h, C.byref(opt), C.c_double(0.3), C.c_uint64(10), C.c_void_p(out.ctypes.data), C.byref(n))
    assert rc == KGL_B200_ERR_NOMEM and n.value == len(want) > 10 and not out.view(np.uint8).any()
    assert_same_pairs(gpu.ld_pairs(0.3, 50, capacity=10), want)
    assert_same_pairs(gpu.ld_pairs(0.3, 50, capacity=len(want)), want)


@pytest.mark.parametrize("miss,wl,wb,t", [(0.0, 100, 0, 0.2), (0.003, 100, 0, 0.2), (0.003, 0, 500, 0.5), (0.01, 40, 300, 0.1)])
def test_prune_equals_the_oracle_scan(gpu, miss, wl, wb, t):
    codes = LD.planted(300, 3000, seed=11, block=50, founders=2, mutation=0.01, missing=miss, multi_rows=5)
    off = np.cumsum(np.random.default_rng(2).integers(1, 20, size=3000)) + 10
    off = upload(gpu, codes, off)
    keep, n_kept = gpu.ld_prune(t, wl, wb)
    want = LD.ld_prune(codes, t, off, wl, wb)
    assert np.array_equal(keep, want) and n_kept == int(want.sum()) > 0
    assert gpu.pca(k=3, keep=keep)["n_loci_used"] == n_kept


def test_prune_across_slabs(gpu):
    """110,000 loci with code-3 cells and a 40-locus window: every 256-locus block row holds its diagonal tile (4 int32 blocks)
    and the next one (6), so the band takes ~4,300 blocks, more than one 1 GiB slab (4,096 blocks). Pairs whose second locus lies
    past a slab stay pending across the cut."""
    codes = LD.planted(48, 110_000, seed=3, block=30, founders=2, mutation=0.01, missing=0.01)
    off = upload(gpu, codes)
    elig = LD.eligible(codes)
    a, b, n, r = LD.all_window_r2(codes, off, 40)
    blocks = sum(4 if i == j else 6 for i, j in set(zip((a // 256).tolist(), (b // 256).tolist())))
    assert blocks * 65536 * 4 > 1 << 30
    keep, n_kept = gpu.ld_prune(0.3, 40)
    want = LD.prune_scan(codes.shape[0], elig, a, b, r, 0.3)
    assert np.array_equal(keep, want) and n_kept == int(want.sum())
    got = gpu.ld_pairs(0.5, 40)
    take = r >= 0.5
    assert np.array_equal(got["a"], a[take]) and np.array_equal(got["b"], b[take]) and np.array_equal(got["n_valid"], n[take])
    assert np.array_equal(got["r2"].view(np.uint64), r[take].view(np.uint64))


def test_deterministic(gpu):
    codes = LD.planted(400, 2000, seed=6, missing=0.005)
    upload(gpu, codes)
    x, y = gpu.ld_pairs(0.0, 200), gpu.ld_pairs(0.0, 200)
    assert x.tobytes() == y.tobytes()
    assert gpu.ld_prune(0.2, 200)[0].tobytes() == gpu.ld_prune(0.2, 200)[0].tobytes()


def test_errors(gpu):
    from kgl_gene_b200.capi import KglB200, KglError, LdOptions
    fresh = KglB200(0)
    fresh.n_loci = 10
    with pytest.raises(KglError, match=r"run_ld_pairs failed \[2\]"):
        fresh.ld_pairs(0.1, 10)
    with pytest.raises(KglError, match=r"run_ld_prune failed \[2\]"):
        fresh.ld_prune(0.1, 10)
    fresh.close()
    codes = LD.planted(30, 500, seed=2)
    pop = population(codes)
    gpu.upload_genotypes(pop.packed, 30)
    gpu.upload_loci(pop.af, None)                                      # no offsets: a bp window cannot be applied
    for call in (lambda: gpu.ld_pairs(0.1, 0, 100), lambda: gpu.ld_prune(0.1, 10, 100)):
        with pytest.raises(KglError, match=r"failed \[2\]"):
            call()
    gpu.upload_loci(pop.af, pop.offsets[::-1].copy())                  # decreasing offsets
    with pytest.raises(KglError, match=r"run_ld_pairs failed \[1\]"):
        gpu.ld_pairs(0.1, 0, 100)
    gpu.upload_loci(pop.af, pop.offsets)
    for bad in (dict(min_r2=float("nan"), window_loci=10), dict(min_r2=0.1)):
        with pytest.raises(KglError, match=r"run_ld_pairs failed \[1\]"):
            gpu.ld_pairs(**bad)
    for bad in (dict(max_r2=float("nan"), window_loci=10), dict(max_r2=0.1)):
        with pytest.raises(KglError, match=r"run_ld_prune failed \[1\]"):
            gpu.ld_prune(**bad)
    opt, n = LdOptions(window_loci=10), C.c_uint64(0)
    out = np.zeros(500, dtype=np.uint8)
    assert gpu.lib.kgl_b200_run_ld_pairs(gpu.h, C.byref(opt), C.c_double(0.1), C.c_uint64(10), None, C.byref(n)) == 1
    assert gpu.lib.kgl_b200_run_ld_pairs(gpu.h, C.byref(opt), C.c_double(0.1), C.c_uint64(10), C.c_void_p(out.ctypes.data), None) == 1
    assert gpu.lib.kgl_b200_run_ld_prune(gpu.h, C.byref(opt), C.c_double(0.1), None, C.byref(n)) == 1
    assert gpu.lib.kgl_b200_run_ld_prune(gpu.h, C.byref(opt), C.c_double(0.1), C.c_void_p(out.ctypes.data), None) == 1


def test_error_too_many_genomes(gpu):
    """n_genomes >= 2^25 would let the int64 terms reach 2^53: refused before any work (device-generated matrix)."""
    from kgl_gene_b200.capi import KglB200, KglError
    ctx = KglB200(0)
    n = 1 << 25
    ctx.upload_loci(np.zeros((1, 2), dtype=np.float32))
    ctx.set_genome_superpop(np.zeros(n, dtype=np.uint8))
    ctx.synth_genotypes(1, n, 2, np.zeros(n), missing_rate=0.0)
    with pytest.raises(KglError, match=r"run_ld_pairs failed \[1\]"):
        ctx.ld_pairs(0.1, 2)
    with pytest.raises(KglError, match=r"run_ld_prune failed \[1\]"):
        ctx.ld_prune(0.1, 2)
    ctx.close()


def test_no_interference(gpu):
    pop, _ = make_population(300, 3000, seed=21, missing_rate=0.003)
    gpu.upload_population(pop)
    gpu.select_loci(spacing=0)
    gpu.count_and_inbreed()
    x = np.random.default_rng(0).standard_normal((300, 5))
    before = (gpu.fetch_locus_counts(), gpu.grm_product(x)[0], gpu.king_pairs(-1.0), gpu.ibs(), gpu.gram())
    gpu.ld_pairs(0.0, 300)
    gpu.ld_prune(0.2, 0, 2000)
    after = (gpu.fetch_locus_counts(), gpu.grm_product(x)[0], gpu.king_pairs(-1.0), gpu.ibs(), gpu.gram())
    assert np.array_equal(before[0], after[0])                           # LD counts into PCA's buffer, not the caller's
    assert before[1].tobytes() == after[1].tobytes() and before[2].tobytes() == after[2].tobytes()
    assert np.array_equal(before[3], after[3]) and np.array_equal(before[4], after[4])
