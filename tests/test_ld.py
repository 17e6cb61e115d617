"""CPU checks of linkage disequilibrium: the host restatement (tests/ld_oracle.py) against numpy.corrcoef, the prune oracle's
defining properties, the band tile list of the device path (ld_band, compiled as tests/ld_band_probe.cu) and the C ABI's structs."""
import ctypes as C
import json
import subprocess

import numpy as np
import pytest

import ld_oracle as LD
import plan_probe


def test_oracle_r2_is_the_squared_pairwise_complete_correlation():
    rng = np.random.default_rng(3)
    codes = LD.planted(150, 120, seed=4, block=20, mutation=0.05, missing=0.04)
    codes[7] = np.where(rng.random(150) < 0.5, 3, 0)                     # a multi-allelic-like row: never eligible
    codes[9] = np.where(codes[9] == 3, 3, 1)                              # all heterozygous: p = 1/2, variance 0 -> NaN
    a, b, n, r = LD.all_window_r2(codes, window_loci=30)
    assert len(a) > 1000 and 7 not in a and 7 not in b
    for i, j, nv, rv in zip(a, b, n, r):
        ok = (codes[i] != 3) & (codes[j] != 3)
        assert nv == ok.sum()
        x, y = codes[i][ok].astype(float), codes[j][ok].astype(float)
        if x.std() == 0 or y.std() == 0:
            assert np.isnan(rv)
        else:
            assert abs(rv - np.corrcoef(x, y)[0, 1] ** 2) <= 1e-12
    assert np.isnan(r[(a == 9) | (b == 9)]).all()


def test_window_definition():
    elig = np.ones(10, dtype=bool)
    elig[[2, 5]] = False
    off = np.array([0, 5, 9, 10, 20, 21, 22, 40, 41, 100])
    a, b = LD.window_pairs(elig, off, 2, 0)
    assert list(zip(a, b)) == [(0, 1), (1, 3), (3, 4), (4, 6), (6, 7), (7, 8), (8, 9)]     # adjacent eligible loci
    a, b = LD.window_pairs(elig, off, 0, 10)
    assert list(zip(a, b)) == [(0, 1), (0, 3), (1, 3), (3, 4), (4, 6), (7, 8)]               # offset distance <= 10
    a, b = LD.window_pairs(elig, off, 3, 10)
    assert list(zip(a, b)) == [(0, 1), (0, 3), (1, 3), (3, 4), (4, 6), (7, 8)]


@pytest.mark.parametrize("missing", [0.0, 0.02])
def test_prune_oracle_is_independent_and_maximal(missing):
    codes = LD.planted(200, 600, seed=8, block=30, founders=2, mutation=0.02, missing=missing, multi_rows=5)
    off = np.cumsum(np.random.default_rng(1).integers(1, 50, size=600))
    for wl, wb, t in [(50, 0, 0.2), (0, 400, 0.5), (20, 300, 0.1)]:
        elig = LD.eligible(codes)
        a, b, n, r = LD.all_window_r2(codes, off, wl, wb)
        keep = LD.ld_prune(codes, t, off, wl, wb)
        assert not keep[~elig].any() and 0 < keep.sum() < elig.sum()
        both = (keep[a] == 1) & (keep[b] == 1)
        assert not (r[both] > t).any()                                    # independent
        for l in np.flatnonzero(elig & (keep == 0)):                      # maximal: pruned by an earlier kept partner
            hit = (b == l) & (keep[a] == 1) & (r > t)
            assert hit.any()


# ---- the band tile list ------------------------------------------------------------------------------------------------

def band(rank, offsets, window_loci, window_bp, code3, budget):
    exe = plan_probe.probe_binary("ld_band_probe")
    text = f"{len(rank)} {window_loci} {window_bp} {int(code3)} {budget}\n" + " ".join(map(str, rank)) + "\n" + " ".join(map(str, offsets)) + "\n"
    return json.loads(subprocess.run([exe], input=text, capture_output=True, text=True, check=True).stdout)


def band_cases():
    rng = np.random.default_rng(11)
    cases = []
    for i in range(36):
        l = int(rng.choice([1, 255, 256, 257, 1000, 3001, 9000]))
        keep_rate = [1.0, 0.9, 0.3, 0.02][i % 4]
        elig = rng.random(l) < keep_rate
        if i % 9 == 4:                                                    # long stretches without an eligible locus
            elig[l // 5: l // 2] = False
        off = np.cumsum(rng.integers(0, 3 if i % 3 else 200, size=l)).astype(np.int64) + 1000
        kind = i % 3
        wl = int(rng.choice([2, 3, 256, 257, 700, 5000])) if kind != 1 else 0
        wb = int(rng.choice([1, 50, 600, 30000])) if kind != 0 else 0
        code3 = bool(i % 2)
        budget = int(rng.choice([1, 6, 40, 1 << 30])) << 18
        cases.append((elig, off, wl, wb, code3, budget))
    return cases


@pytest.mark.parametrize("case", range(36))
def test_band_tiles_cover_exactly_the_window(case):
    try:
        plan_probe.probe_binary("ld_band_probe")
    except FileNotFoundError:
        pytest.skip("no nvcc")
    elig, off, wl, wb, code3, budget = band_cases()[case]
    rank = np.where(elig, np.cumsum(elig) - 1, 0xFFFFFFFF)
    got = band(rank, off, wl, wb, code3, budget)
    tiles = [tuple(t) for t in got["tiles"]]
    a, b = LD.window_pairs(elig, off, wl, wb)
    want = sorted(set(zip((a // 256).tolist(), (b // 256).tolist())))
    assert tiles == want                  # every in-window pair is in a listed tile, and every listed tile holds one
    assert all(i <= j for i, j in tiles) and tiles == sorted(set(tiles))   # I <= J, ascending, no repeats
    sb = got["slab_begin"]
    assert sb[0] == 0 and sb[-1] == len(tiles)
    blocks = np.asarray(got["tile_blocks"], dtype=np.int64)
    assert np.array_equal(blocks, [(4 if i == j else 6) if code3 else 1 for i, j in tiles])
    for s0, s1 in zip(sb, sb[1:]):
        assert s1 > s0
        assert s1 - s0 == 1 or blocks[s0:s1].sum() * got["block_bytes"] <= budget      # a slab holds at least one tile


def test_band_slabs_cut_where_the_budget_says():
    """Diagonal band of 40 blocks, window of 2 loci: 40 diagonal tiles and 39 off-diagonal ones (loci 255 / 256 of each block
    boundary). With code-3 cells they cost 4 and 6 blocks; a budget of 10 blocks takes one pair of them per slab."""
    try:
        plan_probe.probe_binary("ld_band_probe")
    except FileNotFoundError:
        pytest.skip("no nvcc")
    l = 40 * 256
    got = band(np.arange(l), np.arange(l), 2, 0, True, 10 << 18)
    assert len(got["tiles"]) == 79
    assert got["slab_begin"] == list(range(0, 79, 2)) + [79]
    got = band(np.arange(l), np.arange(l), 2, 0, False, 10 << 18)
    assert got["slab_begin"] == list(range(0, 79, 10)) + [79]


def test_structs_match_the_header():
    from kgl_gene_b200 import capi
    assert C.sizeof(capi.LdOptions) == 16
    assert [getattr(capi.LdOptions, f).offset for f in ("keep", "window_loci", "window_bp")] == [0, 8, 12]
    assert capi.LD_PAIR_DTYPE.itemsize == 24 and C.sizeof(capi.LdPair) == 24
    assert capi.LD_PAIR_DTYPE.names == ("a", "b", "n_valid", "reserved", "r2") and capi.LD_PAIR_DTYPE.fields["r2"][1] == 16
    assert np.dtype(LD.PAIR_FIELDS) == capi.LD_PAIR_DTYPE
