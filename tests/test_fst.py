"""Population differentiation on the host: the F_ST oracle (tests/fst_oracle.py) against an independent per-locus implementation
written from the papers' formulas, a hand-computed Weir & Cockerham example, the limits of Hudson's estimator, the window
boundaries, and the layout of kgl_b200_fst_options."""
import ctypes as C
import os
import re
from fractions import Fraction

import numpy as np
import pytest

import fst_oracle as FO
from conftest import ROOT


def hudson_paper(n_a, n_b):
    """Hudson et al. 1992 / Bhatia et al. 2013 eq. 10 for one locus: n_x = (ref, alt) allele counts of each population."""
    na, nb = n_a[0] + n_a[1], n_b[0] + n_b[1]
    pa, pb = n_a[1] / na, n_b[1] / nb
    num = (pa - pb) ** 2 - pa * (1 - pa) / (na - 1) - pb * (1 - pb) / (nb - 1)
    den = pa * (1 - pb) + pb * (1 - pa)
    return num, den


def wc_paper(g, allele=1):
    """Weir & Cockerham 1984 eqs. 2-4 for one locus and one allele, r populations: g[i] = (n0, n1, n2) genotype counts of
    population i (called individuals only). Returns (a, b, c)."""
    g = np.asarray(g, dtype=np.float64)
    r = len(g)
    n = g.sum(axis=1)
    alt = (g[:, 1] + 2 * g[:, 2]) / (2 * n)
    p = alt if allele == 1 else 1 - alt
    h = g[:, 1] / n                                   # heterozygotes carry one copy of either allele
    n_bar = n.sum() / r
    n_c = (r * n_bar - (n ** 2).sum() / (r * n_bar)) / (r - 1)
    p_bar = (n * p).sum() / (r * n_bar)
    s2 = (n * (p - p_bar) ** 2).sum() / ((r - 1) * n_bar)
    h_bar = (n * h).sum() / (r * n_bar)
    a = n_bar / n_c * (s2 - 1 / (n_bar - 1) * (p_bar * (1 - p_bar) - (r - 1) / r * s2 - h_bar / 4))
    b = n_bar / (n_bar - 1) * (p_bar * (1 - p_bar) - (r - 1) / r * s2 - (2 * n_bar - 1) / (4 * n_bar) * h_bar)
    c = h_bar / 2
    return a, b, c


def random_counts(rng, l, n_groups, n_max=40):
    counts = np.zeros((l, n_groups, 4), dtype=np.uint32)
    for k in range(n_groups):
        n = rng.integers(0, n_max, size=l)
        p = rng.random(l)
        counts[:, k, 2] = rng.binomial(n, p * p)
        counts[:, k, 1] = rng.binomial(n - counts[:, k, 2], np.clip(2 * p * (1 - p) / np.maximum(1 - p * p, 1e-9), 0, 1))
        counts[:, k, 3] = rng.binomial(n - counts[:, k, 2] - counts[:, k, 1], 0.05)
        counts[:, k, 0] = n - counts[:, k, 1] - counts[:, k, 2] - counts[:, k, 3]
    counts[::37] = 0                                   # all missing / empty
    counts[5::41, :, 1:3] = 0                          # monomorphic
    return counts


@pytest.mark.parametrize("method", ["hudson", "weir_cockerham"])
def test_oracle_matches_the_papers(method):
    rng = np.random.default_rng(1)
    counts = random_counts(rng, 3000, 3)
    keep = (rng.random(3000) < 0.9).astype(np.uint8)
    for a, b in FO.all_pairs(3):
        num, den, ok = FO.terms(counts, int(a), int(b), method, keep)
        want_num, want_den = np.zeros(3000), np.zeros(3000)
        want_ok = np.zeros(3000, dtype=bool)
        for l in range(3000):
            ca, cb = counts[l, a].astype(np.int64), counts[l, b].astype(np.int64)
            va, vb = ca[:3].sum(), cb[:3].sum()
            if not keep[l] or va < 1 or vb < 1:
                continue
            if method == "hudson":
                x, y = hudson_paper((2 * ca[0] + ca[1], ca[1] + 2 * ca[2]), (2 * cb[0] + cb[1], cb[1] + 2 * cb[2]))
            else:
                if va + vb < 3:
                    continue
                aa, bb, cc = wc_paper([ca[:3], cb[:3]])
                assert np.allclose(wc_paper([ca[:3], cb[:3]], allele=0), (aa, bb, cc), rtol=1e-12, atol=1e-15)
                x, y = aa, aa + bb + cc
            if y == 0:
                continue
            want_num[l], want_den[l], want_ok[l] = x, y, True
        assert np.array_equal(ok, want_ok)
        assert np.allclose(num, want_num, rtol=1e-12, atol=1e-14)
        assert np.allclose(den, want_den, rtol=1e-12, atol=1e-14)
        f = FO.fst(counts, [(a, b)], method, keep)[0]
        assert abs(f - want_num.sum() / want_den.sum()) <= 1e-12 * max(1.0, abs(f))


def test_weir_cockerham_hand_example():
    # group a: 2 hom-ref, 2 het, 1 hom-alt (p = 0.4, h = 0.4); group b: 0, 2, 3 (p = 0.8, h = 0.4). By hand: n_bar = 5,
    # n_c = 2*25/10 = 5, p_bar = 12/20 = 0.6, s2 = (5*0.04 + 5*0.04)/5 = 0.08, h_bar = 0.4, p_bar(1 - p_bar) = 0.24;
    # a = (5/5)(0.08 - (0.24 - 0.04 - 0.1)/4) = 0.055, b = (5/4)(0.24 - 0.04 - (9/20) 0.4) = 0.025, c = 0.2.
    a, b, c = Fraction(11, 200), Fraction(1, 40), Fraction(1, 5)
    counts = np.array([[[2, 2, 1, 0], [0, 2, 3, 7]]], dtype=np.uint32)      # code-3 cells are missing: they change nothing
    num, den, ok = FO.terms(counts, 0, 1, "weir_cockerham")
    assert ok[0]
    assert abs(num[0] - float(a)) < 1e-15 and abs(den[0] - float(a + b + c)) < 1e-15
    assert abs(FO.fst(counts, [(0, 1)], "weir_cockerham")[0] - float(a / (a + b + c))) < 1e-15
    assert np.allclose(wc_paper([[2, 2, 1], [0, 2, 3]]), (float(a), float(b), float(c)), rtol=1e-13)


def test_hudson_limits():
    rng = np.random.default_rng(2)
    l, n = 4000, 400
    p = rng.uniform(0.05, 0.95, size=l)
    dosage = rng.binomial(2, p[:, None], size=(l, 2 * n)).astype(np.uint8)
    group = np.repeat([0, 1], n).astype(np.uint8)
    counts = FO.group_counts(dosage, group, 2)
    f = FO.fst(counts, [(0, 1)], "hudson")[0]
    assert abs(f) < 2e-3, f                                  # one frequency: unbiased, near 0
    fixed = np.zeros((50, 2 * n), dtype=np.uint8)
    fixed[:, n:] = 2                                          # a fixed difference at every locus
    counts = FO.group_counts(fixed, group, 2)
    assert FO.fst(counts, [(0, 1)], "hudson")[0] == 1.0
    assert FO.fst(counts, [(0, 1)], "weir_cockerham")[0] > 0.99
    mono = np.zeros((20, 2 * n), dtype=np.uint8)              # monomorphic across both groups: no locus used
    assert np.isnan(FO.fst(FO.group_counts(mono, group, 2), [(0, 1)], "hudson")[0])


def test_summation_order_is_a_tree_then_blocks():
    rng = np.random.default_rng(3)
    x = rng.standard_normal(1000) * 10.0 ** rng.integers(-8, 8, size=1000)
    blocks = FO.tree_blocks(x)
    assert len(blocks) == 4
    for b in range(4):
        v = np.zeros(256)
        seg = x[256 * b: 256 * (b + 1)]
        v[: len(seg)] = seg
        s = 128
        while s:
            for i in range(s):
                v[i] = v[i] + v[i + s]
            s //= 2
        assert v[0] == blocks[b]
    total = 0.0
    for v in blocks:
        total += v
    assert FO.fold(blocks) == total


@pytest.mark.parametrize("window,step", [(100, 0), (100, 50), (100, 30), (7, 7), (1000, 1000)])
def test_window_boundaries(window, step):
    rng = np.random.default_rng(window + step)
    off = np.sort(rng.choice(np.arange(1, 600), size=120, replace=False)).astype(np.int64)
    st = step or window
    off = np.union1d(off, [st + window, 2 * st + window - 1, 3 * st])   # a locus exactly at w step + window, one just inside
    begin, end = FO.window_rows(off, window, step)
    assert len(begin) == off.max() // st + 1
    for w in range(len(begin)):
        inside = np.flatnonzero((off >= w * st) & (off < w * st + window))
        assert list(range(begin[w], end[w])) == list(inside)
    w = 1
    assert np.flatnonzero(off == st + window)[0] == end[w]          # excluded from window 1, which ends there


def test_windows_oracle_against_direct_sums():
    rng = np.random.default_rng(4)
    counts = random_counts(rng, 500, 2)
    off = np.sort(rng.choice(np.arange(0, 5000), size=500, replace=False))
    got = FO.windows(counts, [(0, 1)], "hudson", off, 400, 150)
    num, den, ok = FO.terms(counts, 0, 1, "hudson")
    for w in range(got.shape[1]):
        sel = ok & (off >= 150 * w) & (off < 150 * w + 400)
        assert got[0, w, 2] == sel.sum()
        assert np.isclose(got[0, w, 0], num[sel].sum(), rtol=1e-12, atol=1e-15)
        assert np.isclose(got[0, w, 1], den[sel].sum(), rtol=1e-12, atol=1e-15)


def test_fst_options_layout():
    from kgl_gene_b200 import capi
    O = capi.FstOptions
    assert C.sizeof(O) == 56
    assert [(f, getattr(O, f).offset) for f, _ in O._fields_] == [
        ("group", 0), ("n_groups", 8), ("keep", 16), ("method", 24), ("n_pairs", 28), ("pairs", 32), ("window_bp", 40), ("step_bp", 48)]
    header = open(os.path.join(ROOT, "include", "kgl_b200.h")).read()
    assert re.search(r"typedef struct kgl_b200_fst_options \{\s*/\* zero-initialise; 56 bytes \*/", header)
    assert "#define KGL_B200_FST_HUDSON 0" in header and "#define KGL_B200_FST_WEIR_COCKERHAM 1" in header
    assert capi.FST_METHODS == {"hudson": 0, "weir_cockerham": 1}
