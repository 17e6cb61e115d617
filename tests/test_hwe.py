"""Hardy-Weinberg contract on the CPU: the float restatement (tests/hwe_oracle.py) against exact rationals for every genotype count
with v <= 40 and against 200-bit mpmath at up to 2 x 10^5 allele copies; p <= 1 and p == 1.0 exactly when every term qualifies;
the early stop of the device walk leaves both sums unchanged bit for bit; the QC rule; the layout of the two option structs."""
import ctypes as C
import math
import random

import numpy as np
import pytest

import hwe_oracle as HO


def all_counts(max_v):
    for v in range(1, max_v + 1):
        for n1 in range(v + 1):
            for n2 in range(v - n1 + 1):
                yield v - n1 - n2, n1, n2


def test_exact_rationals_up_to_40_genomes():
    """The tie margin makes the float qualifying set the exact one (ties included), and p / mid-p agree to 1e-13 relative."""
    worst = 0.0
    for n0, n1, n2 in all_counts(40):
        pf, q = HO.exact_fraction(n0, n1, n2)
        assert HO.float_qualifying(n0, n1, n2) == q, (n0, n1, n2)
        for midp in (False, True):
            want = float(HO.exact_fraction(n0, n1, n2, midp)[0]) if midp else float(pf)
            got = HO.exact(n0, n1, n2, midp)
            if HO.rare_common(n0, n1, n2)[1] == 0:
                assert got == 1.0
                continue
            assert 0.0 <= got <= 1.0
            worst = max(worst, abs(got - want) / want)
    assert worst < 1e-13, worst


def test_exact_ties_exist_and_count():
    """Exact ties occur (symmetric supports, e.g. equal allele counts); the tied terms count for N."""
    ties = 0
    for n0, n1, n2 in all_counts(20):
        pf, q = HO.exact_fraction(n0, n1, n2)
        v, nr, nc = HO.rare_common(n0, n1, n2)
        if nr == 0:
            continue
        m, below, above = HO.terms(nr, nc, v)
        po = HO.p_obs(m, below, above, n1)
        ties += sum(1 for h in q if h != n1 and (h == m and po == 1.0 or h != m and HO.p_obs(m, below, above, h) == po))
    assert ties > 0


def test_rounding_tie_needs_the_margin():
    """At 188 genomes with 30 heterozygotes and 3 rare homozygotes an exact tie lands, after rounding, just above P(obs): only
    the 2^-40 margin keeps it in N, as the exact rationals do. The only such counts up to 200 genomes."""
    for c in ((155, 30, 3), (3, 30, 155)):
        q = HO.exact_fraction(*c)[1]
        assert HO.float_qualifying(*c) == q
        v, nr, nc = HO.rare_common(*c)
        m, below, above = HO.terms(nr, nc, v)
        po = HO.p_obs(m, below, above, c[1])
        assert any(po < t <= po * HO.TIE for t in below + above)


def mp_p(n0, n1, n2, midp=False):
    import mpmath
    mpmath.mp.prec = 200
    v, nr, nc = HO.rare_common(n0, n1, n2)
    m = HO.mode(nr, nc, v)
    t = {m: mpmath.mpf(1)}
    h, x = m, mpmath.mpf(1)
    while h >= 2:
        r, c = (nr - h) // 2, (nc - h) // 2
        x = x * (h * (h - 1)) / (4 * (r + 1) * (c + 1))
        h -= 2
        t[h] = x
    h, x = m, mpmath.mpf(1)
    while h + 2 <= nr:
        r, c = (nr - h) // 2, (nc - h) // 2
        x = x * (4 * r * c) / ((h + 2) * (h + 1))
        h += 2
        t[h] = x
    po = t[n1]
    thr = po * (1 + mpmath.mpf(2) ** -40)
    s = mpmath.fsum(t.values())
    n = mpmath.fsum(x for x in t.values() if x <= thr)
    return (n - po / 2) / s if midp else n / s


@pytest.mark.parametrize("v,frac_het,p_alt", [
    (100_000, 0.5, 0.5), (100_000, 0.45, 0.5), (100_000, 0.52, 0.5), (100_000, 0.18, 0.1), (100_000, 0.17, 0.1),
    (100_000, 0.0199, 0.01), (50_000, 0.002, 0.001), (2504, 0.42, 0.3), (2504, 0.3, 0.3), (20_000, 0.2, 0.2),
])
def test_against_mpmath_at_large_v(v, frac_het, p_alt):
    n1 = int(v * frac_het)
    n2 = int(round(v * p_alt * p_alt))
    n0 = v - n1 - n2
    for midp in (False, True):
        want = mp_p(n0, n1, n2, midp)
        got = HO.exact(n0, n1, n2, midp)
        assert 0.0 <= got <= 1.0
        if want > 1e-300:
            assert abs(got - float(want)) <= 1e-12 * float(want), (n0, n1, n2, midp, got, float(want))


def test_p_at_most_one_and_one_when_all_qualify():
    rng = random.Random(5)
    cases = list(all_counts(12))
    for _ in range(300):
        v = rng.randint(1, 30_000)
        n1 = rng.randint(0, v)
        n2 = rng.randint(0, v - n1)
        cases.append((v - n1 - n2, n1, n2))
    for n0, n1, n2 in cases:
        v, nr, nc = HO.rare_common(n0, n1, n2)
        p = HO.exact(n0, n1, n2)
        assert p <= 1.0 and HO.exact(n0, n1, n2, True) <= 1.0
        if nr == 0:
            assert p == 1.0
            continue
        m, below, above = HO.terms(nr, nc, v)
        if len(HO.float_qualifying(n0, n1, n2)) == len(below) + len(above) + 1:
            assert p == 1.0, (n0, n1, n2)


def test_monomorphic_and_empty():
    assert HO.exact(50, 0, 0) == 1.0 and HO.exact(0, 0, 50) == 1.0 and HO.exact(0, 0, 50, True) == 1.0
    assert math.isnan(HO.exact(0, 0, 0)) and math.isnan(HO.f_stat(0, 0, 0))
    assert math.isnan(HO.f_stat(10, 0, 0)) and math.isnan(HO.f_stat(0, 0, 10))
    assert HO.f_stat(0, 10, 0) == -1.0                  # all heterozygous: H_obs = 1, H_exp = 1/2
    assert HO.f_stat(5, 0, 5) == 1.0                    # no heterozygote
    assert HO.f_stat(25, 50, 25) == 1.0 - 10000.0 / 10000.0


def test_underflow_floor():
    """All heterozygous at 5,000 genomes: P(obs) underflows relative to the mode, p and mid-p are exactly 0."""
    assert HO.exact(0, 5000, 0) == 0.0 and HO.exact(0, 5000, 0, True) == 0.0
    s, n, _ = HO.early_stop(0, 5000, 0)
    assert n == 0.0


def early_stop_cases():
    rng = random.Random(11)
    cases = [(0, 5000, 0), (2500, 0, 2500), (25_000, 50_000, 25_000), (49_000, 2_000, 49_000), (30_000, 40_000, 30_000),
             (0, 2, 99_998), (1, 99_998, 1), (99_000, 1_000, 0), (4_000, 2, 996_000 // 1000), (60, 40, 0), (1, 1, 1)]
    # observations far out in one tail: the other tail's terms join S only for a while, then must still reach N
    for v in (2504, 20_000, 100_000):
        for frac in (0.3, 0.45, 0.49, 0.55, 0.7):
            n1 = int(v * frac)
            n2 = (v - n1) // 2
            cases.append((v - n1 - n2, n1, n2))
    for _ in range(200):
        v = rng.choice([rng.randint(1, 200), rng.randint(200, 5000), rng.randint(5000, 60_000)])
        n1 = rng.randint(0, v)
        n2 = rng.randint(0, v - n1)
        cases.append((v - n1 - n2, n1, n2))
    return cases


def test_early_stop_is_exact():
    """The device's stopping rule skips only terms that change neither sum: S and N equal the full sums bit for bit."""
    skipped = 0
    for n0, n1, n2 in early_stop_cases():
        v, nr, nc = HO.rare_common(n0, n1, n2)
        if nr == 0:
            continue
        m, below, above = HO.terms(nr, nc, v)
        po = HO.p_obs(m, below, above, n1)
        thr = po * HO.TIE
        s, n = 1.0, (1.0 if 1.0 <= thr else 0.0)
        for t in below + above:
            s += t
            if t <= thr:
                n += t
        es, en, walked = HO.early_stop(n0, n1, n2)
        if po == 0.0:
            assert en == 0.0 and n == 0.0
            continue
        assert (es, en) == (s, n), (n0, n1, n2)
        skipped += int(HO.walk_terms(n0, n1, n2)) - walked
    assert skipped > 100_000


def test_stop_against_s_alone_would_be_wrong():
    """A case that needs the N half of the rule: stopping a side on S alone loses the small qualifying terms of the other tail."""
    n0, n1, n2 = 25_925, 48_150, 25_925        # het deficit 1,850 below the mode (m = 50,000): P(obs) ~ 1.8e-30
    v, nr, nc = HO.rare_common(n0, n1, n2)
    m, below, above = HO.terms(nr, nc, v)
    thr = HO.p_obs(m, below, above, n1) * HO.TIE
    n_full = sum(t for t in below + above if t <= thr)
    s = 1.0 + sum(below)
    n_s_only = 0.0
    for t in below:
        if t <= thr:
            n_s_only += t
    for t in above:                             # stop where t < 2^-54 S without looking at N
        if t < s * HO.ABSORB:
            break
        s += t
        if t <= thr:
            n_s_only += t
    assert n_full > 0.0 and n_s_only != n_full


def test_walk_terms_and_lane_efficiency():
    rng = np.random.default_rng(3)
    n = 2504
    p = rng.beta(0.2, 2.0, size=4000)
    n1 = rng.binomial(n, 2 * p * (1 - p))
    n2 = rng.binomial(n - n1, np.clip(p * p / np.maximum(1 - 2 * p * (1 - p), 1e-12), 0, 1))
    counts = np.stack([n - n1 - n2, n1, n2, np.zeros_like(n1)], axis=1).reshape(-1, 1, 4)
    work = HO.walk_terms(counts[:, 0, 0], counts[:, 0, 1], counts[:, 0, 2])
    for i in range(0, 4000, 397):
        v, nr, nc = HO.rare_common(*map(int, counts[i, 0, :3]))
        if nr:
            m, b, a = HO.terms(nr, nc, v)
            assert work[i] == abs(m - int(counts[i, 0, 1])) // 2 + len(b) + len(a)
    order = HO.length_order(counts)
    assert HO.lane_efficiency(work, order) > HO.lane_efficiency(work)


def test_variant_qc_rule():
    pooled = np.array([[10, 0, 0, 0],       # monomorphic: MAF 0
                       [5, 4, 1, 0],        # MAF 0.3
                       [5, 4, 1, 10],       # call rate 0.5
                       [0, 0, 0, 20],       # no call
                       [8, 2, 0, 0]], dtype=np.uint32)   # MAF 0.1
    n = 20
    p = np.array([[1.0, np.nan], [0.5, 0.2], [1e-7, 0.9], [np.nan, np.nan], [0.01, np.nan]])
    k, m = HO.variant_qc(pooled, n, p)
    assert m == 5 and k.tolist() == [1] * 5
    assert HO.variant_qc(pooled, n, p, min_maf=0.1)[0].tolist() == [0, 1, 1, 0, 1]
    assert HO.variant_qc(pooled, n, p, min_call_rate=0.5)[0].tolist() == [1, 1, 1, 0, 1]        # 10 of 20 called: 0.5 passes
    assert HO.variant_qc(pooled, n, p, min_call_rate=0.6)[0].tolist() == [1, 1, 0, 0, 1]
    assert HO.variant_qc(pooled, n, p, min_hwe_p=1e-6)[0].tolist() == [1, 1, 0, 1, 1]
    assert HO.variant_qc(pooled, n, p, min_hwe_p=0.3)[0].tolist() == [1, 0, 0, 1, 0]
    assert HO.variant_qc(pooled, n, p, keep=[1, 1, 1, 1, 0], multi_rows=[1])[0].tolist() == [1, 0, 1, 1, 0]


def test_option_struct_layout():
    from kgl_gene_b200 import capi
    assert C.sizeof(capi.HardyOptions) == 16
    assert C.sizeof(capi.QcOptions) == 48
    assert capi.QcOptions.min_call_rate.offset == 8 and capi.QcOptions.group.offset == 32 and capi.QcOptions.midp.offset == 44
