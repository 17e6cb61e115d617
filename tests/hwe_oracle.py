"""Hardy-Weinberg equilibrium and variant QC restated on the host. TEST INFRASTRUCTURE ONLY (never imported by kgl_gene_b200/).

exact() restates the contract of include/kgl_b200.h in Python floats, which are IEEE doubles rounded to nearest one operation at a
time: every term of the support from the mode, in the stated order, and no early stop. Every integer is formed exactly and converted
once, as the device converts it, so p, mid-p and F are bit-equal to the device's. early_stop() replays the device's stopping rule on
the same terms (hwe.cuh), so the CPU suite can show that the terms it skips change neither sum. walk_terms() counts the terms a full
walk computes (the pre-walk to P(obs) plus the support), for the load-balance figures."""
from __future__ import annotations

import math

import numpy as np

TIE = 1.0 + 2.0 ** -40
ABSORB = 2.0 ** -54
NAN = float("nan")


def rare_common(n0: int, n1: int, n2: int):
    v = n0 + n1 + n2
    nr = min(n1 + 2 * n2, n1 + 2 * n0)
    return v, nr, 2 * v - nr


def mode(nr: int, nc: int, v: int) -> int:
    m = nr * nc // (2 * v)
    if (m ^ nr) & 1:
        m += 1
    return m


def terms(nr: int, nc: int, v: int):
    """(m, below, above): P(m) = 1.0, below = [P(m-2), P(m-4), ..], above = [P(m+2), ..], each from the one before."""
    m = mode(nr, nc, v)
    below, t, h = [], 1.0, m
    while h >= 2:
        r, c = (nr - h) // 2, (nc - h) // 2
        t = (t * float(h * (h - 1))) / float(4 * (r + 1) * (c + 1))
        below.append(t)
        h -= 2
    above, t, h = [], 1.0, m
    while h + 2 <= nr:
        r, c = (nr - h) // 2, (nc - h) // 2
        t = (t * float(4 * r * c)) / float((h + 2) * (h + 1))
        above.append(t)
        h += 2
    return m, below, above


def p_obs(m: int, below, above, n1: int) -> float:
    if n1 == m:
        return 1.0
    return below[(m - n1) // 2 - 1] if n1 < m else above[(n1 - m) // 2 - 1]


def exact(n0: int, n1: int, n2: int, midp: bool = False) -> float:
    """The exact test's p (or mid-p) of one group's counts."""
    v, nr, nc = rare_common(n0, n1, n2)
    if v == 0:
        return NAN
    if nr == 0:
        return 1.0
    m, below, above = terms(nr, nc, v)
    po = p_obs(m, below, above, n1)
    thr = po * TIE
    s, n = 1.0, (1.0 if 1.0 <= thr else 0.0)
    for t in below + above:
        s = s + t
        if t <= thr:
            n = n + t
    return (n - 0.5 * po) / s if midp else n / s


def f_stat(n0: int, n1: int, n2: int) -> float:
    v = n0 + n1 + n2
    s = n1 + 2 * n2
    if v == 0 or s == 0 or s == 2 * v:
        return NAN
    return 1.0 - float(2 * v * n1) / float(s * (2 * v - s))


def early_stop(n0: int, n1: int, n2: int):
    """(S, N, terms walked) under the device's rule: a side stops once its next exact ratio is below 1 and the current term is
    below 2^-54 of both sums (or 0); the pre-walk to P(obs) stops at 0. Bit-equal to the full sums when the rule is exact."""
    v, nr, nc = rare_common(n0, n1, n2)
    if v == 0 or nr == 0:
        return 1.0, 1.0, 0
    m, below, above = terms(nr, nc, v)
    walked = 0
    po, step = 1.0, (below if n1 < m else above)
    for i in range(abs(m - n1) // 2):
        po = step[i]
        walked += 1
        if po == 0.0:
            break
    if po == 0.0:
        return 1.0, 0.0, walked
    thr = po * TIE
    s, n = 1.0, (1.0 if 1.0 <= thr else 0.0)
    for side, sign in ((below, -1), (above, 1)):
        t, h = 1.0, m
        for nxt in side:
            r, c = (nr - h) // 2, (nc - h) // 2
            a, b = (h * (h - 1), 4 * (r + 1) * (c + 1)) if sign < 0 else (4 * r * c, (h + 2) * (h + 1))
            if a < b and s * ABSORB > t and n * ABSORB > t:
                break
            t = nxt
            walked += 1
            s = s + t
            if t <= thr:
                n = n + t
            h += 2 * sign
            if t == 0.0:
                break
    return s, n, walked


def walk_terms(n0, n1, n2):
    """Terms a full walk computes, vectorised: |obs - m| / 2 to reach P(obs), then every term of the support but the mode."""
    n0, n1, n2 = (np.asarray(x, dtype=np.int64) for x in (n0, n1, n2))
    v = n0 + n1 + n2
    nr = np.minimum(n1 + 2 * n2, n1 + 2 * n0)
    nc = 2 * v - nr
    m = np.where(v > 0, nr * nc // np.maximum(2 * v, 1), 0)
    m = m + ((m ^ nr) & 1)
    return np.where((v > 0) & (nr > 0), np.abs(m - n1) // 2 + nr // 2, 0)


def lane_efficiency(work, order=None, warp: int = 32) -> float:
    """Useful lane-steps over issued lane-steps when consecutive cells of `order` share a warp that runs as long as its longest."""
    w = np.asarray(work, dtype=np.float64).ravel()
    if order is not None:
        w = w[order]
    pad = (-w.size) % warp
    w = np.concatenate([w, np.zeros(pad)]).reshape(-1, warp)
    issued = w.max(axis=1).sum() * warp
    return float(w.sum() / issued) if issued else 1.0


def length_order(counts: np.ndarray, multi=None) -> np.ndarray:
    """The device's cell order: by bit length of n_r, longest first, stable (k_hwe_keys + one radix pass)."""
    c = np.asarray(counts).reshape(-1, 4).astype(np.int64)
    v = c[:, 0] + c[:, 1] + c[:, 2]
    nr = np.minimum(c[:, 1] + 2 * c[:, 2], c[:, 1] + 2 * c[:, 0])
    if multi is not None:
        g = np.asarray(counts).shape[1]
        nr = np.where(np.repeat(np.asarray(multi, dtype=bool), g), 0, nr)
    nr = np.where(v > 0, nr, 0)
    bits = np.zeros(nr.shape, dtype=np.int64)
    nz = nr > 0
    bits[nz] = np.floor(np.log2(nr[nz])).astype(np.int64) + 1
    return np.argsort(31 - bits, kind="stable")


def hardy(counts: np.ndarray, multi_rows=None, midp: bool = False):
    """(p, f) float64[L][G] from group counts uint32[L][G][4]; NaN on the multi-allelic rows."""
    counts = np.asarray(counts)
    l, g = counts.shape[:2]
    p = np.full((l, g), np.nan)
    f = np.full((l, g), np.nan)
    multi = np.zeros(l, dtype=bool)
    if multi_rows is not None:
        multi[np.asarray(multi_rows, dtype=np.int64)] = True
    cache = {}
    for i in range(l):
        if multi[i]:
            continue
        for k in range(g):
            key = (int(counts[i, k, 0]), int(counts[i, k, 1]), int(counts[i, k, 2]))
            if key not in cache:
                cache[key] = (exact(*key, midp=midp), f_stat(*key))
            p[i, k], f[i, k] = cache[key]
    return p, f


def variant_qc(pooled: np.ndarray, n_genomes: int, p=None, keep=None, multi_rows=None, min_call_rate=0.0, min_maf=0.0, min_hwe_p=0.0):
    """The QC rule of include/kgl_b200.h in numpy: (keep uint8[L], n_kept) from the raw counts uint32[L][4] over all genomes."""
    c = np.asarray(pooled).astype(np.int64)
    ok = np.ones(c.shape[0], dtype=bool) if keep is None else np.asarray(keep) != 0
    if multi_rows is not None:
        ok[np.asarray(multi_rows, dtype=np.int64)] = False
    with np.errstate(divide="ignore", invalid="ignore"):
        if min_call_rate:
            ok &= (n_genomes - c[:, 3]).astype(np.float64) / float(n_genomes) >= min_call_rate
        if min_maf:
            v2 = 2 * (c[:, 0] + c[:, 1] + c[:, 2])
            s = c[:, 1] + 2 * c[:, 2]
            ok &= (v2 > 0) & (np.minimum(s, v2 - s).astype(np.float64) / v2.astype(np.float64) >= min_maf)
        if min_hwe_p:
            ok &= ~(np.asarray(p) < min_hwe_p).any(axis=1)
    return ok.astype(np.uint8), int(ok.sum())


def exact_fraction(n0: int, n1: int, n2: int, midp: bool = False):
    """(p as a Fraction, the exact qualifying set) from exact probabilities: P(h) = n! / (r! h! c!) 2^h / C(2n, n_r) up to a factor."""
    from fractions import Fraction
    v, nr, nc = rare_common(n0, n1, n2)
    w = {}
    for h in range(nr % 2, nr + 1, 2):
        r, c = (nr - h) // 2, (nc - h) // 2
        w[h] = Fraction(math.factorial(v) * 2 ** h, math.factorial(r) * math.factorial(h) * math.factorial(c))
    po = w[n1]
    q = {h for h, x in w.items() if x <= po}
    tot = sum(w.values())
    num = sum(w[h] for h in q)
    if midp:
        num -= po / 2
    return num / tot, q


def float_qualifying(n0: int, n1: int, n2: int):
    """The heterozygote counts whose float term qualifies for N."""
    v, nr, nc = rare_common(n0, n1, n2)
    m, below, above = terms(nr, nc, v)
    thr = p_obs(m, below, above, n1) * TIE
    q = {m} if 1.0 <= thr else set()
    q |= {m - 2 * (i + 1) for i, t in enumerate(below) if t <= thr}
    q |= {m + 2 * (i + 1) for i, t in enumerate(above) if t <= thr}
    return q
