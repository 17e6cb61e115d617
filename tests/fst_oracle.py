"""Population differentiation restated on the host. TEST INFRASTRUCTURE ONLY (never imported by kgl_gene_b200/).

group_counts is a bincount of the codes per (locus, group). terms restates fst_term (kgl_gene_b200/csrc/fst.cuh) operation for
operation: numpy float64 arithmetic is IEEE round-to-nearest, one operation at a time (numpy never fuses a multiply and an add),
and the integer inputs are converted exactly as the device converts them, so the terms are bit-equal to the device's. fst and
windows restate the summation order of include/kgl_b200.h: blocks of 256 loci summed as a halving tree, then the block sums in
order from 0.0; a window adds its used loci in row order from 0.0."""
from __future__ import annotations

import numpy as np

BLOCK = 256


def group_counts(codes: np.ndarray, group, n_groups: int) -> np.ndarray:
    """uint32[L][G][4]: genomes of group k with code c at locus l; label 0xFF = in no group."""
    codes = np.asarray(codes)
    group = np.asarray(group)
    l = codes.shape[0]
    out = np.zeros((l, n_groups, 4), dtype=np.uint32)
    for k in range(n_groups):
        sub = codes[:, group == k]
        for c in range(4):
            out[:, k, c] = (sub == c).sum(axis=1)
    return out


def all_pairs(n_groups: int) -> np.ndarray:
    return np.array([(a, b) for a in range(n_groups) for b in range(a + 1, n_groups)], dtype=np.uint32).reshape(-1, 2)


def terms(counts: np.ndarray, a: int, b: int, method: str, keep=None):
    """(num, den, used) float64[L], float64[L], bool[L] of the pair (a, b); (0, 0) where not used."""
    ca = counts[:, a, :].astype(np.uint64)
    cb = counts[:, b, :].astype(np.uint64)
    va, vb = ca[:, 0] + ca[:, 1] + ca[:, 2], cb[:, 0] + cb[:, 1] + cb[:, 2]
    sa, sb = ca[:, 1] + 2 * ca[:, 2], cb[:, 1] + 2 * cb[:, 2]
    ok = (va >= 1) & (vb >= 1)
    if keep is not None:
        ok &= np.asarray(keep) != 0
    f = np.float64
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        if method == "hudson":
            pa = sa.astype(f) / (2 * va).astype(f)
            pb = sb.astype(f) / (2 * vb).astype(f)
            d = pa - pb
            ta = (pa * (1.0 - pa)) / (2 * va - 1).astype(f)
            tb = (pb * (1.0 - pb)) / (2 * vb - 1).astype(f)
            num = ((d * d) - ta) - tb
            den = (pa * (1.0 - pb)) + (pb * (1.0 - pa))
        elif method == "weir_cockerham":
            ok &= (va + vb) >= 3
            na, nb, nt = va.astype(f), vb.astype(f), (va + vb).astype(f)
            nbar = nt * 0.5
            nc = ((va * vb).astype(f) * 2.0) / nt
            pa = sa.astype(f) / (na * 2.0)
            pb = sb.astype(f) / (nb * 2.0)
            pbar = (sa + sb).astype(f) / (nt * 2.0)
            da, db = pa - pbar, pb - pbar
            s2 = ((na * (da * da)) + (nb * (db * db))) / nbar
            hbar = (ca[:, 1] + cb[:, 1]).astype(f) / nt
            pq = pbar * (1.0 - pbar)
            nbar1 = nbar - 1.0
            inner = (pq - (s2 * 0.5)) - (hbar * 0.25)
            aa = (nbar / nc) * (s2 - (inner / nbar1))
            q = ((nbar * 2.0) - 1.0) / (nbar * 4.0)
            bb = (nbar / nbar1) * ((pq - (s2 * 0.5)) - (q * hbar))
            cc = hbar * 0.5
            num = aa
            den = (aa + bb) + cc
        else:
            raise ValueError(method)
    ok &= den != 0.0
    num = np.where(ok, num, 0.0)
    den = np.where(ok, den, 0.0)
    return num, den, ok


def fold(x: np.ndarray) -> float:
    """x[0] + x[1] + ... added in order from 0.0."""
    return float(np.add.accumulate(np.concatenate([[0.0], np.asarray(x, dtype=np.float64)]))[-1])


def tree_blocks(x: np.ndarray) -> np.ndarray:
    """Per block of 256: the halving tree (element i += element i + s for s = 128 .. 1), 0.0 past the end."""
    nb = (len(x) + BLOCK - 1) // BLOCK
    a = np.zeros(nb * BLOCK, dtype=np.float64)
    a[: len(x)] = x
    a = a.reshape(nb, BLOCK)
    s = BLOCK // 2
    while s:
        a[:, :s] = a[:, :s] + a[:, s:2 * s]
        s //= 2
    return a[:, 0].copy()


def fst(counts: np.ndarray, pairs, method: str, keep=None) -> np.ndarray:
    out = []
    for a, b in np.asarray(pairs).reshape(-1, 2):
        num, den, ok = terms(counts, int(a), int(b), method, keep)
        if not ok.any():
            out.append(np.nan)
            continue
        with np.errstate(divide="ignore", invalid="ignore"):
            out.append(np.float64(fold(tree_blocks(num))) / np.float64(fold(tree_blocks(den))))
    return np.array(out, dtype=np.float64)


def per_locus(counts, pairs, method, keep=None) -> np.ndarray:
    rows = []
    for a, b in np.asarray(pairs).reshape(-1, 2):
        num, den, _ = terms(counts, int(a), int(b), method, keep)
        rows.append(np.stack([num, den], axis=1))
    return np.array(rows, dtype=np.float64).reshape(len(rows), counts.shape[0], 2)


def window_rows(offsets, window_bp: int, step_bp: int = 0):
    """(begin, end) row ranges of windows w = 0 .. max offset // step over offsets [w step, w step + window_bp)."""
    off = np.asarray(offsets, dtype=np.int64)
    step = step_bp or window_bp
    start = np.arange(int(off.max()) // step + 1, dtype=np.int64) * step
    return np.searchsorted(off, start, "left"), np.searchsorted(off, start + window_bp, "left")


def windows(counts, pairs, method, offsets, window_bp: int, step_bp: int = 0, keep=None) -> np.ndarray:
    begin, end = window_rows(offsets, window_bp, step_bp)
    out = np.zeros((len(np.asarray(pairs).reshape(-1, 2)), len(begin), 3), dtype=np.float64)
    for i, (a, b) in enumerate(np.asarray(pairs).reshape(-1, 2)):
        num, den, ok = terms(counts, int(a), int(b), method, keep)
        for w, (lo, hi) in enumerate(zip(begin, end)):
            sel = ok[lo:hi]
            out[i, w] = (fold(num[lo:hi][sel]), fold(den[lo:hi][sel]), float(sel.sum()))
    return out
