"""Linkage disequilibrium restated on the host. TEST INFRASTRUCTURE ONLY (never imported by kgl_gene_b200/).

r2 restates k_ld_pairs (kgl_gene_b200/csrc/ld.cuh) operation for operation: the per-pair sums GG, CC, GC and QC are float64
products of the {0,1,2} dosage, {0,1,4} squared-dosage and {0,1} code-3 matrices (integers <= 4 N, exact), the identities run in
int64 and the double part is the same three IEEE operations, so the result is bit-equal to the device's. The window, the pair
list and the greedy prune are plain loops over the definitions of include/kgl_b200.h, and planted() makes populations with
haplotype blocks of strong LD."""
from __future__ import annotations

import numpy as np

from pca_oracle import locus_stats

PAIR_FIELDS = [("a", "<u4"), ("b", "<u4"), ("n_valid", "<u4"), ("reserved", "<u4"), ("r2", "<f8")]


def eligible(codes: np.ndarray, keep=None) -> np.ndarray:
    """PCA's used set: keep[l] != 0 (None = all) and 0 < p < 1."""
    return locus_stats(codes, keep)[2]


def window_pairs(elig: np.ndarray, offsets, window_loci: int, window_bp: int):
    """(a, b) int64 arrays of every in-window pair a < b of eligible loci, ascending by (a, b)."""
    assert window_loci or window_bp
    e = np.flatnonzero(elig)
    off = None if offsets is None else np.asarray(offsets, dtype=np.int64)
    a_all, b_all = [], []
    for d in range(1, len(e)):
        if window_loci and d >= window_loci:
            break
        a, b = e[:-d], e[d:]
        if window_bp:
            ok = off[b] - off[a] <= window_bp
            if not ok.any():          # offsets are sorted: no pair further apart in rank is closer in bp
                break
            a, b = a[ok], b[ok]
        a_all.append(a)
        b_all.append(b)
    if not a_all:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64)
    a, b = np.concatenate(a_all), np.concatenate(b_all)
    order = np.lexsort((b, a))
    return a[order], b[order]


def r2(codes: np.ndarray, a: np.ndarray, b: np.ndarray, chunk: int = 1 << 22):
    """(n_valid int64, r2 float64) of the pairs (a[i], b[i]) by the sequence of include/kgl_b200.h."""
    codes = np.asarray(codes)
    n_genomes = codes.shape[1]
    G = np.where(codes == 3, 0, codes).astype(np.float64)
    Q = G * G
    Cm = (codes == 3).astype(np.float64)
    s, q, c = G.sum(axis=1).astype(np.int64), Q.sum(axis=1).astype(np.int64), Cm.sum(axis=1).astype(np.int64)
    n_out = np.zeros(len(a), dtype=np.int64)
    r_out = np.zeros(len(a), dtype=np.float64)
    step = max(1, chunk // max(n_genomes, 1))
    for i0 in range(0, len(a), step):
        ia, ib = a[i0:i0 + step], b[i0:i0 + step]
        dot = lambda X, Y: (X[ia] * Y[ib]).sum(axis=1).astype(np.int64)
        gg, cc = dot(G, G), dot(Cm, Cm)
        gc_ab, gc_ba = dot(G, Cm), (G[ib] * Cm[ia]).sum(axis=1).astype(np.int64)
        qc_ab, qc_ba = dot(Q, Cm), (Q[ib] * Cm[ia]).sum(axis=1).astype(np.int64)
        n = n_genomes - c[ia] - c[ib] + cc
        sa, sb = s[ia] - gc_ab, s[ib] - gc_ba
        qa, qb = q[ia] - qc_ab, q[ib] - qc_ba
        cov = n * gg - sa * sb
        va, vb = n * qa - sa * sa, n * qb - sb * sb
        with np.errstate(invalid="ignore", divide="ignore"):
            r = (cov.astype(np.float64) * cov.astype(np.float64)) / (va.astype(np.float64) * vb.astype(np.float64))
        r[(va == 0) | (vb == 0)] = np.nan
        n_out[i0:i0 + step], r_out[i0:i0 + step] = n, r
    return n_out, r_out


def all_window_r2(codes, offsets=None, window_loci=0, window_bp=0, keep=None):
    """(a, b, n_valid, r2) of every in-window pair, ascending by (a, b)."""
    a, b = window_pairs(eligible(codes, keep), offsets, window_loci, window_bp)
    n, r = r2(codes, a, b)
    return a, b, n, r


def ld_pairs(codes, min_r2, offsets=None, window_loci=0, window_bp=0, keep=None) -> np.ndarray:
    """kgl_b200_run_ld_pairs: the in-window pairs with r^2 >= min_r2 (NaN never), ascending by (a, b)."""
    a, b, n, r = all_window_r2(codes, offsets, window_loci, window_bp, keep)
    take = r >= min_r2
    out = np.zeros(int(take.sum()), dtype=PAIR_FIELDS)
    out["a"], out["b"], out["n_valid"], out["r2"] = a[take], b[take], n[take], r[take]
    return out


def prune_scan(n_loci: int, elig: np.ndarray, a: np.ndarray, b: np.ndarray, r: np.ndarray, max_r2: float) -> np.ndarray:
    """The greedy rule over in-window pairs (a, b, r2): eligible l is kept unless an earlier kept i has r2(i, l) > max_r2."""
    partners = {}
    for i, j in zip(a[r > max_r2].tolist(), b[r > max_r2].tolist()):
        partners.setdefault(j, []).append(i)
    keep = np.zeros(n_loci, dtype=np.uint8)
    for l in range(n_loci):
        if elig[l] and not any(keep[i] for i in partners.get(l, ())):
            keep[l] = 1
    return keep


def ld_prune(codes, max_r2, offsets=None, window_loci=0, window_bp=0, keep=None) -> np.ndarray:
    """kgl_b200_run_ld_prune's keep_out."""
    a, b, n, r = all_window_r2(codes, offsets, window_loci, window_bp, keep)
    return prune_scan(codes.shape[0], eligible(codes, keep), a, b, r, max_r2)


def planted(n_genomes: int, n_loci: int, seed: int, block: int = 40, founders: int = 3, mutation: float = 0.01,
            missing: float = 0.0, multi_rows: int = 0) -> np.ndarray:
    """uint8 [L][N] codes with planted LD: each block of `block` loci has a few founder haplotypes; every one of the 2 N
    haplotypes copies a random founder per block, with each allele flipped at rate `mutation`, and pairs of haplotypes make the
    diploid genotypes. Then code-3 cells at rate `missing` and `multi_rows` multi-allelic rows (only 0 and 3)."""
    rng = np.random.default_rng(seed)
    hap = np.zeros((n_loci, 2 * n_genomes), dtype=np.uint8)
    for b0 in range(0, n_loci, block):
        b1 = min(n_loci, b0 + block)
        p = rng.uniform(0.1, 0.9, size=(b1 - b0, 1))
        f = (rng.random((b1 - b0, founders)) < p).astype(np.uint8)
        pick = rng.integers(0, founders, size=2 * n_genomes)
        h = f[:, pick]
        hap[b0:b1] = h ^ (rng.random(h.shape) < mutation)
    codes = hap[:, 0::2] + hap[:, 1::2]
    if missing:
        codes[rng.random(codes.shape) < missing] = 3
    if multi_rows:
        rows = rng.choice(n_loci, size=multi_rows, replace=False)
        codes[rows] = np.where(rng.random((multi_rows, n_genomes)) < 0.2, 3, 0)
    return codes.astype(np.uint8)
