"""Genotype PCA restated on the host. TEST INFRASTRUCTURE ONLY (never imported by kgl_gene_b200/).

grm_product restates kgl_b200_run_grm_product (kgl_gene_b200/csrc/pca.cuh) operation for operation: the same per-locus
statistics, the same per-column fixed-point quantisation, the same exact integer contractions and the same sequence of double
operations after them, so its result is bit-equal to the device's. The contractions are float64 matrix products of the
{0,1,2} dosage / {0,1} code-3 matrices with the quantised block: every partial sum is an integer of magnitude <= 2 * 2^29 * K,
exact whatever order BLAS adds in while that is < 2^53, i.e. for K < 2^23 genomes and loci (8.4 M; the tests stay far below).
Beyond that a float64 product may round differently from the device's int64 sums, and the restatement is no longer exact.
The device adds the same integers as base-4 digit rows (digits()), which sum_d 4^d digit_d turns back into F_q.
"""
from __future__ import annotations

import numpy as np

from kgl_gene_b200.synth import mix64

Q_MAX = float(2**29 - 1)
OFFSET = 2**29
N_DIGITS = 15


def locus_stats(codes: np.ndarray, keep=None):
    """codes uint8 [L][N] -> (p, d, used): p_l = (n1 + 2 n2) / (2 v), d_l = 1 / sqrt(2 p (1 - p)) on the used loci (keep, 0 < p < 1)."""
    n0, n1, n2 = [(codes == c).sum(axis=1).astype(np.uint64) for c in (0, 1, 2)]
    v = n0 + n1 + n2
    used = v > 0
    if keep is not None:
        used &= np.asarray(keep) != 0
    p = np.zeros(codes.shape[0])
    p[used] = (n1 + 2 * n2)[used].astype(np.float64) / (2 * v)[used].astype(np.float64)
    used &= (p > 0.0) & (p < 1.0)
    p[~used] = 0.0
    d = np.zeros_like(p)
    d[used] = 1.0 / np.sqrt((2.0 * p[used]) * (1.0 - p[used]))
    return p, d, used


def shifts(F: np.ndarray) -> np.ndarray:
    """s_j = the largest integer with max |F[:, j] 2^s_j| < 2^29 (0 for a zero column)."""
    m = np.abs(F).max(axis=0)
    return np.where(m == 0.0, 0, 29 - np.frexp(m)[1]).astype(np.int64)


def quantise(F: np.ndarray, s: np.ndarray, counted: np.ndarray | None = None) -> np.ndarray:
    """int64 min(rint(F 2^s), 2^29 - 1) at the positions that count, 0 elsewhere."""
    q = np.minimum(np.rint(np.ldexp(F, s[None, :].astype(np.int32))), Q_MAX).astype(np.int64)
    if counted is not None:
        q[~counted] = 0
    return q


def digits(fq: np.ndarray) -> np.ndarray:
    """The 15 base-4 digits of F_q = q + 2^29 in [0, 2^30): uint8 [15][...]."""
    f = np.asarray(fq, dtype=np.int64)
    return np.stack([(f >> (2 * d)) & 3 for d in range(N_DIGITS)]).astype(np.uint8)


def _contract(A: np.ndarray, q: np.ndarray) -> np.ndarray:
    return (A @ q.astype(np.float64)).astype(np.int64)


def grm_product(codes: np.ndarray, x: np.ndarray, keep=None):
    """y = Z^T Z x as kgl_b200_run_grm_product computes it (codes uint8 [L][N], x float64 [N][b]); returns (y, M)."""
    x = np.asarray(x, dtype=np.float64).reshape(codes.shape[1], -1)
    p, d, used = locus_stats(codes, keep)
    G = np.where(codes == 3, 0, codes).astype(np.float64)        # [L][N]
    C = (codes == 3).astype(np.float64)
    # pass 1 (K = genomes): Y = Z x
    s = shifts(x)
    xq = quantise(x, s)
    S = xq.sum(axis=0)
    gx, cx = _contract(G, xq), _contract(C, xq)
    p2 = (2.0 * p)[:, None]
    num = gx.astype(np.float64) - p2 * (S[None, :] - cx).astype(np.float64)
    y = np.where(used[:, None], d[:, None] * np.ldexp(num, -s[None, :].astype(np.int32)), 0.0)
    w = d[:, None] * y
    v = p2 * w
    # pass 2 (K = loci, the used ones count): Z^T Y = G^T W - (sum_l V - C^T V)
    t, tv = shifts(w), shifts(v)
    wq, vq = quantise(w, t, used), quantise(v, tv, used)
    T = vq.sum(axis=0)
    gw, cv = _contract(G.T, wq), _contract(C.T, vq)
    out = np.ldexp(gw.astype(np.float64), -t[None, :].astype(np.int32)) - np.ldexp((T[None, :] - cv).astype(np.float64), -tv[None, :].astype(np.int32))
    return out, int(used.sum())


def z_matrix(codes: np.ndarray, keep=None) -> np.ndarray:
    """Dense Z [L][N] in float64 (small shapes)."""
    p, d, used = locus_stats(codes, keep)
    z = (codes.astype(np.float64) - 2.0 * p[:, None]) * d[:, None]
    return np.where(used[:, None] & (codes != 3), z, 0.0)


def psi(codes: np.ndarray, keep=None) -> np.ndarray:
    """Dense Psi = Z^T Z / M."""
    z = z_matrix(codes, keep)
    m = int(locus_stats(codes, keep)[2].sum())
    return (z.T @ z) / m


def start_block(seed: int, n_genomes: int, n_cols: int) -> np.ndarray:
    """The Gaussian start block of kgl_b200_run_pca (pca_start_entry): Box-Muller on splitmix64 draws keyed by (seed, g, j)."""
    g = np.arange(n_genomes, dtype=np.uint64)[:, None]
    j = np.arange(n_cols, dtype=np.uint64)[None, :]
    h1 = mix64(mix64(np.uint64(seed)) ^ ((g << np.uint64(8)) | j))
    h2 = mix64(h1 ^ np.uint64(0xD6E8FEB86659FD93))
    u1 = ((h1 >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0**-53
    u2 = (h2 >> np.uint64(11)).astype(np.float64) * 2.0**-53
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(6.283185307179586 * u2)
