"""KING-robust kinship restated on the host with indicator matrices. TEST INFRASTRUCTURE ONLY (never imported by kgl_gene_b200/).

Every count is its own float64 matrix product (exact below 2^53); none is derived from another through an identity, so the
restatement is independent of the device path (kgl_gene_b200/csrc/king.cuh), which uses het_a + het_b = IBS1 + 2 het_het.
"""
from __future__ import annotations

import numpy as np

COUNTS = ("n_valid", "ibs0", "ibs1", "het_het", "het_a", "het_b")


def king(pop) -> dict:
    """Over the loci where neither genome is coded 3 (V = valid indicator; R / H / A = hom-ref / heterozygous / hom-alt):
    n_valid = V V^T, ibs0 = A R^T + R A^T, ibs1 = H (R + A)^T + (R + A) H^T, het_het = H H^T, het_a = H V^T, het_b = V H^T,
    kinship = 0.5 - (4 ibs0 + ibs1) / (4 min(het_a, het_b)), NaN where the minimum is 0. Returns int64 [N][N] count matrices
    and the float64 kinship matrix."""
    return king_codes(pop.codes())


def king_codes(codes: np.ndarray, weights=None, rows=None, chunk: int = 1 << 16) -> dict:
    """king() of the code matrix uint8 [L][N], rows `rows` (a slice or index array of genomes; None = all) against all genomes.
    weights int [L] (None = 1): locus l counts weights[l] times, so a population whose loci repeat a few patterns is given by
    the patterns and their multiplicities. Loci are taken `chunk` at a time."""
    codes = np.asarray(codes)
    rows = slice(None) if rows is None else rows
    w = np.ones(codes.shape[0]) if weights is None else np.asarray(weights, dtype=np.float64)
    out = None
    for l0 in range(0, codes.shape[0], chunk):
        c = codes[l0:l0 + chunk].T                        # [N][l]
        R, H, A, V = [(c == k).astype(np.float64) for k in (0, 1, 2)] + [(c != 3).astype(np.float64)]
        wl = w[l0:l0 + chunk]
        Rw, Hw, Aw, Vw = R[rows] * wl, H[rows] * wl, A[rows] * wl, V[rows] * wl
        part = {"n_valid": Vw @ V.T, "ibs0": Aw @ R.T + Rw @ A.T, "ibs1": Hw @ (R + A).T + (Rw + Aw) @ H.T, "het_het": Hw @ H.T,
                "het_a": Hw @ V.T, "het_b": Vw @ H.T}
        out = part if out is None else {k: out[k] + part[k] for k in COUNTS}
    num = 4.0 * out["ibs0"] + out["ibs1"]
    den = 4.0 * np.minimum(out["het_a"], out["het_b"])
    with np.errstate(divide="ignore", invalid="ignore"):
        kin = np.where(den > 0, 0.5 - num / np.where(den > 0, den, 1.0), np.nan)
    out = {k: v.astype(np.int64) for k, v in out.items()}
    out["kinship"] = kin
    return out
