"""KING-robust kinship restated on the host with indicator matrices. TEST INFRASTRUCTURE ONLY (never imported by kgl_gene_b200/).

Every count is its own float64 matrix product (exact below 2^53); none is derived from another through an identity, so the
restatement is independent of the device path (kgl_gene_b200/csrc/king.cuh), which uses het_a + het_b = IBS1 + 2 het_het.
"""
from __future__ import annotations

import numpy as np


def king(pop) -> dict:
    """Over the loci where neither genome is coded 3 (V = valid indicator; R / H / A = hom-ref / heterozygous / hom-alt):
    n_valid = V V^T, ibs0 = A R^T + R A^T, ibs1 = H (R + A)^T + (R + A) H^T, het_het = H H^T, het_a = H V^T, het_b = V H^T,
    kinship = 0.5 - (4 ibs0 + ibs1) / (4 min(het_a, het_b)), NaN where the minimum is 0. Returns int64 [N][N] count matrices
    and the float64 kinship matrix."""
    codes = pop.codes().T                                 # [N][L]
    R, H, A, V = [(codes == c).astype(np.float64) for c in (0, 1, 2)] + [(codes != 3).astype(np.float64)]
    out = {"n_valid": V @ V.T, "ibs0": A @ R.T + R @ A.T, "ibs1": H @ (R + A).T + (R + A) @ H.T, "het_het": H @ H.T,
           "het_a": H @ V.T, "het_b": V @ H.T}
    num = 4.0 * out["ibs0"] + out["ibs1"]
    den = 4.0 * np.minimum(out["het_a"], out["het_b"])
    with np.errstate(divide="ignore", invalid="ignore"):
        kin = np.where(den > 0, 0.5 - num / np.where(den > 0, den, 1.0), np.nan)
    out = {k: v.astype(np.int64) for k, v in out.items()}
    out["kinship"] = kin
    return out
