"""Relationship degrees from KING-robust kinship coefficients (KglB200.king / king_pairs).

The bounds are the ones of Manichaikul et al. (Bioinformatics 2010, table 1) and PLINK 2's --king-cutoff: powers of two halfway
(in log2) between the expected kinships 1/2, 1/4, 1/8, 1/16 of duplicates / monozygotic twins and first-, second- and
third-degree relatives.
"""
from __future__ import annotations

import numpy as np

DUPLICATE = 2.0 ** -1.5      # > : duplicate / MZ twin
FIRST = 2.0 ** -2.5          # >= : first degree (parent-offspring, full siblings)
SECOND = 2.0 ** -3.5         # >= : second degree
THIRD = 2.0 ** -4.5          # >= : third degree; below: unrelated


def king_degree(kinship):
    """0 (duplicate / MZ twin), 1, 2, 3 (degree of relationship) or -1 (unrelated, or NaN) for each kinship coefficient.
    Returns an int8 array of the input's shape, or an int for a scalar."""
    k = np.asarray(kinship, dtype=np.float64)
    out = np.full(k.shape, -1, dtype=np.int8)
    with np.errstate(invalid="ignore"):
        out[k >= THIRD] = 3
        out[k >= SECOND] = 2
        out[k >= FIRST] = 1
        out[k > DUPLICATE] = 0
    return int(out) if out.ndim == 0 else out
