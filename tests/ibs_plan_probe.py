"""The launch plan of pairwise IBS on the popcount kernel (plan_ibs, ibs_words_used and ibs_repair_segments in
kgl_gene_b200/csrc/ibs_launch.cuh) compiled as a host program (tests/ibs_plan_probe.cu), for tests/test_ibs_plan.py and for the
GPU tests that size their inputs to reach a given plan. Needs nvcc, not a GPU (tests/plan_probe.py compiles it).

How the IBS and KING calls size their launches (kgl_gene_b200/csrc/kgl_b200_api.cu), so that a test can name the plan it reaches:
  * one launch of k_ibs_tiles (and of k_ibs_missing_fix) per tile list of at most 8,192 64 x 64 tiles;
  * ibs() / king() of the whole matrix (run_pairwise): the upper-triangle tiles, 8,192 per launch, when the N x N result takes
    at most 2 GiB; otherwise, and for a band of rows, slabs of whole tile rows (every tile of the row) of at most 1 GiB of result
    and 8,192 tiles;
  * ibs_tiles / ibs_tile_list: the tiles of the call, 8,192 per launch; king_pairs: the upper-triangle tiles (or the listed
    ones), 8,192 per launch."""
from __future__ import annotations

import plan_probe

NAME = "ibs_plan_probe"
TILE = 64                    # kIbsT: genomes per tile side
MAX_TILES = 8192             # kIbsMaxTilesPerLaunch


def probe_binary() -> str:
    return plan_probe.probe_binary(NAME)


def plans(requests) -> tuple[dict, dict]:
    """requests: iterable of (n_tiles, n_loci, sm_count, n_dropped, n_genomes) or with max_rows (the most dropped rows of one
    genome) appended. Returns (constants, {field: int64 array, one entry per request})."""
    return plan_probe.run(NAME, requests)


def plan(n_tiles: int, n_loci: int, sm_count: int, n_dropped: int = 0, n_genomes: int = 1, max_rows: int = 0) -> dict:
    """The plan of one launch as a dict of ints."""
    _, cols = plans([(n_tiles, n_loci, sm_count, n_dropped, n_genomes, max_rows)])
    return {f: int(v[0]) for f, v in cols.items()}


def side(n_genomes: int) -> int:
    return (n_genomes + TILE - 1) // TILE


def upper_tiles(n_genomes: int) -> int:
    s = side(n_genomes)
    return s * (s + 1) // 2


def pairwise_launches(n_genomes: int, row_begin: int, row_end: int, bytes_per_pair: int) -> list[int]:
    """Tiles of each launch of run_pairwise (kgl_b200_api.cu) for rows [row_begin, row_end): 16 bytes a pair for IBS, 8 for KING."""
    n, s = n_genomes, side(n_genomes)
    if row_begin == 0 and row_end == n and n * n * bytes_per_pair <= 2 << 30:
        total = upper_tiles(n)
        return [min(MAX_TILES, total - t0) for t0 in range(0, total, MAX_TILES)]
    rows = max(1, min((1 << 30) // (n * bytes_per_pair * TILE), MAX_TILES // s))
    out, tr0 = [], row_begin // TILE
    while tr0 * TILE < row_end:
        tr1 = min((row_end + TILE - 1) // TILE, tr0 + rows)
        out.append((tr1 - tr0) * s)
        tr0 += rows
    return out


def describe(name: str, p: dict) -> str:
    kind = "split" if p["n_chunks"] > 1 else "one chunk"
    text = (f"{name}: {p['n_tiles']} tiles x {p['words_used']} words ({p['n_loci']} loci) on {p['sm_count']} SMs -> "
            f"{p['n_chunks']} chunk(s) of {p['stages_per_chunk']} stages (last {p['last_chunk_words']} words = "
            f"{p['last_chunk_stages']} stages, last stage {p['last_stage_words']} words), {p['units']} units on {p['grid']} CTAs, "
            f"up to {p['max_units_per_cta']} per CTA ({kind})")
    if p["n_dropped"]:
        text += f"; repair: {p['segs']} segment(s)"
        if p["max_rows"]:
            text += f", a thread walks up to {p['walk_rows']} rows in {p['walk_passes']} counter pass(es)"
    return text
