"""The launch plans of the estimator sweeps (plan_fast and plan_terms in kgl_gene_b200/csrc/terms_launch.cuh) compiled as a host
program (tests/terms_plan_probe.cu), for tests/test_terms_plan.py and for the GPU tests that size their inputs to reach a given
plan. Needs nvcc, not a GPU (tests/plan_probe.py compiles it).

How the C ABI sizes the sweeps (kgl_gene_b200/csrc/kgl_b200_api.cu), so that a test can name the plan it reaches:
  * k_terms_fast sweeps ceil(N / 32) genome blocks (in late Newton sweeps: ceil(list length / 32) compact blocks) over the
    sample-major words, ceil(L / 32) rounded up to a multiple of 4, restricted to the 256-locus tiles of the rows the last
    select_loci window can select;
  * k_genome_terms (loglik_grid, the exact Newton fallback) runs over every genome block of the device row pitch:
    2 * units, units = ceil(N / 64), rounded up to a multiple of 40 above 56."""
from __future__ import annotations

import plan_probe

NAME = "terms_plan_probe"
MODES = {"RITLAND": 0, "HALL": 1, "NEWTON": 2, "LIMITS": 3, "NEWTON_U": 4}
B200_SMEM_OPTIN = 232_448      # cudaDevAttrMaxSharedMemoryPerBlockOptin of the B200 (227 KB)
NO_WINDOW = -1                 # sel_row_hi of a selection without a window: every tile


def probe_binary() -> str:
    return plan_probe.probe_binary(NAME)


def plans(requests) -> tuple[dict, dict]:
    """requests: iterable of (mode, gblocks, n_words, sel_row_lo, sel_row_hi, sm_count, smem_limit). Returns (constants,
    {field: int64 array, one entry per request})."""
    return plan_probe.run(NAME, requests)


def plan(mode: str, gblocks: int, n_words: int, sm_count: int, sel_row_lo: int = 0, sel_row_hi: int = NO_WINDOW,
         smem_limit: int = B200_SMEM_OPTIN) -> dict:
    """The plan of one sweep as a dict of ints."""
    _, cols = plans([(MODES[mode], gblocks, n_words, sel_row_lo, sel_row_hi, sm_count, smem_limit)])
    return {f: int(v[0]) for f, v in cols.items()}


def term_words(n_loci: int) -> int:
    """Words of the sample-major copy: ceil(L / 32), rounded up to whole 4-word tiles of k_genome_terms."""
    return ((n_loci + 31) // 32 + 3) // 4 * 4


def gblocks_of(n_genomes: int) -> int:
    return (n_genomes + 31) // 32


def device_gblocks(n_genomes: int) -> int:
    """Genome blocks of the device row pitch (what plan_terms is given)."""
    units = (n_genomes + 63) // 64
    return 2 * ((units + 39) // 40 * 40 if units > 56 else units)


def describe(name: str, p: dict) -> str:
    mode = {v: k for k, v in MODES.items()}[p["mode"]]
    if not p["ok"]:
        return f"{name}: {mode}, {p['gblocks']} genome blocks: no plan fits {p['smem_limit']} B"
    return (f"{name}: {mode}, {p['gblocks']} genome blocks x {p['n_words']} words on {p['sm_count']} SMs -> {p['warps']} warps x "
            f"{p['slots']} slots, {p['ctas_per_sm']} CTA(s) per SM, gy {p['gy']}, tiles [{p['tile_begin']}, {p['tile_end']}) in "
            f"{p['n_chunks']} chunk(s) of {p['tiles_per_chunk']} (last {p['last_chunk_tiles']}), {p['smem']} B of shared memory; "
            f"k_genome_terms: {p['term_n_chunks']} chunk(s) of {p['term_words_per_chunk']} words (last {p['term_last_chunk_words']})")
