"""The tensor-core Gram kernel's launch planner (plan_gram in kgl_gene_b200/csrc/gram_launch.cuh) compiled as a host program
(tests/gram_plan_probe.cu), for tests/test_gram_plan.py and for the GPU tests that size their loci or tile lists to reach a given
plan. Needs nvcc, not a GPU (tests/plan_probe.py compiles it).

How the callers of k_gram_i8 size their runs (kgl_gene_b200/csrc/kgl_b200_api.cu), so that a test can name the plan it reaches:
  * run_gram / enqueue_gram_tiles: the upper-triangle 256 x 256 tiles of the ld x ld matrix (every stride-th from `first`),
    K = loci;
  * IBS on the tensor cores and KING: the distinct 256 x 256 blocks under the 64 x 64 tiles of the call, K = loci;
  * PCA pass 1: (loci of the slab / 256) x (column blocks of 16) tiles, K = genomes; pass 2: (ld / 256) x (column blocks)
    tiles per run, K = loci."""
from __future__ import annotations

import plan_probe

NAME = "gram_plan_probe"
TILE = 256           # kGramM = kGramN
STAGE = 128          # loci (or genomes) per k-stage


def probe_binary() -> str:
    return plan_probe.probe_binary(NAME)


def plans(requests) -> tuple[dict, dict]:
    """requests: iterable of (n_tiles, k_stages, sm_count) or (n_tiles, k_stages, sm_count, chunk_stages_hint).
    Returns (constants, {field: int64 array, one entry per request})."""
    return plan_probe.run(NAME, requests)


def plan(n_tiles: int, k_stages: int, sm_count: int) -> dict:
    """The plan of one run as a dict of ints."""
    _, cols = plans([(n_tiles, k_stages, sm_count)])
    return {f: int(v[0]) for f, v in cols.items()}


def k_stages(k: int) -> int:
    return (k + STAGE - 1) // STAGE


def upper_tiles(n_genomes: int) -> int:
    """Tiles of a run_gram call."""
    t = (n_genomes + TILE - 1) // TILE
    return t * (t + 1) // 2


def pca_tiles(n_genomes: int, n_loci: int, cols: int) -> tuple[int, int]:
    """Tiles of the PCA pass-1 run (one slab: up to ~174,000 loci at 48 columns) and of each pass-2 run."""
    nb = (cols + 15) // 16
    return (n_loci + TILE - 1) // TILE * nb, (n_genomes + TILE - 1) // TILE * nb


def describe(name: str, p: dict) -> str:
    kind = "split-K" if p["n_chunks"] > 1 else "one chunk"
    return (f"{name}: {p['n_tiles']} tiles x {p['k_stages']} k-stages on {p['sm_count']} SMs -> {p['n_chunks']} chunk(s) of "
            f"{p['stages_per_chunk']} stages (last {p['last_stages']}), {p['units']} units on {p['grid']} CTAs, up to "
            f"{p['max_units_per_cta']} per CTA ({kind})")
