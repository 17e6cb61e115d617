"""The streaming pass's launch planner (plan_stream in kgl_gene_b200/csrc/stream_common.cuh) compiled as a host program
(tests/stream_plan_probe.cu), for the tests that check its plans and for the GPU tests that size their populations to reach
a given plan. Needs nvcc, not a GPU (tests/plan_probe.py compiles it)."""
from __future__ import annotations

import plan_probe

NAME = "stream_plan_probe"


def probe_binary() -> str:
    """Compiles the probe once per process; raises FileNotFoundError without nvcc."""
    return plan_probe.probe_binary(NAME)


def plans(requests) -> tuple[dict, dict]:
    """requests: iterable of (units, n_loci, sm_count). Returns (constants, {field: int64 array, one entry per request})."""
    return plan_probe.run(NAME, requests)


def plan(units: int, n_loci: int, sm_count: int) -> dict:
    """The plan of one population as a dict of ints."""
    _, cols = plans([(units, n_loci, sm_count)])
    return {f: int(v[0]) for f, v in cols.items()}


def units_of(n_genomes: int) -> int:
    return (n_genomes + 63) // 64
