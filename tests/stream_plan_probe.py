"""The streaming pass's launch planner (plan_stream in kgl_gene_b200/csrc/stream_common.cuh) compiled as a host program
(tests/stream_plan_probe.cu), for the tests that check its plans and for the GPU tests that size their populations to reach
a given plan. Needs nvcc, not a GPU; the binary goes to a temporary directory."""
from __future__ import annotations

import atexit
import functools
import json
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def nvcc() -> str | None:
    from kgl_gene_b200.build import nvcc_path
    p = nvcc_path()
    return p if os.path.exists(p) else shutil.which(p)


@functools.lru_cache(maxsize=None)
def probe_binary() -> str:
    """Compiles the probe once per process; raises FileNotFoundError without nvcc."""
    compiler = nvcc()
    if compiler is None:
        raise FileNotFoundError("nvcc")
    out_dir = tempfile.mkdtemp(prefix="kgl_plan_probe_")
    atexit.register(shutil.rmtree, out_dir, True)
    exe = os.path.join(out_dir, "stream_plan_probe")
    cmd = [compiler, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++",
           "-I", os.path.join(ROOT, "kgl_gene_b200", "csrc"), "-o", exe, os.path.join(HERE, "stream_plan_probe.cu")]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed on stream_plan_probe.cu:\n" + proc.stdout + proc.stderr)
    return exe


def plans(requests) -> tuple[dict, dict]:
    """requests: iterable of (units, n_loci, sm_count). Returns (constants, {field: int64 array, one entry per request})."""
    text = "".join(f"{int(u)} {int(l)} {int(s)}\n" for u, l, s in requests)
    proc = subprocess.run([probe_binary()], input=text, capture_output=True, text=True, check=True)
    head, _, body = proc.stdout.partition("\n")
    consts = json.loads(head)
    fields = consts.pop("fields")
    rows = np.array(json.loads("[" + body.strip().replace("\n", ",") + "]"), dtype=np.int64).reshape(-1, len(fields))
    return consts, {f: rows[:, i] for i, f in enumerate(fields)}


def plan(units: int, n_loci: int, sm_count: int) -> dict:
    """The plan of one population as a dict of ints."""
    _, cols = plans([(units, n_loci, sm_count)])
    return {f: int(v[0]) for f, v in cols.items()}


def units_of(n_genomes: int) -> int:
    return (n_genomes + 63) // 64
