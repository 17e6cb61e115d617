"""Launch planners compiled as host programs (tests/*_plan_probe.cu), for the tests that check their plans and for the GPU tests
that size their inputs to reach a given plan. Needs nvcc, not a GPU; the binaries go to a temporary directory.

A probe reads one request per line on stdin and prints one JSON object (its field names under "fields", and its constants),
then one JSON array per request in that field order."""
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
def probe_binary(name: str) -> str:
    """Compiles tests/<name>.cu once per process; raises FileNotFoundError without nvcc."""
    compiler = nvcc()
    if compiler is None:
        raise FileNotFoundError("nvcc")
    out_dir = tempfile.mkdtemp(prefix="kgl_plan_probe_")
    atexit.register(shutil.rmtree, out_dir, True)
    exe = os.path.join(out_dir, name)
    cmd = [compiler, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "/usr/bin/g++",
           "-I", os.path.join(ROOT, "kgl_gene_b200", "csrc"), "-o", exe, os.path.join(HERE, name + ".cu")]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"nvcc failed on {name}.cu:\n" + proc.stdout + proc.stderr)
    return exe


def run(name: str, requests) -> tuple[dict, dict]:
    """requests: iterable of tuples of ints, one line each. Returns (constants, {field: int64 array, one entry per request})."""
    text = "".join(" ".join(str(int(v)) for v in r) + "\n" for r in requests)
    proc = subprocess.run([probe_binary(name)], input=text, capture_output=True, text=True, check=True)
    head, _, body = proc.stdout.partition("\n")
    consts = json.loads(head)
    fields = consts.pop("fields")
    rows = np.array(json.loads("[" + body.strip().replace("\n", ",") + "]"), dtype=np.int64).reshape(-1, len(fields))
    return consts, {f: rows[:, i] for i, f in enumerate(fields)}
