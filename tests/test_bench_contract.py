"""The command-line contract of bench.py: the reference arm prints exactly one JSON line on stdout with the keys a caller
reads and times exactly --steps repeats, the GPU arm refuses to run (no CPU fallback) when there is no device, and
--dump-outputs writes the step's per-locus counts and per-genome results (checked against the oracle on a GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                           "--reference-sample", "256x4000"],      # (the default BASELINE sample takes minutes on this container's 8 cores)
                          capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, proc.stdout[:500]
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "inbreeding genotype-loci/s" and line["unit"] == "genotype-loci/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]


def test_reference_arm_times_the_steps_asked_for():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3",
                           "--reference-sample", "64x2000"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    line = json.loads(proc.stdout)
    assert line["steps"] == 3 and line["warmup"] == 1


@pytest.mark.parametrize("args", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_arguments_that_do_not_fit_are_refused(args):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert proc.returncode == 2 and proc.stdout == "", proc.stderr[-2000:]


@pytest.mark.parametrize("n_genomes", [300, 5000])
def test_dump_stays_within_its_budget(tmp_path, monkeypatch, n_genomes):
    """Beyond the budget the dump holds fixed, seeded samples of rows (per-locus counts; per-genome results past half of it),
    .npy headers included."""
    import numpy as np
    import bench
    from kgl_gene_b200.capi import RESULT_DTYPE
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    lc = np.arange(20_000 * 4, dtype=np.uint32).reshape(20_000, 4)
    res = np.zeros(n_genomes, dtype=RESULT_DTYPE)
    res["inbred_allele_sum"] = np.linspace(-0.5, 0.5, n_genomes)
    res["total_allele_count"] = np.arange(n_genomes)
    bench.dump_outputs(str(tmp_path), lc, res)
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= bench.DUMP_BYTES
    rows = np.load(tmp_path / "locus_rows.npy")
    counts = np.load(tmp_path / "locus_counts.npy")
    assert rows.dtype == np.float64 and rows.size > 1000 and np.all(np.diff(rows) > 0)
    assert counts.dtype == np.float32 and np.array_equal(counts, lc[rows.astype(np.int64)])
    genomes = np.arange(n_genomes)
    if n_genomes * 80 > bench.DUMP_BYTES // 2:
        genomes = np.load(tmp_path / "genome_rows.npy").astype(np.int64)
        assert 1000 < genomes.size < n_genomes
    else:
        assert not os.path.exists(tmp_path / "genome_rows.npy")
    for f in ("inbred_allele_sum", "total_allele_count"):
        got = np.load(tmp_path / f"genome_{f}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, res[f][genomes])
    bench.dump_outputs(str(tmp_path / "again"), lc, res)           # the samples are fixed: the same rows every run
    for f in os.listdir(tmp_path / "again"):
        assert np.array_equal(np.load(tmp_path / "again" / f), np.load(tmp_path / f)), f


@pytest.mark.gpu
def test_dumped_outputs_are_what_the_oracle_computes(tmp_path):
    """--dump-outputs on one GPU: the step's per-locus counts and per-genome Simple results, against the CPU oracle on the
    population the bench generates (the device generator equals the oracle's, tests/test_gpu_baseline_sizes.py)."""
    import numpy as np
    import oracle_py as O
    from bench import SEED
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    n, l = 300, 40_000
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--genomes", str(n), "--loci", str(l), "--steps", "4",
                           "--warmup", "1", "--no-e2e", "--no-kinship", "--no-estimators", "--no-cpu-baseline",
                           "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    assert json.loads(proc.stdout)["steps"] == 4
    offsets, af = make_loci(l, SEED)
    superpop, inbreeding = make_genomes(n, SEED)
    pop = FlatPopulation(offsets, af, superpop, O.synth_genotypes(SEED, n, l, af, superpop, inbreeding), n, False)
    counts = np.load(tmp_path / "locus_counts.npy")
    assert counts.dtype == np.float32 and not os.path.exists(tmp_path / "locus_rows.npy")
    assert np.array_equal(counts, O.allele_count(pop)[0])
    want = O.inbreed(pop, O.select_all_pops(pop), "Simple")
    for f in want.dtype.names:
        got = np.load(tmp_path / f"genome_{f}.npy")
        assert got.dtype == np.float64 and got.shape == (n,)
        if f.endswith("_count"):
            assert np.array_equal(got, want[f]), f
        else:
            assert np.max(np.abs(got - want[f]) / np.maximum(np.abs(want[f]), 1e-3)) < 1e-6, f


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode != 0 and proc.stdout.strip() == ""
    assert "no CPU fallback" in proc.stderr or "no CUDA device" in proc.stderr
