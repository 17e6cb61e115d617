"""GPU parity at the sizes BASELINE.json's configs are quoted on (VERDICT r1, "no parity at any BASELINE config size").

The populations are generated on the device (k_synth is bit-identical to the oracle's generator, test_device_generator_matches_numpy),
downloaded once and handed to the CPU oracle (OpenMP C restatement, pinned to the reference through tests/golden/): full
2,504 x 1.1 M (config 2) for the allele counts and all four estimators, a 256-genome band of the pairwise matrix at the same
width against the popcount restatement, the 100,000-genome wide path (config 5 width), and the peer-memory exchange of the
locus-sharded step on ONE GPU (two contexts) against the oracle -- including its timeout branch."""
import numpy as np
import pytest

import oracle_py as O
from conftest import results_matrix

pytestmark = pytest.mark.gpu

SEED = 20261018          # bench.py's population


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)) if a.size else 0.0


def device_population(gpu, n, l, seed, missing_rate=0.001, unphased=False):
    """Generates on the device, returns the host copy as a FlatPopulation (the oracle's input)."""
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    offsets, af = make_loci(l, seed)
    superpop, f = make_genomes(n, seed)
    gpu.upload_loci(af, offsets)
    gpu.set_genome_superpop(superpop)
    gpu.set_unphased(unphased)
    gpu.synth_genotypes(seed, n, l, f, missing_rate=missing_rate)
    return FlatPopulation(offsets, af, superpop, gpu.download_genotypes(), n, unphased), f


@pytest.fixture(scope="module")
def c2():
    """BASELINE config 2: 2,504 genomes x 1.1 M loci, the population bench.py times."""
    from kgl_gene_b200.capi import KglB200
    gpu = KglB200(0)
    pop, f = device_population(gpu, 2504, 1_100_000, SEED)
    # a few rare-major rows (q <= 0.01) and very rare alt alleles (p <= 0.001): the sparse side paths at full size
    pop.af[:, ::9973] = np.float32(0.996)
    pop.af[:, 5::7919] = np.float32(0.0004)
    gpu.upload_loci(pop.af, pop.offsets)
    gpu.select_loci()
    sel = O.select_all_pops(pop)
    yield gpu, pop, sel, f
    gpu.close()


def test_c2_generator_and_counts(c2):
    gpu, pop, sel, _ = c2
    from kgl_gene_b200.synth import make_genomes, make_loci
    _, af0 = make_loci(pop.n_loci, SEED)                         # the frequencies the matrix was drawn from (before the c2 fixture's edits)
    _, f0 = make_genomes(pop.n_genomes, SEED)
    want = O.synth_genotypes(SEED, pop.n_genomes, pop.n_loci, af0, pop.superpop, f0)
    assert np.array_equal(pop.packed, want)                      # device generator == oracle generator at full size
    lc, gc = gpu.allele_count()
    olc, ogc = O.allele_count(pop)
    assert np.array_equal(lc, olc) and np.array_equal(gc, ogc)   # bit-exact, all 1.1 M loci and 2,504 genomes
    bits = gpu.get_locus_selection()
    assert np.array_equal(bits, np.bitwise_or.reduce(sel.astype(np.uint8) << np.arange(6, dtype=np.uint8)[:, None], axis=0))


@pytest.mark.parametrize("algo", ["Simple", "RitlandLocus", "HallME", "Loglikelihood"])
def test_c2_estimators(c2, algo):
    """Class counts bit-exact, expected sums and F within the 1e-6 contract (asserted at 1e-8) on the full config-2 matrix.
    Simple / RitlandLocus: every genome. HallME (50 sweeps) / Loglikelihood: the device runs every genome, the CPU oracle
    checks every fourth (626 genomes x 1.1 M loci; all of them would be minutes of host time on the GPU box)."""
    gpu, pop, sel, _ = c2
    kw, okw = {}, {}
    some = None if algo in ("Simple", "RitlandLocus") else np.arange(1, pop.n_genomes, 4)
    if algo == "HallME":
        start = np.linspace(0.05, 0.5, pop.n_genomes)
        kw, okw = dict(hall_start=start, hall_sweeps=50), dict(start=start, sweeps=50)
    if algo == "Simple":
        lc, got = gpu.count_and_inbreed()
        assert np.array_equal(lc, O.allele_count(pop)[0])
    else:
        got = gpu.inbreed(algo, **kw)
    want = O.inbreed(pop, sel, algo, genomes=some, **okw)
    if some is not None:
        got = got[some]
    c_got, f_got = results_matrix(got)
    c_want, f_want = results_matrix(want)
    assert np.array_equal(c_got, c_want)
    assert rel_err(f_got[:, :3], f_want[:, :3]) < 1e-9
    err = np.max(np.abs(got["inbred_allele_sum"] - want["inbred_allele_sum"]) / np.maximum(np.abs(want["inbred_allele_sum"]), 1e-3))
    assert err < 1e-8, err


def test_c2_ibs_band_against_popcount_oracle(c2):
    """256 genomes x all 2,504 partners over 1.1 M loci: 7e11 pair-loci, bit-exact against the popcount CPU restatement."""
    gpu, pop, _, _ = c2
    got = gpu.ibs(1000, 1256)
    want = O.ibs_band_popcount(pop, 1000, 1256)
    assert np.array_equal(got, want)
    tiles = gpu.ibs_tiles(first=3, stride=97, count=8)           # the tile path of the multi-GPU decomposition, same width
    from kgl_gene_b200.shards import upper_tile_coords
    coords = upper_tile_coords(pop.n_genomes)[3::97][:8]
    for (ti, tj), blk in zip(coords, tiles):
        if 1000 <= ti * 64 and ti * 64 + 64 <= 1256:
            assert np.array_equal(blk[:, : min(64, pop.n_genomes - tj * 64)], want[ti * 64 - 1000: ti * 64 - 936, tj * 64: tj * 64 + 64])


def test_wide_population_100k_genomes():
    """BASELINE config 5 width: 100,000 genomes (1,563 units -> 40 slices of the <40,64> kernel, global-atomic locus counts)
    x 4,096 loci against the oracle: allele counts and Simple / RitlandLocus."""
    from kgl_gene_b200.capi import KglB200
    gpu = KglB200(0)
    try:
        pop, _ = device_population(gpu, 100_000, 4096, 31)
        pop.af[:, ::211] = np.float32(0.995)
        gpu.upload_loci(pop.af, pop.offsets)
        gpu.select_loci(spacing=15)
        sel = O.select_all_pops(pop, spacing=15)
        lc, gc = gpu.allele_count()
        olc, ogc = O.allele_count(pop)
        assert np.array_equal(lc, olc) and np.array_equal(gc, ogc)
        lc2, res = gpu.count_and_inbreed()
        assert np.array_equal(lc2, olc)
        for algo, got in (("Simple", res), ("RitlandLocus", gpu.inbreed("RitlandLocus"))):
            want = O.inbreed(pop, sel, algo)
            c_got, f_got = results_matrix(got)
            c_want, f_want = results_matrix(want)
            assert np.array_equal(c_got, c_want), algo
            assert rel_err(f_got[:, :3], f_want[:, :3]) < 1e-10, algo
            assert np.max(np.abs(got["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-8, algo
    finally:
        gpu.close()


def test_c1_width_full_contig():
    """BASELINE config 1 shape: 500 genomes x 500,000 loci (one of the 14 contigs), unphased (Pf7, SURVEY Q6): the <8,256>
    kernel, all four estimators against the oracle. At 148 SMs a CTA runs 14 stages, one counter chunk; the flushes between
    chunks are tested in tests/test_gpu_stream_plans.py."""
    from kgl_gene_b200.capi import KglB200
    gpu = KglB200(0)
    try:
        pop, _ = device_population(gpu, 500, 500_000, 1001, missing_rate=0.002, unphased=True)
        gpu.select_loci(spacing=25, min_af=0.0005, max_af=0.9)
        sel = O.select_all_pops(pop, spacing=25, min_af=0.0005, max_af=0.9)
        lc, res = gpu.count_and_inbreed()
        assert np.array_equal(lc, O.allele_count(pop)[0])
        start = np.linspace(0.05, 0.5, pop.n_genomes)
        for algo, kw, okw in (("Simple", None, {}), ("RitlandLocus", {}, {}), ("HallME", dict(hall_start=start, hall_sweeps=50), dict(start=start, sweeps=50)),
                              ("Loglikelihood", {}, {})):
            got = res if kw is None else gpu.inbreed(algo, **kw)
            want = O.inbreed(pop, sel, algo, **okw)
            assert np.array_equal(results_matrix(got)[0], results_matrix(want)[0]), algo
            assert rel_err(results_matrix(got)[1][:, :3], results_matrix(want)[1][:, :3]) < 1e-10, algo
            assert np.max(np.abs(got["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-8, algo
    finally:
        gpu.close()


# ------------------------------------------------------------------------------------------- peer exchange, one GPU ----
def _two_shards(pop, cut):
    from kgl_gene_b200.flatfile import FlatPopulation
    return [FlatPopulation(pop.offsets[a:b], np.ascontiguousarray(pop.af[:, a:b]), pop.superpop, np.ascontiguousarray(pop.packed[a:b]),
                           pop.n_genomes, pop.unphased) for a, b in ((0, cut), (cut, pop.n_loci))]


def test_peer_exchange_on_one_gpu_matches_oracle():
    """kgl_b200_enqueue_count_and_inbreed_peer with two contexts of one process on one GPU (the regions are mapped directly):
    both 'ranks' must hold the oracle's result for the UNSHARDED population, bit-identical to each other, over several steps
    (both parities of the exchange region)."""
    from kgl_gene_b200.capi import KglB200
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(700, 40_000, seed=71, missing_rate=0.003)
    pop.af[:, ::173] = np.float32(0.997)
    shards = _two_shards(pop, 17_000 + 13)
    ctxs = [KglB200(0) for _ in shards]
    try:
        for c, sh in zip(ctxs, shards):
            c.upload_population(sh)
            c.select_loci()
        handles = [c.peer_export() for c in ctxs]
        for r, c in enumerate(ctxs):
            c.peer_attach(r, 2, handles)
        sel = O.select_all_pops(pop)
        want = O.inbreed(pop, sel, "Simple")
        olc, _ = O.allele_count(pop)
        for step in range(3):
            for c in ctxs:
                c.enqueue_count_and_inbreed_peer()
            got = [c.inbreed_fetch() for c in ctxs]
            for g in got:
                assert np.array_equal(results_matrix(g)[0], results_matrix(want)[0])
                assert rel_err(results_matrix(g)[1][:, :3], results_matrix(want)[1][:, :3]) < 1e-11
                assert np.max(np.abs(g["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-9
            assert got[0].tobytes() == got[1].tobytes()
            lcs = [c.fetch_locus_counts() for c in ctxs]
            assert np.array_equal(np.concatenate(lcs), olc)
    finally:
        for c in ctxs:
            c.close()


def test_peer_exchange_timeout_is_an_error():
    """A peer that never reaches the exchange: the step gives up after the timeout, the fetch entry points return
    KGL_B200_ERR_PEER (6) instead of silent NaNs, and the context asks for a new export / attach."""
    from kgl_gene_b200.capi import KglB200, KglError
    from kgl_gene_b200.synth import make_population
    pop, _ = make_population(130, 3000, seed=72)
    ctxs = [KglB200(0), KglB200(0)]
    try:
        for c in ctxs:
            c.upload_population(pop)
            c.select_loci()
        handles = [c.peer_export() for c in ctxs]
        for r, c in enumerate(ctxs):
            c.peer_attach(r, 2, handles)
        ctxs[0].peer_set_timeout_ms(300)
        ctxs[0].enqueue_count_and_inbreed_peer()          # rank 1 never steps
        with pytest.raises(KglError, match=r"\[6\].*timed out"):
            ctxs[0].inbreed_fetch()
        with pytest.raises(KglError, match="peer_export"):
            ctxs[0].enqueue_count_and_inbreed_peer()
        # a fresh export / attach on both sides works again
        handles = [c.peer_export() for c in ctxs]
        for r, c in enumerate(ctxs):
            c.peer_attach(r, 2, handles)
        for c in ctxs:
            c.enqueue_count_and_inbreed_peer()
        a, b = (c.inbreed_fetch() for c in ctxs)
        assert a.tobytes() == b.tobytes() and np.all(np.isfinite(a["inbred_allele_sum"]))
    finally:
        for c in ctxs:
            c.close()


def test_run_inbreed_sharded_two_gpus(tmp_path):
    """shards.run_inbreed_sharded itself (the shipped helper: context stream bound to torch's stream, NCCL all-reduce between
    accumulate and update) on two GPUs, against the oracle on the unsharded population."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(here, "sharded_worker.py"), str(tmp_path)]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stderr[-3000:]
    assert os.path.exists(tmp_path / "ok0") and os.path.exists(tmp_path / "ok1")
