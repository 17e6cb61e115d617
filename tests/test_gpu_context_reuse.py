"""Reuse of one context across inputs. A context keeps caches derived from its inputs (sample-major planes, code-3 index, IBS
planes and tile lists, Gram codes, unit and group tables, the per-locus preparation, moment tables). After one input changes --
a new matrix of the same shape, new super-population labels, new allele frequencies, the multi-allelic loci cleared, the IBS
tensor-core switch flipped -- every analysis on the reused context must equal, bit for bit, the same analysis on a fresh context
given the same inputs: a cache that outlived its input would return results of the previous population."""
from dataclasses import dataclass, replace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, L, N_MULTI = 300, 6000, 40

# Every entry point whose caches a change of input could leave stale, in the order they run on the reused context.
CALLS = [
    ("ibs", lambda g: g.ibs()),
    ("king", lambda g: g.king()),
    ("king_pairs", lambda g: g.king_pairs(0.0)),
    ("gram", lambda g: g.gram()),
    ("grm", lambda g: g.grm(pop=0)),
    ("pca", lambda g: g.pca(k=4, iterations=4, loadings=True)),
    ("ld_pairs", lambda g: g.ld_pairs(0.05, window_loci=40)),
    ("ld_prune", lambda g: g.ld_prune(0.2, window_loci=40)),
    ("group_counts", lambda g: g.group_counts()),
    ("fst", lambda g: g.fst(per_locus=True)),
    ("hardy", lambda g: g.hardy(f=True)),
    ("variant_qc", lambda g: g.variant_qc(min_call_rate=0.99, min_maf=0.01, min_hwe_p=1e-4)),
    ("binned_genome_counts", lambda g: g.binned_genome_counts([0.0, 0.05, 0.3], [0.05, 0.3, 1.0], pop=1)),
    ("select_loci", lambda g: g.select_loci(spacing=0)),
    ("inbreed_simple", lambda g: g.inbreed("Simple")),
    ("inbreed_hallme", lambda g: g.inbreed("HallME")),
]


@dataclass(frozen=True)
class Inputs:
    """What a context holds. af is the frequency table as the device holds it: an upload of multi-allelic loci marks their rows
    "no value" (NaN) there, and clearing the loci leaves the table as it is."""
    packed: np.ndarray
    af: np.ndarray
    offsets: np.ndarray
    superpop: np.ndarray
    multi: tuple | None
    tensor: bool = True


def masked(af, multi):
    af = af.copy()
    af[:, multi[0]] = np.nan
    return af


def populations():
    from kgl_gene_b200.synth import add_multi_allelic, make_population
    a, _ = make_population(N, L, seed=71, missing_rate=0.003)
    b, _ = make_population(N, L, seed=72, missing_rate=0.003)
    add_multi_allelic(a, N_MULTI, seed=73)
    add_multi_allelic(b, N_MULTI, seed=74)
    return a, b


def multi_of(pop):
    return (pop.multi_rows, pop.multi_af, pop.multi_cells)


def load(gpu, s):
    gpu.upload_genotypes(s.packed, N)
    gpu.upload_loci(s.af, s.offsets)
    gpu.set_genome_superpop(s.superpop)
    if s.multi is not None:
        gpu.upload_multi_allelic(*s.multi)
    gpu.set_ibs_tensor_cores(s.tensor)


def run_all(gpu):
    return {name: call(gpu) for name, call in CALLS}


def arrays(v):
    """The arrays of one result (dicts, tuples and scalars included), in a fixed order."""
    if isinstance(v, dict):
        return [a for k in sorted(v) for a in arrays(v[k])]
    if isinstance(v, (tuple, list)):
        return [a for x in v for a in arrays(x)]
    return [np.ascontiguousarray(v)]


def same(x, y):
    ax, ay = arrays(x), arrays(y)
    return len(ax) == len(ay) and all(a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes() for a, b in zip(ax, ay))


def test_reused_context_equals_fresh_context():
    from kgl_gene_b200.capi import KglB200
    a, b = populations()
    rng = np.random.default_rng(75)
    s = Inputs(a.packed, masked(a.af, multi_of(a)), a.offsets, a.superpop, multi_of(a))
    gpu = KglB200(0)
    load(gpu, s)
    run_all(gpu)
    assert gpu.ibs_used_tensor_cores(), "population A should take the tensor-core IBS form"

    def new_matrix(g):          # population B's matrix and its multi-allelic loci (they belong to the matrix)
        g.upload_genotypes(b.packed, N)
        g.upload_multi_allelic(*multi_of(b))
        return replace(s, packed=b.packed, multi=multi_of(b), af=masked(s.af, multi_of(b)))

    def new_labels(g):
        sp = rng.integers(0, 6, size=N).astype(np.uint8)
        g.set_genome_superpop(sp)
        return replace(s, superpop=sp)

    def new_frequencies(g):     # the multi-allelic loci come after the frequency table: uploaded again
        g.upload_loci(b.af, s.offsets)
        g.upload_multi_allelic(*s.multi)
        return replace(s, af=masked(b.af, s.multi))

    def multi_cleared(g):
        g.upload_multi_allelic(None, None, None)
        return replace(s, multi=None)

    def tensor_flipped(g):
        g.set_ibs_tensor_cores(not s.tensor)
        return replace(s, tensor=not s.tensor)

    stale = []
    try:
        for change in (new_matrix, new_labels, new_frequencies, multi_cleared, tensor_flipped):
            s = change(gpu)
            got = run_all(gpu)
            fresh = KglB200(0)
            try:
                load(fresh, s)
                want = run_all(fresh)
            finally:
                fresh.close()
            stale += [f"{change.__name__}: {name}" for name in want if not same(got[name], want[name])]
            assert gpu.ibs_used_tensor_cores() == s.tensor
    finally:
        gpu.close()
    assert not stale, "reused context differs from a fresh one: " + ", ".join(stale)
