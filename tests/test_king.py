"""KING-robust kinship, CPU side: the oracle's matrix-product restatement against a naive per-pair loop, the count identities,
the degree bounds, the pair record's layout and the gather of per-rank pair lists on two gloo ranks."""
import ctypes as C
import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

import king_oracle as K
import oracle_py as O
from kgl_gene_b200 import capi, shards
from kgl_gene_b200.kinship import king_degree
from kgl_gene_b200.synth import add_multi_allelic, make_population


def naive_king(pop):
    """Pair by pair over the loci valid in both, in plain Python integers."""
    codes = pop.codes().T.astype(np.int64)
    n = codes.shape[0]
    names = ("n_valid", "ibs0", "ibs1", "het_het", "het_a", "het_b")
    out = {k: np.zeros((n, n), dtype=np.int64) for k in names}
    kin = np.zeros((n, n), dtype=np.float64)
    for a in range(n):
        for b in range(n):
            x, y = codes[a], codes[b]
            v = (x != 3) & (y != 3)
            d = np.abs(x - y)
            vals = (int(v.sum()), int((v & (d == 2)).sum()), int((v & (d == 1)).sum()), int((v & (x == 1) & (y == 1)).sum()),
                    int((v & (x == 1)).sum()), int((v & (y == 1)).sum()))
            for k, val in zip(names, vals):
                out[k][a, b] = val
            m = min(vals[4], vals[5])
            kin[a, b] = float("nan") if m == 0 else 0.5 - (4 * vals[1] + vals[2]) / (4 * m)
    out["kinship"] = kin
    return out


def bit_equal(x, y):
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    nx, ny = np.isnan(x), np.isnan(y)
    return x.shape == y.shape and np.array_equal(nx, ny) and np.array_equal(x[~nx].view(np.uint64), y[~ny].view(np.uint64))


def _pops():
    for miss in (0.0, 0.03, 0.2):
        yield f"miss{miss}", make_population(23, 700, seed=31, missing_rate=miss)[0]
    yield "multi", add_multi_allelic(make_population(30, 500, seed=32, missing_rate=0.01)[0], 60, seed=33)
    yield "one-genome", make_population(1, 90, seed=34, missing_rate=0.1)[0]
    yield "N64", make_population(64, 300, seed=35, missing_rate=0.05)[0]


@pytest.mark.parametrize("name,pop", list(_pops()), ids=[n for n, _ in _pops()])
def test_oracle_matches_naive_loop(name, pop):
    want = naive_king(pop)
    got = K.king(pop)
    for k in ("n_valid", "ibs0", "ibs1", "het_het", "het_a", "het_b"):
        assert np.array_equal(got[k], want[k]), k
    assert bit_equal(got["kinship"], want["kinship"])
    # the diagonal is 0.5 wherever the genome has a heterozygous locus
    d = np.arange(pop.n_genomes)
    het = got["het_a"][d, d] > 0
    assert np.all(got["kinship"][d, d][het] == 0.5) and np.all(np.isnan(got["kinship"][d, d][~het]))


@pytest.mark.parametrize("miss,multi", [(0.0, False), (0.02, False), (0.1, True)])
def test_count_identities(miss, multi):
    pop, _ = make_population(90, 1500, seed=36, missing_rate=miss)
    if multi:
        add_multi_allelic(pop, 100, seed=37)
    k = K.king(pop)
    ibs = O.ibs(pop).astype(np.int64)
    assert np.array_equal(k["het_a"] + k["het_b"], k["ibs1"] + 2 * k["het_het"])
    assert np.array_equal(k["ibs0"], ibs[..., 0]) and np.array_equal(k["ibs1"], ibs[..., 1])
    assert np.array_equal(k["n_valid"], ibs[..., 3]) and np.array_equal(ibs[..., :3].sum(-1), k["n_valid"])
    assert np.array_equal(k["het_a"], k["het_b"].T) and bit_equal(k["kinship"], k["kinship"].T)


def test_degrees_at_the_bounds():
    up = np.nextafter
    cases = [(0.5, 0), (up(2 ** -1.5, 1), 0), (2 ** -1.5, 1), (up(2 ** -1.5, 0), 1), (2 ** -2.5, 1), (up(2 ** -2.5, 0), 2),
             (2 ** -3.5, 2), (up(2 ** -3.5, 0), 3), (2 ** -4.5, 3), (up(2 ** -4.5, 0), -1), (0.0, -1), (-0.3, -1), (np.nan, -1)]
    for k, deg in cases:
        assert king_degree(k) == deg, (k, deg)
    ks, degs = zip(*cases)
    assert np.array_equal(king_degree(np.array(ks)), np.array(degs, dtype=np.int8))
    assert king_degree(np.zeros((2, 3))).shape == (2, 3)


def test_pair_struct_layout():
    assert C.sizeof(capi.KingPair) == 40 and capi.KING_PAIR_DTYPE.itemsize == 40
    offsets = {"a": 0, "b": 4, "n_valid": 8, "ibs0": 12, "ibs1": 16, "het_het": 20, "het_a": 24, "het_b": 28, "kinship": 32}
    for name, off in offsets.items():
        assert getattr(capi.KingPair, name).offset == off
        assert capi.KING_PAIR_DTYPE.fields[name][1] == off


WORLD = 2


def _rank_pairs(rank):
    rng = np.random.default_rng(100 + rank)
    n = 5 if rank == 0 else 13                     # lists of different lengths
    p = np.zeros(n, dtype=capi.KING_PAIR_DTYPE)
    p["a"] = rng.integers(0, 50, n) + 100 * rank
    p["b"] = p["a"] + 1 + rng.integers(0, 50, n)
    p["ibs0"] = rng.integers(0, 1000, n)
    p["kinship"] = rng.random(n)
    return p


def _gather_worker(rank, port, tmp):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=WORLD)
    try:
        got = shards.gather_king_pairs(_rank_pairs(rank))
        want = np.concatenate([_rank_pairs(r) for r in range(WORLD)])
        want = want[np.lexsort((want["b"], want["a"]))]
        assert got.dtype == capi.KING_PAIR_DTYPE and got.tobytes() == want.tobytes()
        empty = shards.gather_king_pairs(np.zeros(0, dtype=capi.KING_PAIR_DTYPE))
        assert empty.shape == (0,)
        open(os.path.join(tmp, f"ok{rank}"), "w").close()
    finally:
        dist.destroy_process_group()


def test_gather_king_pairs_gloo(tmp_path):
    port = 31500 + os.getpid() % 2000
    mp.spawn(_gather_worker, args=(port, str(tmp_path)), nprocs=WORLD, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(WORLD))
