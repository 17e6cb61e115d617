"""ctypes wrapper over oracle/_build/libkgl_oracle.so and the reference harness. TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs; never from the
product package (kgl_gene_b200/).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "libkgl_oracle.so")
HARNESS_PATH = os.path.join(HERE, "_ref", "kgl_ref_harness")

ALGORITHMS = {"Simple": 0, "RitlandLocus": 1, "HallME": 2, "Loglikelihood": 3}

RESULT_DTYPE = np.dtype([  # kga::LocusResults field order (kga_analysis_inbreed_output.h:21-35)
    ("major_hetero_count", "<u8"), ("major_hetero_freq", "<f8"),
    ("minor_hetero_count", "<u8"), ("minor_hetero_freq", "<f8"),
    ("minor_homo_count", "<u8"), ("minor_homo_freq", "<f8"),
    ("major_homo_count", "<u8"), ("major_homo_freq", "<f8"),
    ("total_allele_count", "<u8"), ("inbred_allele_sum", "<f8"),
])

_lib = None


def build() -> None:
    subprocess.run(["make", "-s", "-C", HERE, "oracle"], check=True)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        _lib = C.CDLL(LIB_PATH)
        _lib.kgl_oracle_select_loci.restype = C.c_size_t
        _lib.kgl_oracle_threads.restype = C.c_int
    return _lib


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def select_loci(offsets, af_pop, lower=0, upper=10**9, spacing=0, count=10**9, min_af=0.0, max_af=1.0, mode=0):
    """RetrieveLociiVector restatement; returns (selected uint8 [L], last_index)."""
    offsets = np.ascontiguousarray(offsets, dtype=np.uint32)
    af_pop = np.ascontiguousarray(af_pop, dtype=np.float32)
    sel = np.zeros(offsets.shape[0], dtype=np.uint8)
    last = C.c_size_t(0)
    lib().kgl_oracle_select_loci(_p(offsets), _p(af_pop), C.c_size_t(offsets.shape[0]), C.c_uint64(lower), C.c_uint64(upper),
                                 C.c_uint64(spacing), C.c_uint64(count), C.c_double(min_af), C.c_double(max_af), C.c_int(mode),
                                 _p(sel), C.byref(last))
    return sel, int(last.value)


def set_multi(pop) -> None:
    """Hands the population's multi-allelic loci (or none) to the C restatement; every entry point below calls it."""
    if getattr(pop, "n_multi", 0):
        rows = np.ascontiguousarray(pop.multi_rows, dtype=np.uint32)
        af = np.ascontiguousarray(pop.multi_af, dtype=np.float32)
        cells = np.ascontiguousarray(pop.multi_cells, dtype=np.uint8)
        lib().kgl_oracle_set_multi(C.c_size_t(rows.shape[0]), _p(rows), _p(af), _p(cells), C.c_size_t(af.shape[0]),
                                   C.c_size_t(pop.n_genomes), C.c_size_t(pop.n_loci))
    else:
        lib().kgl_oracle_set_multi(C.c_size_t(0), None, None, None, C.c_size_t(0), C.c_size_t(0), C.c_size_t(0))


def select_all_pops(pop, lower=0, upper=10**9, spacing=0, count=10**9, min_af=0.0, max_af=1.0, mode=0):
    """uint8 [6, L] selection masks, one per super-population (multi-allelic loci included)."""
    set_multi(pop)
    lib().kgl_oracle_select_loci_pop.restype = C.c_size_t
    offsets = np.ascontiguousarray(pop.offsets, dtype=np.uint32)
    out = []
    for k in range(pop.af.shape[0]):
        af_pop = np.ascontiguousarray(pop.af[k], dtype=np.float32)
        sel = np.zeros(offsets.shape[0], dtype=np.uint8)
        lib().kgl_oracle_select_loci_pop(_p(offsets), _p(af_pop), C.c_size_t(offsets.shape[0]), C.c_size_t(k), C.c_uint64(lower),
                                         C.c_uint64(upper), C.c_uint64(spacing), C.c_uint64(count), C.c_double(min_af),
                                         C.c_double(max_af), C.c_int(mode), _p(sel), None)
        out.append(sel)
    return np.stack(out)


def inbreed(pop, selected, algorithm: str, start=None, sweeps: int = 50, genomes=None, compensated: bool = False) -> np.ndarray:
    """genomes: optional list of genome indices -- the result then has one row per listed genome (start stays indexed by genome).
    compensated: the per-genome sums over the loci are added with Neumaier's compensation instead of in the reference's order
    and precision (double, locus by locus), whose rounding grows with the number of loci."""
    set_multi(pop)
    gl = None if genomes is None else np.ascontiguousarray(genomes, dtype=np.uint32)
    n_some = pop.n_genomes if gl is None else gl.shape[0]
    out = np.zeros(n_some, dtype=RESULT_DTYPE)
    packed = np.ascontiguousarray(pop.packed)
    af = np.ascontiguousarray(pop.af, dtype=np.float32)
    selected = np.ascontiguousarray(selected, dtype=np.uint8)
    sp = np.ascontiguousarray(pop.superpop, dtype=np.uint8)
    st = None if start is None else np.ascontiguousarray(start, dtype=np.float64)
    lib().kgl_oracle_set_compensated_sums(C.c_int(int(compensated)))
    try:
        lib().kgl_oracle_inbreed_some(_p(packed), C.c_size_t(pop.row_bytes), C.c_size_t(pop.n_genomes), C.c_size_t(pop.n_loci),
                                      _p(af), C.c_size_t(af.shape[0]), _p(selected), _p(sp), C.c_int(int(pop.unphased)),
                                      C.c_int(ALGORITHMS[algorithm]), None if st is None else _p(st), C.c_int(sweeps),
                                      None if gl is None else _p(gl), C.c_size_t(n_some), _p(out))
    finally:
        lib().kgl_oracle_set_compensated_sums(C.c_int(0))
    return out


def loglik_grid(pop, selected, grid) -> np.ndarray:
    set_multi(pop)
    grid = np.ascontiguousarray(grid, dtype=np.float64)
    out = np.zeros((pop.n_genomes, grid.shape[0]), dtype=np.float64)
    packed = np.ascontiguousarray(pop.packed)
    af = np.ascontiguousarray(pop.af, dtype=np.float32)
    selected = np.ascontiguousarray(selected, dtype=np.uint8)
    sp = np.ascontiguousarray(pop.superpop, dtype=np.uint8)
    lib().kgl_oracle_loglik_grid(_p(packed), C.c_size_t(pop.row_bytes), C.c_size_t(pop.n_genomes), C.c_size_t(pop.n_loci),
                                 _p(af), C.c_size_t(af.shape[0]), _p(selected), _p(sp), C.c_int(int(pop.unphased)),
                                 _p(grid), C.c_size_t(grid.shape[0]), _p(out))
    return out


def allele_count(pop):
    lc = np.zeros((pop.n_loci, 4), dtype=np.uint32)
    gc = np.zeros((pop.n_genomes, 4), dtype=np.uint64)
    packed = np.ascontiguousarray(pop.packed)
    lib().kgl_oracle_allele_count(_p(packed), C.c_size_t(pop.row_bytes), C.c_size_t(pop.n_genomes), C.c_size_t(pop.n_loci), _p(lc), _p(gc))
    return lc, gc


def ibs(pop) -> np.ndarray:
    out = np.zeros((pop.n_genomes, pop.n_genomes, 4), dtype=np.uint32)
    packed = np.ascontiguousarray(pop.packed)
    lib().kgl_oracle_ibs(_p(packed), C.c_size_t(pop.row_bytes), C.c_size_t(pop.n_genomes), C.c_size_t(pop.n_loci), _p(out))
    return out


def ibs_band_popcount(pop, row_begin: int, row_end: int) -> np.ndarray:
    """IBS of genomes [row_begin, row_end) against all genomes by the popcount restatement (scale checker)."""
    out = np.zeros((row_end - row_begin, pop.n_genomes, 4), dtype=np.uint32)
    packed = np.ascontiguousarray(pop.packed)
    lib().kgl_oracle_ibs_band_popcount(_p(packed), C.c_size_t(pop.row_bytes), C.c_size_t(pop.n_genomes), C.c_size_t(pop.n_loci),
                                       C.c_size_t(row_begin), C.c_size_t(row_end), _p(out))
    return out


def fws_bins(pop, af_col: int, bins, present_only=True):
    """CalcFWS restated on the flat matrix with plain numpy loops (kga_PfEMP/kga_analysis_PfEMP_FWS.cpp:15-101; filter
    kgl_variant_filter_Pf7.cpp:20-66): returns (counts uint64[n_bins][N][4], rows uint64[n_bins])."""
    codes = pop.codes()                                  # [L][N]
    af = pop.af[af_col].astype(np.float64)
    present = ((codes == 1) | (codes == 2)).any(axis=1)
    out = np.zeros((len(bins), pop.n_genomes, 4), dtype=np.uint64)
    rows = np.zeros(len(bins), dtype=np.uint64)
    for b, (lo, hi) in enumerate(bins):
        with np.errstate(invalid="ignore"):
            m = ~np.isnan(af) & (af >= lo) & ~(af >= hi)
        if present_only:
            m &= present
        rows[b] = int(m.sum())
        sub = codes[m]
        for c in range(4):
            out[b, :, c] = (sub == c).sum(axis=0)
    if getattr(pop, "n_multi", 0):
        # every listed allele of a multi-allelic locus is a variant with its own AF (its element of the Number=A list,
        # kgl_variant_filter_Pf7.cpp:22-48); a genome has 0, 1 or 2 copies of it (kgl_variant_db_variant.cpp:73-103). Cells with
        # more than two variants (0xFF) do not record which alleles: no copy (flattener contract).
        copies = multi_allele_copies(pop)                  # [M][3][N]
        for b, (lo, hi) in enumerate(bins):
            for m_i in range(pop.n_multi):
                for a in range(3):
                    v = float(pop.multi_af[af_col, m_i, a])
                    if np.isnan(v) or not (v >= lo and not v >= hi):
                        continue
                    if present_only and not (copies[m_i, a] > 0).any():
                        continue
                    rows[b] += np.uint64(1)
                    for c in range(3):
                        out[b, :, c] += (copies[m_i, a] == c).astype(np.uint64)
    return out, rows


def hetero_homo(pop, other_allele_entries: int = 1) -> np.ndarray:
    """HeteroHomoZygous::updateVariantAnalysisType (kga_PfEMP/kga_analysis_PfEMP_heterozygous.cpp:61-105) per genome over every
    offset: uint64[N][7] = total, snp, indel, homMinor, hetMinor, hetRefMinor, homRef. One entry at an offset ->
    heterozygous_reference_minor_alleles_; otherwise homozygous_minor_alleles_ += distinct alleles, heterozygous_minor_alleles_ +=
    alleles that occur once. A 0xFF side cell stands for three entries, two of one allele and one of another (what the reference
    harness builds for it)."""
    codes = pop.codes()
    out = np.zeros((pop.n_genomes, 7), dtype=np.uint64)
    is_multi = np.zeros(pop.n_loci, dtype=bool)
    if getattr(pop, "n_multi", 0):
        is_multi[pop.multi_rows] = True
    for g in range(pop.n_genomes):
        col = codes[~is_multi, g]
        n1, n2, n3 = int((col == 1).sum()), int((col == 2).sum()), int((col == 3).sum()) * (1 if other_allele_entries else 0)
        single = same = diff = many = 0
        for m in range(getattr(pop, "n_multi", 0)):
            cell = int(pop.multi_cells[m, g])
            if cell == 0:
                continue
            if cell == 0xFF:
                many += 1
            elif cell >> 4 == 0:
                single += 1
            elif cell >> 4 == cell & 15:
                same += 1
            else:
                diff += 1
        total = n1 + 2 * n2 + n3 + single + 2 * same + 2 * diff + 3 * many
        out[g] = (total, total, 0, n2 + same + 2 * diff + 2 * many, 2 * diff + many, n1 + n3 + single, 0)
    return out


def multi_allele_copies(pop) -> np.ndarray:
    """int64[M][3][N]: copies of allele slot a genome g carries at multi-allelic locus m (side cells: low nibble = first variant's
    slot + 1, high nibble = the second's, 0xFF = more than two variants, counted as none)."""
    cells = pop.multi_cells.astype(np.int64)
    out = np.zeros((pop.n_multi, 3, pop.n_genomes), dtype=np.int64)
    for a in range(3):
        out[:, a, :] = ((cells & 15) == a + 1).astype(np.int64) + ((cells >> 4) == a + 1).astype(np.int64)
    out[:, :, :] *= (cells != 0xFF)[:, None, :]
    return out


def gram(pop, af_pop=None):
    """(gram int32 [N][N], grm float64 [N][N] or None): dosage Gram matrix and its centred form for one AF column."""
    n = pop.n_genomes
    g = np.zeros((n, n), dtype=np.int32)
    packed = np.ascontiguousarray(pop.packed)
    if af_pop is None:
        lib().kgl_oracle_gram(_p(packed), C.c_size_t(pop.row_bytes), C.c_size_t(n), C.c_size_t(pop.n_loci), None, _p(g), None)
        return g, None
    af_pop = np.ascontiguousarray(af_pop, dtype=np.float32)
    c = np.zeros((n, n), dtype=np.float64)
    lib().kgl_oracle_gram(_p(packed), C.c_size_t(pop.row_bytes), C.c_size_t(n), C.c_size_t(pop.n_loci), _p(af_pop), _p(g), _p(c))
    return g, c


def synth_genotypes(seed, n_genomes, n_loci, af, superpop, inbreeding, missing_rate=0.001, locus_base=0) -> np.ndarray:
    rb = 16 * ((n_genomes + 63) // 64)
    packed = np.zeros((n_loci, rb), dtype=np.uint8)
    af = np.ascontiguousarray(af, dtype=np.float32)
    sp = np.ascontiguousarray(superpop, dtype=np.uint8)
    fi = np.ascontiguousarray(inbreeding, dtype=np.float64)
    lib().kgl_oracle_synth_genotypes(C.c_uint64(seed), C.c_size_t(n_genomes), C.c_size_t(n_loci), C.c_size_t(locus_base), _p(af),
                                     C.c_size_t(af.shape[0]), _p(sp), _p(fi), C.c_double(missing_rate), _p(packed), C.c_size_t(rb))
    return packed


def threads() -> int:
    return int(lib().kgl_oracle_threads())


def have_reference_harness() -> bool:
    return os.path.exists(HARNESS_PATH) and os.access(HARNESS_PATH, os.X_OK)


def run_reference(pop, algos=("Simple", "RitlandLocus", "HallME", "Loglikelihood"), spacing=0, min_af=0.0, max_af=1.0,
                  lower=0, upper=10**9, grid=0, threads=0, variantdb=True, seed=None, repeat=1, timeout=3600, fws=False, count=None):
    """Runs the reference's own code (oracle/_ref/kgl_ref_harness) on `pop`; returns the dumped arrays."""
    from kgl_gene_b200.flatfile import read_tensors
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "in.flat"), os.path.join(d, "out.tens")
        pop.write(fin)
        cmd = [HARNESS_PATH, fin, fout, "--algos", ",".join(algos), "--spacing", str(spacing), "--min-af", repr(float(min_af)),
               "--max-af", repr(float(max_af)), "--lower", str(lower), "--upper", str(upper), "--grid", str(grid), "--threads", str(threads)]
        if not variantdb:
            cmd.append("--no-variantdb")
        if fws:
            cmd.append("--fws")
        if count is not None:
            cmd += ["--count", str(int(count))]
        if seed is not None:
            cmd += ["--seed", str(int(seed))]
        if repeat > 1:
            cmd += ["--repeat", str(int(repeat))]
        env = dict(os.environ, KGL_REF_LOG=os.path.join(d, "ref.log"))
        proc = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        if proc.returncode != 0:
            raise RuntimeError(f"reference harness failed ({proc.returncode}): {proc.stderr[-2000:]}")
        out = read_tensors(fout)
        out["_stderr"] = proc.stderr
        return out
