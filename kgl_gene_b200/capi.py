"""ctypes binding of the C ABI (include/kgl_b200.h). There is no fallback: if libkgl_b200.so is missing or no sm_100 GPU
is usable, construction raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .shards import tiles_of_rank

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkgl_b200.so")

ALGORITHMS = {"Simple": 0, "RitlandLocus": 1, "HallME": 2, "Loglikelihood": 3}   # kga_analysis_inbreed_calc.h:103-106

RESULT_DTYPE = np.dtype([  # kgl_b200_locus_results == kga::LocusResults field order
    ("major_hetero_count", "<u8"), ("major_hetero_freq", "<f8"),
    ("minor_hetero_count", "<u8"), ("minor_hetero_freq", "<f8"),
    ("minor_homo_count", "<u8"), ("minor_homo_freq", "<f8"),
    ("major_homo_count", "<u8"), ("major_homo_freq", "<f8"),
    ("total_allele_count", "<u8"), ("inbred_allele_sum", "<f8"),
])

class KingPair(C.Structure):
    """kgl_b200_king_pair (include/kgl_b200.h), 40 bytes."""
    _fields_ = [("a", C.c_uint32), ("b", C.c_uint32), ("n_valid", C.c_uint32), ("ibs0", C.c_uint32), ("ibs1", C.c_uint32),
                ("het_het", C.c_uint32), ("het_a", C.c_uint32), ("het_b", C.c_uint32), ("kinship", C.c_double)]


KING_PAIR_DTYPE = np.dtype([(name, "<f8" if ctype is C.c_double else "<u4") for name, ctype in KingPair._fields_])

KGL_B200_ERR_NOMEM = 5

EXPORTS = [
    "kgl_b200_version", "kgl_b200_device_count", "kgl_b200_create", "kgl_b200_destroy", "kgl_b200_last_error",
    "kgl_b200_set_stream", "kgl_b200_synchronize", "kgl_b200_upload_genotypes", "kgl_b200_upload_loci",
    "kgl_b200_set_genome_superpop", "kgl_b200_upload_multi_allelic", "kgl_b200_run_multi_allele_count", "kgl_b200_set_unphased", "kgl_b200_select_loci", "kgl_b200_set_locus_selection",
    "kgl_b200_get_locus_selection", "kgl_b200_count_loci", "kgl_b200_set_locus_filter", "kgl_b200_synth_genotypes", "kgl_b200_download_genotypes", "kgl_b200_run_allele_count",
    "kgl_b200_run_inbreed", "kgl_b200_inbreed_used_moment_tables", "kgl_b200_run_count_and_inbreed", "kgl_b200_run_loglik_grid", "kgl_b200_run_ibs", "kgl_b200_run_king", "kgl_b200_run_king_pairs", "kgl_b200_run_pca", "kgl_b200_run_grm_product", "kgl_b200_run_ld_pairs", "kgl_b200_run_ld_prune", "kgl_b200_run_group_counts", "kgl_b200_run_fst", "kgl_b200_run_hardy", "kgl_b200_run_variant_qc", "kgl_b200_last_hardy_terms", "kgl_b200_ibs_tile_grid", "kgl_b200_enqueue_ibs_tile_list", "kgl_b200_run_ibs_tile_list", "kgl_b200_set_ibs_tensor_cores", "kgl_b200_ibs_used_tensor_cores", "kgl_b200_run_ibs_tiles",
    "kgl_b200_run_binned_genome_counts", "kgl_b200_run_hetero_homo", "kgl_b200_location_fis", "kgl_b200_run_gram", "kgl_b200_run_grm", "kgl_b200_enqueue_gram", "kgl_b200_last_gram_kernel_ms", "kgl_b200_enqueue_gram_tiles", "kgl_b200_gram_buffer", "kgl_b200_fetch_gram",
    "kgl_b200_enqueue_ibs_tiles", "kgl_b200_ibs_tiles_buffer", "kgl_b200_ibs_timer_reset", "kgl_b200_ibs_timer_read",
    "kgl_b200_enqueue_count_and_inbreed", "kgl_b200_flush", "kgl_b200_launch_count", "kgl_b200_last_stream_kernel_ms",
    "kgl_b200_inbreed_begin", "kgl_b200_inbreed_accumulate", "kgl_b200_inbreed_partials_buffer", "kgl_b200_inbreed_update",
    "kgl_b200_inbreed_fetch", "kgl_b200_kernel_timer_reset", "kgl_b200_kernel_timer_read", "kgl_b200_fetch_locus_counts",
    "kgl_b200_peer_export", "kgl_b200_peer_attach", "kgl_b200_peer_set_timeout_ms", "kgl_b200_enqueue_count_and_inbreed_peer",
]


class InbreedOptions(C.Structure):
    _fields_ = [("hall_start", C.POINTER(C.c_double)), ("hall_sweeps", C.c_int32), ("ll_tolerance", C.c_double),
                ("ll_max_iterations", C.c_int32), ("count_loci", C.c_int32), ("exact_sweeps", C.c_int32), ("moments_on_cuda_cores", C.c_int32), ("sweep_by_sweep", C.c_int32)]


class PcaOptions(C.Structure):
    """kgl_b200_pca_options (include/kgl_b200.h), 24 bytes; zero = the defaults."""
    _fields_ = [("keep", C.c_void_p), ("n_components", C.c_uint32), ("iterations", C.c_uint32), ("seed", C.c_uint64)]


class LdOptions(C.Structure):
    """kgl_b200_ld_options (include/kgl_b200.h), 16 bytes; window limits of 0 mean no limit (not both)."""
    _fields_ = [("keep", C.c_void_p), ("window_loci", C.c_uint32), ("window_bp", C.c_uint32)]


class LdPair(C.Structure):
    """kgl_b200_ld_pair (include/kgl_b200.h), 24 bytes."""
    _fields_ = [("a", C.c_uint32), ("b", C.c_uint32), ("n_valid", C.c_uint32), ("reserved", C.c_uint32), ("r2", C.c_double)]


LD_PAIR_DTYPE = np.dtype([(name, "<f8" if ctype is C.c_double else "<u4") for name, ctype in LdPair._fields_])

KGL_B200_MAX_POP = 6        # super-populations (include/kgl_b200.h); the groups of group_counts / fst with group=None
FST_METHODS = {"hudson": 0, "weir_cockerham": 1}


class FstOptions(C.Structure):
    """kgl_b200_fst_options (include/kgl_b200.h), 56 bytes; zero = Hudson, the super-population labels, every locus and pair."""
    _fields_ = [("group", C.c_void_p), ("n_groups", C.c_uint32), ("keep", C.c_void_p), ("method", C.c_uint32),
                ("n_pairs", C.c_uint32), ("pairs", C.c_void_p), ("window_bp", C.c_uint64), ("step_bp", C.c_uint64)]


class HardyOptions(C.Structure):
    """kgl_b200_hardy_options (include/kgl_b200.h), 16 bytes; zero = p (not mid-p) per super-population."""
    _fields_ = [("group", C.c_void_p), ("n_groups", C.c_uint32), ("midp", C.c_uint32)]


class QcOptions(C.Structure):
    """kgl_b200_qc_options (include/kgl_b200.h), 48 bytes; zero = no filter."""
    _fields_ = [("keep", C.c_void_p), ("min_call_rate", C.c_double), ("min_maf", C.c_double), ("min_hwe_p", C.c_double),
                ("group", C.c_void_p), ("n_groups", C.c_uint32), ("midp", C.c_uint32)]


class KglError(RuntimeError):
    pass


_lib = None


def load_library() -> C.CDLL:
    """Loads libkgl_b200.so; raises if it has not been built (python -m kgl_gene_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KglError(f"{LIB_PATH} is missing: build it with `python kgl_gene_b200/build.py` (nvcc, sm_100a). "
                           "There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        lib.kgl_b200_version.restype = C.c_char_p
        lib.kgl_b200_last_error.restype = C.c_char_p
        lib.kgl_b200_last_error.argtypes = [C.c_void_p]
        lib.kgl_b200_launch_count.restype = C.c_uint64
        lib.kgl_b200_launch_count.argtypes = [C.c_void_p]
        lib.kgl_b200_last_stream_kernel_ms.restype = C.c_float
        lib.kgl_b200_last_stream_kernel_ms.argtypes = [C.c_void_p]
        lib.kgl_b200_last_gram_kernel_ms.restype = C.c_float
        lib.kgl_b200_last_gram_kernel_ms.argtypes = [C.c_void_p]
        lib.kgl_b200_destroy.restype = None
        lib.kgl_b200_last_hardy_terms.restype = C.c_uint64
        lib.kgl_b200_last_hardy_terms.argtypes = [C.c_void_p]
        lib.kgl_b200_destroy.argtypes = [C.c_void_p]
        _lib = lib
    return _lib


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def location_fis(hetero_homo: np.ndarray, location_members: list, city_of_genome, country_of_genome, qc_pass=None,
                 min_location_samples: int = 20) -> np.ndarray:
    """kgl_b200_location_fis: Wright's F_IS of every genome against its location aggregate (UpdateSampleLocation)."""
    lib = load_library()
    hh = np.ascontiguousarray(hetero_homo, dtype=np.uint64)
    n = hh.shape[0]
    begin = np.zeros(len(location_members) + 1, dtype=np.uint64)
    begin[1:] = np.cumsum([len(m) for m in location_members])
    members = np.ascontiguousarray(np.concatenate([np.asarray(m, dtype=np.uint32) for m in location_members]) if location_members else np.zeros(0), dtype=np.uint32)
    city = np.ascontiguousarray(city_of_genome, dtype=np.uint32)
    country = np.ascontiguousarray(country_of_genome, dtype=np.uint32)
    qc = None if qc_pass is None else np.ascontiguousarray(qc_pass, dtype=np.uint8)
    out = np.zeros(n, dtype=np.float64)
    rc = lib.kgl_b200_location_fis(C.c_uint64(n), _ptr(hh), C.c_uint32(len(location_members)), _ptr(begin), _ptr(members), _ptr(city),
                                   _ptr(country), _ptr(qc), C.c_uint32(min_location_samples), _ptr(out))
    if rc != 0:
        raise KglError(f"location_fis failed [{rc}]")
    return out


class KglB200:
    """One context = one GPU. Mirrors the call order of the reference plugin: upload the flattened population
    (fileReadAnalysis), select loci per window and run an estimator (iterationAnalysis)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.kgl_b200_create(C.c_int(device), C.byref(h))
        if rc != 0:
            raise KglError(f"kgl_b200_create({device}) failed [{rc}]: {self.lib.kgl_b200_last_error(None).decode()}")
        self.h = h
        self.n_genomes = self.n_loci = 0
        self._offsets = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.kgl_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise KglError(f"{what} failed [{rc}]: {self.lib.kgl_b200_last_error(self.h).decode()}")

    # ---- upload ----
    def set_stream(self, cuda_stream: int | None):
        self._check(self.lib.kgl_b200_set_stream(self.h, C.c_void_p(cuda_stream or 0)), "set_stream")

    def synchronize(self):
        self._check(self.lib.kgl_b200_synchronize(self.h), "synchronize")

    def upload_genotypes(self, packed: np.ndarray, n_genomes: int):
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        n_loci, row_bytes = packed.shape
        self._keep_packed = packed
        self._check(self.lib.kgl_b200_upload_genotypes(self.h, C.c_uint64(n_genomes), C.c_uint64(n_loci), C.c_uint64(row_bytes),
                                                       _ptr(packed)), "upload_genotypes")
        self.n_genomes, self.n_loci = int(n_genomes), int(n_loci)

    def upload_genotypes_ptr(self, host_ptr: int, n_genomes: int, n_loci: int, row_bytes: int):
        """Raw host pointer variant (e.g. a pinned torch tensor's data_ptr())."""
        self._check(self.lib.kgl_b200_upload_genotypes(self.h, C.c_uint64(n_genomes), C.c_uint64(n_loci), C.c_uint64(row_bytes),
                                                       C.c_void_p(host_ptr)), "upload_genotypes")
        self.n_genomes, self.n_loci = int(n_genomes), int(n_loci)

    def upload_loci(self, af: np.ndarray, offsets: np.ndarray | None = None):
        af = np.ascontiguousarray(af, dtype=np.float32)
        off = None if offsets is None else np.ascontiguousarray(offsets, dtype=np.uint32)
        self._check(self.lib.kgl_b200_upload_loci(self.h, C.c_uint64(af.shape[1]), C.c_uint32(af.shape[0]), _ptr(af), _ptr(off)),
                    "upload_loci")
        self.n_loci = int(af.shape[1])
        self._offsets = off

    def set_genome_superpop(self, superpop: np.ndarray):
        sp = np.ascontiguousarray(superpop, dtype=np.uint8)
        self._check(self.lib.kgl_b200_set_genome_superpop(self.h, C.c_uint64(sp.shape[0]), _ptr(sp)), "set_genome_superpop")
        self.n_genomes = int(sp.shape[0])

    def set_unphased(self, unphased: bool):
        self._check(self.lib.kgl_b200_set_unphased(self.h, C.c_int(int(bool(unphased)))), "set_unphased")

    def upload_multi_allelic(self, rows, af, cells):
        """Loci with several alternate alleles (FlatPopulation.multi_*); rows=None clears them."""
        if rows is None or len(rows) == 0:
            self._check(self.lib.kgl_b200_upload_multi_allelic(self.h, C.c_uint64(0), None, None, None), "upload_multi_allelic")
            return
        r = np.ascontiguousarray(rows, dtype=np.uint32)
        a = np.ascontiguousarray(af, dtype=np.float32)
        c = np.ascontiguousarray(cells, dtype=np.uint8)
        assert a.shape[1:] == (r.shape[0], 3) and c.shape == (r.shape[0], self.n_genomes)
        self._check(self.lib.kgl_b200_upload_multi_allelic(self.h, C.c_uint64(r.shape[0]), _ptr(r), _ptr(a), _ptr(c)), "upload_multi_allelic")

    def multi_allele_count(self, n_multi: int) -> np.ndarray:
        out = np.zeros((n_multi, 3, 3), dtype=np.uint32)
        self._check(self.lib.kgl_b200_run_multi_allele_count(self.h, _ptr(out)), "run_multi_allele_count")
        return out

    def upload_population(self, pop):
        """pop: kgl_gene_b200.flatfile.FlatPopulation."""
        self.upload_genotypes(pop.packed, pop.n_genomes)
        self.upload_loci(pop.af, pop.offsets)
        self.set_genome_superpop(pop.superpop)
        self.set_unphased(pop.unphased)
        if getattr(pop, "n_multi", 0):
            self.upload_multi_allelic(pop.multi_rows, pop.multi_af, pop.multi_cells)

    def select_loci(self, lower=0, upper=10**9, spacing=0, min_af=0.0, max_af=1.0) -> np.ndarray:
        counts = np.zeros(6, dtype=np.uint64)
        self._check(self.lib.kgl_b200_select_loci(self.h, C.c_uint64(lower), C.c_uint64(upper), C.c_uint64(spacing),
                                                  C.c_double(min_af), C.c_double(max_af), _ptr(counts)), "select_loci")
        return counts

    def count_loci(self, pop=5, lower=0, spacing=0, count=1000, min_af=0.0, max_af=1.0):
        """RetrieveLociiVector::getLociiCount: (loci found <= count, offset of the last one)."""
        n, last = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.kgl_b200_count_loci(self.h, C.c_uint32(pop), C.c_uint64(lower), C.c_uint64(spacing), C.c_uint64(count),
                                                 C.c_double(min_af), C.c_double(max_af), C.byref(n), C.byref(last)), "count_loci")
        return int(n.value), int(last.value)

    def set_locus_filter(self, keep):
        if keep is None:
            self._check(self.lib.kgl_b200_set_locus_filter(self.h, C.c_uint64(0), None), "set_locus_filter")
            return
        k = np.ascontiguousarray(keep, dtype=np.uint8)
        self._check(self.lib.kgl_b200_set_locus_filter(self.h, C.c_uint64(k.shape[0]), _ptr(k)), "set_locus_filter")

    def set_locus_selection(self, selected_bits: np.ndarray):
        s = np.ascontiguousarray(selected_bits, dtype=np.uint8)
        self._check(self.lib.kgl_b200_set_locus_selection(self.h, C.c_uint64(s.shape[0]), _ptr(s)), "set_locus_selection")

    def get_locus_selection(self) -> np.ndarray:
        s = np.zeros(self.n_loci, dtype=np.uint8)
        self._check(self.lib.kgl_b200_get_locus_selection(self.h, C.c_uint64(s.shape[0]), _ptr(s)), "get_locus_selection")
        return s

    def synth_genotypes(self, seed: int, n_genomes: int, n_loci: int, inbreeding: np.ndarray, missing_rate=0.001, locus_base=0):
        f = np.ascontiguousarray(inbreeding, dtype=np.float64)
        self._check(self.lib.kgl_b200_synth_genotypes(self.h, C.c_uint64(seed), C.c_uint64(n_genomes), C.c_uint64(n_loci),
                                                      C.c_uint64(locus_base), _ptr(f), C.c_double(missing_rate)), "synth_genotypes")
        self.n_genomes, self.n_loci = int(n_genomes), int(n_loci)

    def download_genotypes(self) -> np.ndarray:
        rb = 16 * ((self.n_genomes + 63) // 64)
        out = np.zeros((self.n_loci, rb), dtype=np.uint8)
        self._check(self.lib.kgl_b200_download_genotypes(self.h, C.c_uint64(out.nbytes), _ptr(out)), "download_genotypes")
        return out

    # ---- hot path ----
    def allele_count(self, want_loci=True, want_genomes=True):
        lc = np.zeros((self.n_loci, 4), dtype=np.uint32) if want_loci else None
        gc = np.zeros((self.n_genomes, 4), dtype=np.uint64) if want_genomes else None
        self._check(self.lib.kgl_b200_run_allele_count(self.h, _ptr(lc), _ptr(gc)), "run_allele_count")
        return lc, gc

    def inbreed(self, algorithm: str, hall_start=None, hall_sweeps: int = 0, ll_tolerance: float = 0.0, ll_max_iterations: int = 0,
                exact_sweeps: bool = False, moments_on_cuda_cores: bool = False, sweep_by_sweep: bool = False):
        out = np.zeros(self.n_genomes, dtype=RESULT_DTYPE)
        opt = InbreedOptions()
        opt.sweep_by_sweep = int(bool(sweep_by_sweep))
        opt.exact_sweeps = int(bool(exact_sweeps))
        opt.moments_on_cuda_cores = int(bool(moments_on_cuda_cores))
        start = None
        if hall_start is not None:
            start = np.ascontiguousarray(hall_start, dtype=np.float64)
            opt.hall_start = start.ctypes.data_as(C.POINTER(C.c_double))
        opt.hall_sweeps, opt.ll_tolerance, opt.ll_max_iterations = int(hall_sweeps), float(ll_tolerance), int(ll_max_iterations)
        self._check(self.lib.kgl_b200_run_inbreed(self.h, C.c_int(ALGORITHMS[algorithm]), C.byref(opt), _ptr(out)), f"run_inbreed({algorithm})")
        return out

    def used_moment_tables(self) -> int:
        """Sweeps of the last HallME / Loglikelihood run: 0 exact kernels, 1 moment tables built on the CUDA cores, 2 on the tensor cores."""
        return int(self.lib.kgl_b200_inbreed_used_moment_tables(self.h))

    def count_and_inbreed(self, want_loci=True):
        lc = np.zeros((self.n_loci, 4), dtype=np.uint32) if want_loci else None
        out = np.zeros(self.n_genomes, dtype=RESULT_DTYPE)
        self._check(self.lib.kgl_b200_run_count_and_inbreed(self.h, _ptr(lc), _ptr(out)), "run_count_and_inbreed")
        return lc, out

    def count_and_inbreed_into(self, lc_ptr: int, out_ptr: int):
        self._check(self.lib.kgl_b200_run_count_and_inbreed(self.h, C.c_void_p(lc_ptr), C.c_void_p(out_ptr)), "run_count_and_inbreed")

    def enqueue_count_and_inbreed(self):
        self._check(self.lib.kgl_b200_enqueue_count_and_inbreed(self.h), "enqueue_count_and_inbreed")

    def flush(self):
        """Orders the context stream after everything enqueued so far (the tail of the last pass runs on a side stream)."""
        self._check(self.lib.kgl_b200_flush(self.h), "flush")

    def loglik_grid(self, grid) -> np.ndarray:
        grid = np.ascontiguousarray(grid, dtype=np.float64)
        out = np.zeros((self.n_genomes, grid.shape[0]), dtype=np.float64)
        self._check(self.lib.kgl_b200_run_loglik_grid(self.h, _ptr(grid), C.c_uint64(grid.shape[0]), _ptr(out)), "run_loglik_grid")
        return out

    def ibs(self, row_begin=0, row_end=None) -> np.ndarray:
        row_end = self.n_genomes if row_end is None else row_end
        out = np.zeros((row_end - row_begin, self.n_genomes, 4), dtype=np.uint32)
        self._check(self.lib.kgl_b200_run_ibs(self.h, C.c_uint64(row_begin), C.c_uint64(row_end), _ptr(out)), "run_ibs")
        return out

    def king(self, row_begin=0, row_end=None) -> np.ndarray:
        """KING-robust kinship float64[row_end - row_begin][N] of genomes [row_begin, row_end) against all genomes."""
        row_end = self.n_genomes if row_end is None else row_end
        out = np.zeros((row_end - row_begin, self.n_genomes), dtype=np.float64)
        self._check(self.lib.kgl_b200_run_king(self.h, C.c_uint64(row_begin), C.c_uint64(row_end), _ptr(out)), "run_king")
        return out

    def king_pairs(self, min_kinship: float, coords=None, capacity: int = 1 << 22) -> np.ndarray:
        """Pairs a < b with KING kinship >= min_kinship inside the 64 x 64 tiles `coords` (uint32[n][2], tile row <= tile column;
        None = the whole upper triangle), sorted by (a, b): a KING_PAIR_DTYPE array. Retries once with the exact capacity; a retry
        computes every tile again, so the default (4 M pairs, 168 MB of host buffer that is only touched as far as it is filled,
        52 B per pair on the device, never more than the tiles hold) is sized for related-pair lists of biobank populations."""
        if coords is not None:
            coords = np.ascontiguousarray(coords, dtype=np.uint32).reshape(-1, 2)
            if coords.shape[0] == 0:
                return np.zeros(0, dtype=KING_PAIR_DTYPE)
        n_coords = 0 if coords is None else coords.shape[0]
        n = C.c_uint64(0)
        for attempt in range(2):
            out = np.zeros(max(int(capacity), 1), dtype=KING_PAIR_DTYPE)
            rc = self.lib.kgl_b200_run_king_pairs(self.h, C.c_uint64(n_coords), _ptr(coords), C.c_double(min_kinship),
                                                  C.c_uint64(capacity), _ptr(out), C.byref(n))
            if rc == KGL_B200_ERR_NOMEM and attempt == 0:
                capacity = int(n.value)
                continue
            self._check(rc, "run_king_pairs")
            break
        return out[: n.value].copy()

    def _keep(self, keep):
        if keep is None:
            return None
        k = np.ascontiguousarray(keep, dtype=np.uint8)
        if k.shape != (self.n_loci,):
            raise ValueError(f"keep must be uint8[{self.n_loci}]")
        return k

    def pca(self, k: int = 10, iterations: int = 10, seed: int = 0, keep=None, loadings: bool = False):
        """Top-k principal components of the variance-standardised genotype matrix (PLINK 2 --pca approx; k = 0 and
        iterations = 0 mean 10): a dict with eigenvalues float64[k] (descending), scores float64[N][k] (unit eigenvectors, largest
        entry positive), n_loci_used and, with loadings=True, loadings float64[L][k]."""
        k = int(k) or 10                                          # 0 = the default of the C ABI, which the buffers must match
        if k < 0 or iterations < 0:
            raise ValueError("k and iterations must be >= 0")
        kp = self._keep(keep)
        opt = PcaOptions(keep=None if kp is None else kp.ctypes.data, n_components=k, iterations=int(iterations), seed=int(seed))
        ev = np.zeros(k, dtype=np.float64)
        sc = np.zeros((self.n_genomes, k), dtype=np.float64)
        ld = np.zeros((self.n_loci, k), dtype=np.float64) if loadings else None
        m = C.c_uint64(0)
        self._check(self.lib.kgl_b200_run_pca(self.h, C.byref(opt), _ptr(ev), _ptr(sc), _ptr(ld), C.byref(m)), "run_pca")
        out = {"eigenvalues": ev, "scores": sc, "n_loci_used": int(m.value)}
        if loadings:
            out["loadings"] = ld
        return out

    def grm_product(self, x, keep=None):
        """Z^T Z x (not divided by M) for x float64[N][n_cols], n_cols <= 48: (y float64[N][n_cols], n_loci_used)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        one = x.ndim == 1
        x2 = x[:, None] if one else x
        if x2.shape[0] != self.n_genomes:
            raise ValueError(f"x must have {self.n_genomes} rows")
        kp = self._keep(keep)
        y = np.zeros_like(x2)
        m = C.c_uint64(0)
        self._check(self.lib.kgl_b200_run_grm_product(self.h, _ptr(kp), C.c_uint32(x2.shape[1]), _ptr(x2), _ptr(y), C.byref(m)), "run_grm_product")
        return (y[:, 0] if one else y), int(m.value)

    def _ld_options(self, window_loci, window_bp, keep):
        kp = self._keep(keep)
        return LdOptions(keep=None if kp is None else kp.ctypes.data, window_loci=int(window_loci), window_bp=int(window_bp)), kp

    def ld_pairs(self, min_r2: float, window_loci: int = 0, window_bp: int = 0, keep=None, capacity: int = 1 << 22) -> np.ndarray:
        """Every in-window pair of eligible loci (PCA's used set) with genotypic r^2 >= min_r2, sorted by (a, b): an LD_PAIR_DTYPE
        array. The window counts eligible loci (window_loci) and / or offset distance (window_bp); 0 = no limit, not both. Retries
        once with the exact capacity (a retry computes everything again)."""
        opt, kp = self._ld_options(window_loci, window_bp, keep)
        n = C.c_uint64(0)
        for attempt in range(2):
            out = np.zeros(max(int(capacity), 1), dtype=LD_PAIR_DTYPE)
            rc = self.lib.kgl_b200_run_ld_pairs(self.h, C.byref(opt), C.c_double(min_r2), C.c_uint64(capacity), _ptr(out), C.byref(n))
            if rc == KGL_B200_ERR_NOMEM and attempt == 0:
                capacity = int(n.value)
                continue
            self._check(rc, "run_ld_pairs")
            break
        return out[: n.value].copy()

    def ld_prune(self, max_r2: float, window_loci: int = 0, window_bp: int = 0, keep=None):
        """Greedy LD pruning in locus order (an eligible locus is kept unless an earlier kept one in its window has r^2 > max_r2):
        (keep uint8[L], n_kept). The mask is meant for pca(keep=...)."""
        opt, kp = self._ld_options(window_loci, window_bp, keep)
        out = np.zeros(self.n_loci, dtype=np.uint8)
        n = C.c_uint64(0)
        self._check(self.lib.kgl_b200_run_ld_prune(self.h, C.byref(opt), C.c_double(max_r2), _ptr(out), C.byref(n)), "run_ld_prune")
        return out, int(n.value)

    def _groups(self, group, n_groups):
        """(labels uint8[N] or None, G): None = the super-population labels, KGL_B200_MAX_POP groups."""
        if group is None:
            return None, KGL_B200_MAX_POP
        g = np.ascontiguousarray(group, dtype=np.uint8)
        if g.shape != (self.n_genomes,):
            raise ValueError(f"group must be uint8[{self.n_genomes}]")
        if n_groups is None:
            valid = g[g != 0xFF]
            n_groups = int(valid.max()) + 1 if valid.size else 1
        return g, int(n_groups)

    def group_counts(self, group=None, n_groups=None) -> np.ndarray:
        """Per-group genotype counts uint32[L][G][4]: genomes of group k with code c at locus l (0xFF = in no group). group=None:
        the super-population labels (G = 6); n_groups=None: the largest label + 1."""
        g, G = self._groups(group, n_groups)
        out = np.zeros((self.n_loci, G, 4), dtype=np.uint32)
        self._check(self.lib.kgl_b200_run_group_counts(self.h, C.c_uint32(G), _ptr(g), _ptr(out)), "run_group_counts")
        return out

    def fst(self, group=None, n_groups=None, method: str = "hudson", pairs=None, keep=None, per_locus: bool = False,
            window_bp: int = 0, step_bp: int = 0):
        """F_ST between pairs of groups (Hudson or Weir & Cockerham, include/kgl_b200.h): a dict with pairs uint32[P][2], fst
        float64[P] (genome-wide ratio of sums, NaN where no locus is used), with per_locus=True per_locus float64[P][L][2] =
        (numerator, denominator), and with window_bp > 0 windows float64[P][W][3] = (sum num, sum den, loci used) and
        window_start uint64[W] (step_bp = 0: step = window_bp). pairs=None: every pair a < b."""
        g, G = self._groups(group, n_groups)
        if pairs is None:
            pr = np.array([(a, b) for a in range(G) for b in range(a + 1, G)], dtype=np.uint32).reshape(-1, 2)
        else:
            pr = np.ascontiguousarray(pairs, dtype=np.uint32).reshape(-1, 2)
            if pr.shape[0] == 0:          # the C ABI reads n_pairs == 0 as "every pair", which the buffers below would not hold
                raise ValueError("pairs is empty: pass pairs=None for every pair")
        kp = self._keep(keep)
        opt = FstOptions(group=None if g is None else g.ctypes.data, n_groups=G, keep=None if kp is None else kp.ctypes.data,
                         method=FST_METHODS[method], n_pairs=0 if pairs is None else pr.shape[0],
                         pairs=None if pairs is None else pr.ctypes.data, window_bp=int(window_bp), step_bp=int(step_bp))
        out = np.full(pr.shape[0], np.nan, dtype=np.float64)
        pl = np.zeros((pr.shape[0], self.n_loci, 2), dtype=np.float64) if per_locus else None
        step = int(step_bp) or int(window_bp)
        nw = int(self._offsets.max()) // step + 1 if window_bp and self._offsets is not None and self._offsets.size else 0
        win = np.zeros((pr.shape[0], nw, 3), dtype=np.float64) if window_bp else None
        n = C.c_uint64(0)
        self._check(self.lib.kgl_b200_run_fst(self.h, C.byref(opt), _ptr(out), _ptr(pl), _ptr(win) if nw else None, C.byref(n)), "run_fst")
        res = {"pairs": pr, "fst": out}
        if per_locus:
            res["per_locus"] = pl
        if window_bp:
            assert n.value == nw, (n.value, nw)
            res["windows"] = win
            res["window_start"] = np.arange(nw, dtype=np.uint64) * np.uint64(step)
        return res

    def hardy(self, group=None, n_groups=None, midp: bool = False, f: bool = False):
        """Exact Hardy-Weinberg test per (locus, group) (include/kgl_b200.h): a dict with p float64[L][G] (mid-p with midp=True; NaN
        where a group has no call and on multi-allelic rows) and, with f=True, f float64[L][G] = 1 - H_obs / H_exp. group=None: the
        super-population labels (G = 6); pass zeros for one pooled group."""
        g, G = self._groups(group, n_groups)
        opt = HardyOptions(group=None if g is None else g.ctypes.data, n_groups=G, midp=int(bool(midp)))
        p = np.zeros((self.n_loci, G), dtype=np.float64)
        fo = np.zeros((self.n_loci, G), dtype=np.float64) if f else None
        self._check(self.lib.kgl_b200_run_hardy(self.h, C.byref(opt), _ptr(p), _ptr(fo)), "run_hardy")
        res = {"p": p}
        if f:
            res["f"] = fo
        return res

    def variant_qc(self, min_call_rate: float = 0.0, min_maf: float = 0.0, min_hwe_p: float = 0.0, group=None, n_groups=None,
                   midp: bool = False, keep=None):
        """Variant QC mask (keep uint8[L], n_kept): call rate over all genomes >= min_call_rate, MAF >= min_maf and the exact HWE
        p >= min_hwe_p in every group with calls; 0 = no filter. The mask is meant for pca / ld_prune / fst(keep=...)."""
        g, G = self._groups(group, n_groups) if min_hwe_p else (None, 0)
        kp = self._keep(keep)
        opt = QcOptions(keep=None if kp is None else kp.ctypes.data, min_call_rate=float(min_call_rate), min_maf=float(min_maf),
                        min_hwe_p=float(min_hwe_p), group=None if g is None else g.ctypes.data, n_groups=G, midp=int(bool(midp)))
        out = np.zeros(self.n_loci, dtype=np.uint8)
        n = C.c_uint64(0)
        self._check(self.lib.kgl_b200_run_variant_qc(self.h, C.byref(opt), _ptr(out), C.byref(n)), "run_variant_qc")
        return out, int(n.value)

    def last_hardy_terms(self) -> int:
        """Terms of the exact test walked by the last hardy / variant_qc call (all cells)."""
        return int(self.lib.kgl_b200_last_hardy_terms(self.h))

    def binned_genome_counts(self, lower, upper, pop: int = 0, present_only: bool = True):
        """(counts uint64[n_bins][N][4], rows uint64[n_bins]) -- CalcFWS' per-genome AlleleSummmary per AF bin."""
        lo = np.ascontiguousarray(lower, dtype=np.float64)
        hi = np.ascontiguousarray(upper, dtype=np.float64)
        out = np.zeros((lo.shape[0], self.n_genomes, 4), dtype=np.uint64)
        rows = np.zeros(lo.shape[0], dtype=np.uint64)
        self._check(self.lib.kgl_b200_run_binned_genome_counts(self.h, C.c_uint32(pop), C.c_uint32(lo.shape[0]), _ptr(lo), _ptr(hi),
                                                               C.c_int(int(present_only)), _ptr(out), _ptr(rows)), "run_binned_genome_counts")
        return out, rows

    def hetero_homo(self, other_allele_entries: int = 1) -> np.ndarray:
        """HeteroHomoZygous::updateVariantAnalysisType per genome: uint64[N][7] = total, snp, indel, homMinor, hetMinor, hetRefMinor, homRef."""
        out = np.zeros((self.n_genomes, 7), dtype=np.uint64)
        self._check(self.lib.kgl_b200_run_hetero_homo(self.h, C.c_int(other_allele_entries), _ptr(out)), "run_hetero_homo")
        return out

    def gram(self) -> np.ndarray:
        """Dosage Gram matrix int32[N][N] on the tensor cores (tcgen05 kind::i8)."""
        out = np.zeros((self.n_genomes, self.n_genomes), dtype=np.int32)
        self._check(self.lib.kgl_b200_run_gram(self.h, _ptr(out)), "run_gram")
        return out

    def grm(self, pop: int = 5) -> np.ndarray:
        """Centred relationship matrix float64[N][N] for the AF column `pop`."""
        out = np.zeros((self.n_genomes, self.n_genomes), dtype=np.float64)
        self._check(self.lib.kgl_b200_run_grm(self.h, C.c_uint32(pop), _ptr(out)), "run_grm")
        return out

    def enqueue_gram(self):
        self._check(self.lib.kgl_b200_enqueue_gram(self.h), "enqueue_gram")

    def enqueue_gram_tiles(self, first: int, stride: int):
        self._check(self.lib.kgl_b200_enqueue_gram_tiles(self.h, C.c_uint64(first), C.c_uint64(stride)), "enqueue_gram_tiles")

    def gram_buffer(self):
        p, n, ld = C.c_void_p(), C.c_uint64(), C.c_uint64()
        self._check(self.lib.kgl_b200_gram_buffer(self.h, C.byref(p), C.byref(n), C.byref(ld)), "gram_buffer")
        return int(p.value), int(n.value), int(ld.value)

    def fetch_gram(self) -> np.ndarray:
        out = np.zeros((self.n_genomes, self.n_genomes), dtype=np.int32)
        self._check(self.lib.kgl_b200_fetch_gram(self.h, _ptr(out)), "fetch_gram")
        return out

    def last_gram_kernel_ms(self) -> float:
        return float(self.lib.kgl_b200_last_gram_kernel_ms(self.h))

    def set_ibs_tensor_cores(self, enable: bool):
        """Dense part of the IBS calls on the tensor cores (default) or on the popcount tile kernel."""
        self._check(self.lib.kgl_b200_set_ibs_tensor_cores(self.h, C.c_int(int(bool(enable)))), "set_ibs_tensor_cores")

    def ibs_used_tensor_cores(self) -> bool:
        return bool(self.lib.kgl_b200_ibs_used_tensor_cores(self.h))

    def enqueue_ibs_tile_list(self, coords: np.ndarray):
        """Resident tiles of an explicit list, coords uint32[count][2]; results in ibs_tiles_buffer()."""
        coords = np.ascontiguousarray(coords, dtype=np.uint32).reshape(-1, 2)
        self._check(self.lib.kgl_b200_enqueue_ibs_tile_list(self.h, C.c_uint64(coords.shape[0]), _ptr(coords)), "enqueue_ibs_tile_list")

    def ibs_tile_list(self, coords: np.ndarray) -> np.ndarray:
        """uint32[count][64][64][4] for an explicit list of tiles."""
        coords = np.ascontiguousarray(coords, dtype=np.uint32).reshape(-1, 2)
        out = np.zeros((coords.shape[0], 64, 64, 4), dtype=np.uint32)
        if coords.shape[0]:
            self._check(self.lib.kgl_b200_run_ibs_tile_list(self.h, C.c_uint64(coords.shape[0]), _ptr(coords), _ptr(out)), "run_ibs_tile_list")
        return out

    def ibs_tile_grid(self):
        side, n = C.c_uint64(), C.c_uint64()
        self._check(self.lib.kgl_b200_ibs_tile_grid(self.h, C.byref(side), C.byref(n)), "ibs_tile_grid")
        return int(side.value), int(n.value)

    def ibs_tiles(self, first=0, stride=1, count=None) -> np.ndarray:
        """Upper-triangle 64x64 tiles first, first+stride, ...: uint32[count][64][64][4] (rank r of R: first=r, stride=R)."""
        if count is None:
            count = tiles_of_rank(self.ibs_tile_grid()[1], first, stride)
        out = np.zeros((count, 64, 64, 4), dtype=np.uint32)
        if count:
            self._check(self.lib.kgl_b200_run_ibs_tiles(self.h, C.c_uint64(first), C.c_uint64(stride), C.c_uint64(count), _ptr(out)), "run_ibs_tiles")
        return out

    def enqueue_ibs_tiles(self, first: int, stride: int, count: int):
        self._check(self.lib.kgl_b200_enqueue_ibs_tiles(self.h, C.c_uint64(first), C.c_uint64(stride), C.c_uint64(count)), "enqueue_ibs_tiles")

    def ibs_tiles_buffer(self):
        p, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.kgl_b200_ibs_tiles_buffer(self.h, C.byref(p), C.byref(n)), "ibs_tiles_buffer")
        return int(p.value), int(n.value)

    def ibs_timer_reset(self):
        self._check(self.lib.kgl_b200_ibs_timer_reset(self.h), "ibs_timer_reset")

    def ibs_timer_read(self) -> np.ndarray:
        ms = np.zeros(256, dtype=np.float32)
        n = C.c_uint32(0)
        self._check(self.lib.kgl_b200_ibs_timer_read(self.h, _ptr(ms), C.c_uint32(256), C.byref(n)), "ibs_timer_read")
        return ms[: n.value].copy()

    # ---- resident / multi-GPU building blocks ----
    def launch_count(self) -> int:
        return int(self.lib.kgl_b200_launch_count(self.h))

    def last_stream_kernel_ms(self) -> float:
        return float(self.lib.kgl_b200_last_stream_kernel_ms(self.h))

    def kernel_timer_reset(self):
        self._check(self.lib.kgl_b200_kernel_timer_reset(self.h), "kernel_timer_reset")

    def kernel_timer_read(self) -> np.ndarray:
        ms = np.zeros(256, dtype=np.float32)
        n = C.c_uint32(0)
        self._check(self.lib.kgl_b200_kernel_timer_read(self.h, _ptr(ms), C.c_uint32(256), C.byref(n)), "kernel_timer_read")
        return ms[: n.value].copy()

    def fetch_locus_counts(self) -> np.ndarray:
        lc = np.zeros((self.n_loci, 4), dtype=np.uint32)
        self._check(self.lib.kgl_b200_fetch_locus_counts(self.h, _ptr(lc)), "fetch_locus_counts")
        return lc

    def peer_export(self) -> bytes:
        """CUDA IPC handle (64 bytes) of this rank's exchange region; gather the handles of all ranks and peer_attach them."""
        buf = C.create_string_buffer(64)
        self._check(self.lib.kgl_b200_peer_export(self.h, buf), "peer_export")
        return buf.raw

    def peer_attach(self, rank: int, world: int, handles: list[bytes]):
        blob = b"".join(handles)
        assert len(blob) == 64 * world
        self._check(self.lib.kgl_b200_peer_attach(self.h, C.c_uint32(rank), C.c_uint32(world), C.c_char_p(blob)), "peer_attach")

    def peer_set_timeout_ms(self, milliseconds: int):
        self._check(self.lib.kgl_b200_peer_set_timeout_ms(self.h, C.c_uint64(milliseconds)), "peer_set_timeout_ms")

    def enqueue_count_and_inbreed_peer(self):
        self._check(self.lib.kgl_b200_enqueue_count_and_inbreed_peer(self.h), "enqueue_count_and_inbreed_peer")

    def inbreed_begin(self, algorithm: str, hall_start=None, hall_sweeps=0, ll_tolerance=0.0, ll_max_iterations=0, count_loci=False,
                      exact_sweeps=False):
        opt = InbreedOptions()
        opt.count_loci = int(bool(count_loci))
        opt.exact_sweeps = int(bool(exact_sweeps))
        self._hall_keep = None
        if hall_start is not None:
            self._hall_keep = np.ascontiguousarray(hall_start, dtype=np.float64)
            opt.hall_start = self._hall_keep.ctypes.data_as(C.POINTER(C.c_double))
        opt.hall_sweeps, opt.ll_tolerance, opt.ll_max_iterations = int(hall_sweeps), float(ll_tolerance), int(ll_max_iterations)
        self._check(self.lib.kgl_b200_inbreed_begin(self.h, C.c_int(ALGORITHMS[algorithm]), C.byref(opt)), "inbreed_begin")

    def inbreed_accumulate(self):
        self._check(self.lib.kgl_b200_inbreed_accumulate(self.h), "inbreed_accumulate")

    def inbreed_partials_buffer(self):
        p, n = C.c_void_p(), C.c_uint64()
        self._check(self.lib.kgl_b200_inbreed_partials_buffer(self.h, C.byref(p), C.byref(n)), "inbreed_partials_buffer")
        return int(p.value), int(n.value)

    def inbreed_update(self) -> bool:
        fin = C.c_int(0)
        self._check(self.lib.kgl_b200_inbreed_update(self.h, C.byref(fin)), "inbreed_update")
        return bool(fin.value)

    def inbreed_fetch(self) -> np.ndarray:
        out = np.zeros(self.n_genomes, dtype=RESULT_DTYPE)
        self._check(self.lib.kgl_b200_inbreed_fetch(self.h, _ptr(out)), "inbreed_fetch")
        return out
