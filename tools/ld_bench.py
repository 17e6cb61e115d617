"""Linkage disequilibrium on one GPU (kgl_b200_run_ld_pairs / kgl_b200_run_ld_prune) on device-synthesised populations
(development tool).

  --config 2 : 2,504 genomes x 1.1 M SNPs      --config 5 : 100,000 x 1 M
Populations with 0.1 % code-3 cells, so that all four Gram products (GG, CC, GC, QC) run, at window_loci = 1,000. For each
config: run_ld_pairs(min_r2 = 0.2) and run_ld_prune(0.2), each timed --repeats times with a host clock around work that ends in
a device synchronise, after a warm-up call (which builds the loci-major code copy). Then one call of each under torch.profiler:
kernel times by phase -- the Gram runs (k_gram_i8), k_ld_pairs, the sort (cub radix sort + gather), the raw counting pass and
code copy -- and the rest of the wall time (the host band list, the host prune scan, copies, gaps). Executed int8 MACs are
counted over the padded tiles the Gram runs cover and divided by the Gram kernel time; the bytes of int32 blocks are what the
runs write and k_ld_pairs reads. Device memory in use and the GPU's name and power limit are read in the same run. Prints one
JSON line per config.
  python tools/ld_bench.py --config 2 5 [--repeats 3] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kgl_gene_b200.capi import KglB200                            # noqa: E402
from kgl_gene_b200.synth import make_genomes, make_loci           # noqa: E402

SEED = 5
CONFIGS = {2: (2504, 1_100_000), 5: (100_000, 1_000_000)}
WINDOW = 1000
THRESHOLD = 0.2
CAPACITY = 1 << 25           # room for every pair of both configs: a call computes once (a NOMEM answer would make it twice)
MMA_PEAK = 3.5e15            # measured int8 MMA rate of k_gram_i8's tcgen05 issue (DESIGN 4c)
TILE = 256


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip()
    except Exception as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def clock(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def band_shape(eligible: np.ndarray, window: int):
    """(band tiles, of them diagonal) of the band ld_band lists for a window of `window` eligible loci (ld.cuh)."""
    e = np.flatnonzero(eligible)
    n_blocks = -(-eligible.shape[0] // TILE)
    last = np.minimum(np.arange(e.shape[0]) + window - 1, e.shape[0] - 1)
    has = last > np.arange(e.shape[0])
    rows = e[has] // TILE
    hi = np.full(n_blocks, -1)
    np.maximum.at(hi, rows, e[last[has]] // TILE)
    first = np.full(n_blocks, np.iinfo(np.int64).max)
    np.minimum.at(first, rows, e[np.flatnonzero(has) + 1] // TILE)
    lo = np.where(hi >= 0, first, -1)
    count = np.bincount(e // TILE, minlength=n_blocks)
    nonempty = np.concatenate([[0], np.cumsum(count > 0)])
    tiles = diag = 0
    for i in np.flatnonzero(hi >= 0):
        tiles += int(nonempty[hi[i] + 1] - nonempty[lo[i]])
        diag += int(lo[i] == i)
    return tiles, diag


def profile(fn, out_dir, tag):
    """Kernel and copy times of one call: {phase: ms}. host_and_gaps is the wall time outside kernels and copies: the raw
    counting pass's host side, the band list and tile lists, the host prune scan, the binding's output buffers, launch gaps."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        wall = clock(fn)
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"ld_{tag}.pt.trace.json"))
    evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    phase = {"gram": 0.0, "k_ld_pairs": 0.0, "sort": 0.0, "counts_and_codes": 0.0, "copies": 0.0, "other": 0.0}
    for e in evs:
        ms = e.time_range.elapsed_us() / 1e3
        name = e.name
        if "k_gram_i8" in name:
            phase["gram"] += ms
        elif "k_ld_pairs" in name:
            phase["k_ld_pairs"] += ms
        elif "Radix" in name or "radix" in name or "k_gather_pairs" in name:
            phase["sort"] += ms
        elif "k_codes16" in name or "k_stream" in name or "count" in name.lower() or "k_pca_loci" in name or "k_fix_locus" in name:
            phase["counts_and_codes"] += ms
        elif "memcpy" in name.lower() or "memset" in name.lower():
            phase["copies"] += ms
        else:
            phase["other"] += ms
    kernels = sum(v for k, v in phase.items() if k != "copies")
    return {"wall_ms": round(wall, 3), **{k: round(v, 3) for k, v in phase.items()}, "kernels_ms": round(kernels, 3),
            "host_and_gaps_ms": round(wall - kernels - phase["copies"], 3)}


def run(config, repeats, out_dir):
    n, l = CONFIGS[config]
    offsets, af = make_loci(l, SEED)
    superpop, f = make_genomes(n, SEED)
    ctx = KglB200(0)
    ctx.upload_loci(af, offsets)
    ctx.set_genome_superpop(superpop)
    ctx.synth_genotypes(SEED, n, l, f, missing_rate=0.001)
    ctx.synchronize()
    pairs = ctx.ld_pairs(THRESHOLD, WINDOW, capacity=CAPACITY)                    # warm-up: loci-major codes, buffers
    keep, n_kept = ctx.ld_prune(THRESHOLD, WINDOW)
    pairs_ms = [clock(lambda: ctx.ld_pairs(THRESHOLD, WINDOW, capacity=CAPACITY)) for _ in range(repeats)]
    prune_ms = [clock(lambda: ctx.ld_prune(THRESHOLD, WINDOW)) for _ in range(repeats)]
    free, total = torch.cuda.mem_get_info(0)
    prof_pairs = profile(lambda: ctx.ld_pairs(THRESHOLD, WINDOW, capacity=CAPACITY), out_dir, f"pairs_config{config}")
    prof_prune = profile(lambda: ctx.ld_prune(THRESHOLD, WINDOW), out_dir, f"prune_config{config}")
    # eligible loci: the raw counts, as the device forms them (0 < p < 1, keep = all)
    lc, _ = ctx.allele_count(want_genomes=False)
    alt = lc[:, 1].astype(np.int64) + 2 * lc[:, 2]
    eligible = (alt > 0) & (alt < 2 * lc[:, :3].sum(axis=1).astype(np.int64))
    tiles, diag = band_shape(eligible, WINDOW)
    runs_tiles = 2 * tiles + 2 * (2 * tiles - diag)             # GG, CC over the band; GC, QC over the band and its mirrors
    k_pad = -(-n // 128) * 128
    macs = runs_tiles * TILE * TILE * k_pad
    block_bytes = runs_tiles * TILE * TILE * 4
    out = {"config": config, "n_genomes": n, "n_loci": l, "window_loci": WINDOW, "threshold": THRESHOLD,
           "eligible_loci": int(eligible.sum()), "band_tiles": tiles, "diagonal_tiles": diag, "n_pairs_r2_ge_0.2": int(len(pairs)),
           "n_kept": n_kept, "pairs_ms": [round(v, 3) for v in pairs_ms], "pairs_median_ms": float(np.median(pairs_ms)),
           "prune_ms": [round(v, 3) for v in prune_ms], "prune_median_ms": float(np.median(prune_ms)),
           "pairs_profile": prof_pairs, "prune_profile": prof_prune,
           "gram_int8_macs": macs, "gram_macs_per_s": macs / (prof_pairs["gram"] / 1e3),
           "share_of_mma_peak": macs / (prof_pairs["gram"] / 1e3) / MMA_PEAK,
           "int32_block_bytes_written": block_bytes, "int32_block_bytes_read_by_k_ld_pairs": block_bytes,
           "gram_write_gb_per_s": block_bytes / (prof_pairs["gram"] / 1e3) / 1e9,
           "k_ld_pairs_read_gb_per_s": block_bytes / (prof_pairs["k_ld_pairs"] / 1e3) / 1e9,
           "device_memory_in_use_gb": (total - free) / 1e9, "loci_major_codes_gb": -(-l // 256) * 256 * -(-n // 128) * 32 / 1e9,
           **gpu_info()}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, nargs="+", default=[2])
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: the benchmark measures the GPU only")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    for c in a.config:
        print(json.dumps(run(c, a.repeats, a.out)), flush=True)


if __name__ == "__main__":
    main()
