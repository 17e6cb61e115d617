"""Population differentiation on one GPU (kgl_b200_run_group_counts / kgl_b200_run_fst) on device-synthesised populations
(development tool).

  --config 2 : 2,504 genomes x 1.1 M SNPs      --config 5 : 100,000 x 1 M
Populations with 0.1 % code-3 cells. Labellings: the synthesised super-populations (6 groups in runs, as in 1000 Genomes order),
6 groups interleaved genome by genome (every 32-genome word holds all six) and, for config 5, 32 groups in runs and 32 random
groups. For each: the k_group_counts kernel time of --repeats calls under torch.profiler (median), against the HBM bound of its
traffic (the matrix rows it reads, N/4 bytes per locus rounded up to 128-bit units, plus the L x G x 16 bytes of counts it writes,
at the data sheet's 7.7 TB/s); the wall time of run_group_counts (which also copies the counts to the host); and run_fst (Hudson,
every pair, no per-locus terms or windows) with its kernels, and run_fst again with 100 kb windows in 50 kb steps (wall time and
the k_fst_windows kernel). The GPU's name and power limit are read in the same run. Prints one
JSON line per (config, labelling).
  python tools/fst_bench.py --config 2 5 [--repeats 5] [--out DIR]
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
HBM_BYTES_PER_S = 7.7e12          # data sheet, one B200
WINDOW_BP, STEP_BP = 100_000, 50_000


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


def kernel_ms(fn, out_dir, tag):
    """{kernel name: [ms per launch]} of the CUDA kernels fn launches."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"fst_{tag}.pt.trace.json"))
    out = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            key = next((k for k in ("k_group_counts", "k_fst_blocks", "k_fst_total", "k_fst_windows") if k in e.name), "other")
            out.setdefault(key, []).append(e.time_range.elapsed_us() / 1e3)
    return out


def labellings(config, superpop):
    n = superpop.shape[0]
    rng = np.random.default_rng(SEED)
    out = [("superpop_6", None, 6), ("interleaved_6", (np.arange(n) % 6).astype(np.uint8), 6)]
    if config == 5:
        out += [("runs_32", (np.arange(n) * 32 // n).astype(np.uint8), 32), ("random_32", rng.integers(0, 32, n).astype(np.uint8), 32)]
    return out


def run(config, repeats, out_dir):
    n, l = CONFIGS[config]
    offsets, af = make_loci(l, SEED)
    superpop, f = make_genomes(n, SEED)
    ctx = KglB200(0)
    ctx.upload_loci(af, offsets)
    ctx.set_genome_superpop(superpop)
    ctx.synth_genotypes(SEED, n, l, f, missing_rate=0.001)
    ctx.synchronize()
    units = -(-n // 64)
    results = []
    for name, group, g in labellings(config, superpop):
        ctx.group_counts(group, g)                                           # warm-up: entry lists, buffers
        wall = [clock(lambda: ctx.group_counts(group, g)) for _ in range(repeats)]
        ks = kernel_ms(lambda: [ctx.group_counts(group, g) for _ in range(repeats)], out_dir, f"counts_config{config}_{name}")
        k = float(np.median(ks["k_group_counts"]))
        read, write = l * units * 16, l * g * 16
        ctx.fst(group, g)
        fst_wall = [clock(lambda: ctx.fst(group, g)) for _ in range(repeats)]
        kf = kernel_ms(lambda: ctx.fst(group, g), out_dir, f"fst_config{config}_{name}")
        win_wall = [clock(lambda: ctx.fst(group, g, window_bp=WINDOW_BP, step_bp=STEP_BP)) for _ in range(repeats)]
        kw = kernel_ms(lambda: ctx.fst(group, g, window_bp=WINDOW_BP, step_bp=STEP_BP), out_dir, f"fst_windows_config{config}_{name}")
        res = {"config": config, "n_genomes": n, "n_loci": l, "labelling": name, "n_groups": g, "n_pairs": g * (g - 1) // 2,
               "k_group_counts_ms": [round(v, 4) for v in ks["k_group_counts"]], "k_group_counts_median_ms": round(k, 4),
               "bytes_read": read, "bytes_written": write,
               "achieved_tb_per_s": round((read + write) / (k / 1e3) / 1e12, 3),
               "hbm_bound_ms": round((read + write) / HBM_BYTES_PER_S * 1e3, 4),
               "fraction_of_hbm_bound": round((read + write) / HBM_BYTES_PER_S / (k / 1e3), 3),
               "group_counts_wall_ms": [round(v, 3) for v in wall],
               "fst_wall_ms": [round(v, 3) for v in fst_wall],
               "fst_kernels_ms": {key: round(sum(v), 4) for key, v in kf.items()},
               "fst_windows": {"window_bp": WINDOW_BP, "step_bp": STEP_BP, "n_windows": int(offsets.max()) // STEP_BP + 1,
                               "wall_ms": [round(v, 3) for v in win_wall], "k_fst_windows_ms": round(sum(kw.get("k_fst_windows", [0.0])), 4)}}
        results.append(res)
    free, total = torch.cuda.mem_get_info(0)
    info = gpu_info()
    for r in results:
        r["device_memory_in_use_gb"] = round((total - free) / 1e9, 3)
        r.update(info)
    ctx.close()
    return results


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, nargs="+", default=[2])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: the benchmark measures the GPU only")
    if a.out:
        os.makedirs(a.out, exist_ok=True)
    for c in a.config:
        for r in run(c, a.repeats, a.out):
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
