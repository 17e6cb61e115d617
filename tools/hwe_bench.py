"""Hardy-Weinberg equilibrium and variant QC on one GPU (kgl_b200_run_hardy / kgl_b200_run_variant_qc) on device-synthesised
populations (development tool).

  --config 2 : 2,504 genomes x 1.1 M SNPs, pooled (one group) and the 6 super-populations
  --config 5 : 100,000 x 1 M, 6 contiguous groups and 32 random groups
Populations with 0.1 % code-3 cells. Per labelling: the wall time of run_hardy (p and F) and of run_variant_qc (call rate >= 0.98,
MAF >= 0.01, p >= 1e-6 in every group), host clock around calls that end in a synchronise, --repeats each; in a separate run under
torch.profiler, the kernel times of k_group_counts, the ordering step (k_hwe_keys and cub's radix pass), k_hwe, the raw counting
pass and k_variant_qc. The terms walked (kgl_b200_last_hardy_terms) against a full walk, and k_hwe's time against its FP64 issue
bound: terms x FP64-pipe instructions per term (DMUL, DFMA, DADD, DSETP, I2F.F64, MUFU.RCP64H in one step of the walk's SASS) at
the data sheet's FP64 rate (37 TFLOP/s per GPU, an FMA counted twice: 18.5 x 10^12 instructions/s). The lane efficiency of the
cell order and of row order comes from the full-walk term counts of the oracle (tests/hwe_oracle.py, counting only). The GPU's
name and power limit are read in the same run. Prints one JSON line per (config, labelling).
  python tools/hwe_bench.py --config 2 5 [--repeats 3] [--out DIR]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
from kgl_gene_b200.capi import KglB200                            # noqa: E402
from kgl_gene_b200.synth import make_genomes, make_loci           # noqa: E402
import hwe_oracle as HO                                           # noqa: E402

SEED = 5
CONFIGS = {2: (2504, 1_100_000), 5: (100_000, 1_000_000)}
FP64_INSTR_PER_S = 18.5e12        # data sheet: 37 TFLOP/s FP64 per B200, an FMA counted as two
FP64_INSTR_PER_TERM = 20          # one step of k_hwe's walk in its SASS
QC = dict(min_call_rate=0.98, min_maf=0.01, min_hwe_p=1e-6)
KERNELS = ("k_group_counts", "k_hwe_keys", "k_hwe", "k_variant_qc", "k_stream", "Radix", "Onesweep")


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
    """{kernel key: total ms} of the CUDA kernels fn launches (the ordering step's cub kernels under "sort")."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"hwe_{tag}.pt.trace.json"))
    out = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name
        if "k_hwe_keys" in name:
            key = "k_hwe_keys"
        elif "k_hwe" in name:
            key = "k_hwe"
        elif "Radix" in name or "Onesweep" in name or "cub" in name.lower():
            key = "sort"
        else:
            key = next((k for k in ("k_group_counts", "k_variant_qc", "k_stream") if k in name), "other")
        out[key] = out.get(key, 0.0) + e.time_range.elapsed_us() / 1e3
    return out


def labellings(config, superpop):
    n = superpop.shape[0]
    rng = np.random.default_rng(SEED)
    if config == 2:
        return [("pooled_1", np.zeros(n, dtype=np.uint8), 1), ("superpop_6", None, 6)]
    return [("contiguous_6", (np.arange(n) * 6 // n).astype(np.uint8), 6), ("random_32", rng.integers(0, 32, n).astype(np.uint8), 32)]


def run(config, repeats, out_dir):
    n, l = CONFIGS[config]
    offsets, af = make_loci(l, SEED)
    superpop, f = make_genomes(n, SEED)
    ctx = KglB200(0)
    ctx.upload_loci(af, offsets)
    ctx.set_genome_superpop(superpop)
    ctx.synth_genotypes(SEED, n, l, f, missing_rate=0.001)
    ctx.synchronize()
    results = []
    for name, group, g in labellings(config, superpop):
        ctx.hardy(group, g, f=True)                                          # warm-up: entry lists, buffers, sort temp
        hardy_wall = [clock(lambda: ctx.hardy(group, g, f=True)) for _ in range(repeats)]
        terms = ctx.last_hardy_terms()
        ctx.variant_qc(group=group, n_groups=g, **QC)
        qc_wall = [clock(lambda: ctx.variant_qc(group=group, n_groups=g, **QC)) for _ in range(repeats)]
        n_kept = ctx.variant_qc(group=group, n_groups=g, **QC)[1]
        kh = kernel_ms(lambda: ctx.hardy(group, g, f=True), out_dir, f"hardy_config{config}_{name}")
        kq = kernel_ms(lambda: ctx.variant_qc(group=group, n_groups=g, **QC), out_dir, f"qc_config{config}_{name}")
        counts = ctx.group_counts(group, g)
        p = ctx.hardy(group, g)["p"]
        work = HO.walk_terms(counts[..., 0], counts[..., 1], counts[..., 2]).ravel()
        order = HO.length_order(counts)
        bound_ms = terms * FP64_INSTR_PER_TERM / FP64_INSTR_PER_S * 1e3
        res = {"config": config, "n_genomes": n, "n_loci": l, "labelling": name, "n_groups": g, "cells": l * g,
               "run_hardy_wall_ms": [round(v, 3) for v in hardy_wall], "run_variant_qc_wall_ms": [round(v, 3) for v in qc_wall],
               "hardy_kernels_ms": {k: round(v, 4) for k, v in kh.items()}, "qc_kernels_ms": {k: round(v, 4) for k, v in kq.items()},
               "terms_walked": int(terms), "terms_full_walk": int(work.sum()),
               "k_hwe_fp64_issue_bound_ms": round(bound_ms, 4),
               "k_hwe_fraction_of_fp64_bound": round(bound_ms / kh["k_hwe"], 3) if kh.get("k_hwe") else None,
               "lane_efficiency_full_walk": {"length_order": round(HO.lane_efficiency(work, order), 3),
                                             "row_order": round(HO.lane_efficiency(work), 3)},
               "qc": QC, "n_kept": n_kept, "p_below_1e-6": int((p < 1e-6).sum()), "p_nan": int(np.isnan(p).sum())}
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
    ap.add_argument("--repeats", type=int, default=3)
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
