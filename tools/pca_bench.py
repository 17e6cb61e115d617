"""Genotype PCA on one GPU (kgl_b200_run_grm_product / kgl_b200_run_pca) on device-synthesised populations (development tool).

  --config 2 : 2,504 genomes x 1.1 M SNPs      --config 4 : 2,504 x 20 M      --config 5 : 100,000 x 1 M
For each config: one Z^T Z apply (kgl_b200_run_grm_product, b = 16 columns, the block of k = 10) and the whole kgl_b200_run_pca
at k = 10, q = 10, each timed --repeats times with a host clock around work that ends in a device synchronise, after a warm-up
call (which builds the code copies). Then one apply and one run_pca under torch.profiler: kernel times by phase -- the pass-1
Gram runs (K = genomes), the pass-2 Gram runs (K = loci), the quantise / recombine kernels (k_pca_*), the raw counting pass --
and the rest of the wall time (host QR / Rayleigh-Ritz, copies, gaps). Executed int8 MACs are counted from the shapes the Gram
runs cover (padded tiles included) and divided by the Gram kernel time. Device memory in use after the runs (the context keeps
its buffers) and the GPU's name and power limit are read in the same run. Prints one JSON line per config.
  python tools/pca_bench.py --config 2 4 5 [--repeats 3] [--out DIR]
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
CONFIGS = {2: (2504, 1_100_000), 4: (2504, 20_000_000), 5: (100_000, 1_000_000)}
MMA_PEAK = 3.5e15            # measured int8 MMA rate of k_gram_i8's tcgen05 issue (DESIGN 4c)


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


def apply_macs(n, l, cols, code3):
    """int8 MACs the Gram runs of one apply execute: pass 1 over the padded loci x digit blocks x padded genomes, pass 2 over
    the padded genomes x digit blocks x padded loci; each twice with code-3 cells."""
    blocks = -(-cols // 16)
    runs = 2 if code3 else 1
    pad = lambda v, m: -(-v // m) * m
    p1 = pad(l, 256) * blocks * 256 * pad(n, 128)
    p2 = pad(n, 256) * blocks * 256 * pad(l, 128)
    return runs * (p1 + p2)


def profile(fn, out_dir, tag):
    """Kernel and copy times of one call, in launch order: {phase: ms}."""
    from torch.profiler import ProfilerActivity, profile as tprofile
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        wall = clock(fn)
    if out_dir:
        prof.export_chrome_trace(os.path.join(out_dir, f"pca_{tag}.pt.trace.json"))
    evs = sorted([e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA], key=lambda e: e.time_range.start)
    phase = {"pass1_gram": 0.0, "pass2_gram": 0.0, "quantise_recombine": 0.0, "codes_and_counts": 0.0, "copies": 0.0, "other": 0.0}
    n_digits = 0
    for e in evs:
        ms = e.time_range.elapsed_us() / 1e3
        name = e.name
        if "k_pca_digits" in name:
            n_digits += 1
        if "k_gram_i8" in name:
            phase["pass1_gram" if n_digits % 2 == 1 else "pass2_gram"] += ms
        elif "k_pca_" in name:
            phase["quantise_recombine"] += ms
        elif "k_codes16" in name or "k_stream" in name or "count" in name.lower() or "k_to_sample_major" in name:
            phase["codes_and_counts"] += ms
        elif "memcpy" in name.lower() or "memset" in name.lower():
            phase["copies"] += ms
        else:
            phase["other"] += ms
    kernels = sum(v for k, v in phase.items() if k != "copies")
    return {"wall_ms": wall, **{k: round(v, 3) for k, v in phase.items()}, "kernels_ms": round(kernels, 3),
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
    x = np.random.default_rng(1).standard_normal((n, 16))
    ctx.grm_product(x)                                            # warm-up: loci-major and genome-major code copies, buffers
    r = ctx.pca(k=10, iterations=10)
    apply_ms = [clock(lambda: ctx.grm_product(x)) for _ in range(repeats)]
    pca_ms = [clock(lambda: ctx.pca(k=10, iterations=10)) for _ in range(repeats)]
    free, total = torch.cuda.mem_get_info(0)
    prof_apply = profile(lambda: ctx.grm_product(x), out_dir, f"apply_config{config}")
    prof_pca = profile(lambda: ctx.pca(k=10, iterations=10), out_dir, f"run_config{config}")
    macs = apply_macs(n, l, 16, True)
    gram_ms = prof_apply["pass1_gram"] + prof_apply["pass2_gram"]
    out = {"config": config, "n_genomes": n, "n_loci": l, "n_loci_used": r["n_loci_used"], "eigenvalues": [round(v, 6) for v in r["eigenvalues"]],
           "apply_ms": [round(v, 3) for v in apply_ms], "apply_median_ms": float(np.median(apply_ms)),
           "pca_k10_q10_ms": [round(v, 3) for v in pca_ms], "pca_median_ms": float(np.median(pca_ms)),
           "apply_profile": prof_apply, "pca_profile": prof_pca,
           "apply_int8_macs": macs, "gram_macs_per_s": macs / (gram_ms / 1e3), "share_of_mma_peak": macs / (gram_ms / 1e3) / MMA_PEAK,
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
