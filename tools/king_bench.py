"""KING-robust kinship against the IBS path it is built on, on device-synthesised populations (development tool).

  --config 4 : 2,504 genomes x 20 M SNPs (missing_rate 0.001): kgl_b200_run_king (whole matrix) against kgl_b200_run_ibs.
  --config 5 : 100,000 x 1 M: kgl_b200_run_king_pairs(0.0442) over every upper tile against the IBS tile sweep of
               tools/c5_kinship_multi.py over the same tiles (shards.block_tile_coords, slabs of 8,192, tensor-core form).
               Under torchrun (one rank per GPU) the tiles are dealt with block_tile_coords and the lists joined with
               shards.gather_king_pairs.
Both sides are timed in the same process, alternating, --repeats times each, host clock around work that ends in a device
synchronise. Prints one JSON line per config (rank 0) with the GPU's name and power limit, read in the same run.
  python tools/king_bench.py --config 4 [--n N --l L]
  torchrun --nproc_per_node=G tools/king_bench.py --config 5 [--n N --l L]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kgl_gene_b200.capi import KING_PAIR_DTYPE, KglB200          # noqa: E402
from kgl_gene_b200.kinship import king_degree                    # noqa: E402
from kgl_gene_b200.shards import block_tile_coords, gather_king_pairs   # noqa: E402
from kgl_gene_b200.synth import make_genomes, make_loci          # noqa: E402

SEED = 5
SLAB = 8192


def gpu_info(local):
    """Name and power limit of the GPU (a query only)."""
    info = {"gpu": torch.cuda.get_device_name(local)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip()
    except Exception as e:                                       # the number stays usable without it
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def spread(ms):
    return {"ms": [round(x, 3) for x in ms], "median_ms": float(np.median(ms)), "min_ms": float(min(ms)), "max_ms": float(max(ms))}


def synth(local, n, l):
    offsets, af = make_loci(l, SEED)
    superpop, f = make_genomes(n, SEED)
    ctx = KglB200(local)
    ctx.upload_loci(af, offsets)
    ctx.set_genome_superpop(superpop)
    ctx.synth_genotypes(SEED, n, l, f, missing_rate=0.001)
    ctx.synchronize()
    return ctx


def clock(fn, barrier=False):
    torch.cuda.synchronize()
    if barrier:
        dist.barrier()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    if barrier:
        dist.barrier()
    return (time.perf_counter() - t0) * 1e3, r


def config4(local, n, l, repeats):
    ctx = synth(local, n, l)
    pair_loci = n * (n + 1) / 2 * l
    ctx.ibs(); ctx.king()                                        # warm-up: planes, code matrices, class counts, buffers
    ibs_ms, king_ms = [], []
    for _ in range(repeats):
        ms, _ = clock(ctx.ibs); ibs_ms.append(ms)
        ms, kin = clock(ctx.king); king_ms.append(ms)
    d = np.arange(n)
    checks = {"symmetric": bool(np.array_equal(kin, kin.T)), "diagonal_half": bool(np.all(kin[d, d] == 0.5)),
              "pairs_ge_0.0442": int((np.triu(kin, 1) >= 0.0442).sum())}
    out = {"workload": f"config 4: {n} genomes x {l} SNPs, whole matrix", "tensor_cores": ctx.ibs_used_tensor_cores(),
           "ibs": spread(ibs_ms), "king": spread(king_ms), "king_over_ibs": float(np.median(king_ms) / np.median(ibs_ms)),
           "ibs_pair_loci_per_s": pair_loci / (np.median(ibs_ms) * 1e-3), "king_pair_loci_per_s": pair_loci / (np.median(king_ms) * 1e-3),
           "king_output_bytes": int(kin.nbytes), "ibs_output_bytes": int(n * n * 16), "free_hbm_gb": torch.cuda.mem_get_info(local)[0] / 1e9,
           "checks": checks}
    ctx.close()
    assert checks["symmetric"] and checks["diagonal_half"]
    return out


def config5(local, rank, world, n, l, repeats, threshold):
    ctx = synth(local, n, l)
    coords = block_tile_coords(n, rank, world)
    pair_loci = n * (n + 1) / 2 * l
    multi = world > 1

    def ibs_sweep():
        for d in range(0, coords.shape[0], SLAB):
            ctx.enqueue_ibs_tile_list(coords[d:d + SLAB])
        ctx.synchronize()

    def king():
        return ctx.king_pairs(threshold, coords)

    ctx.enqueue_ibs_tile_list(coords[:SLAB]); ctx.synchronize()  # warm-up: planes, code matrices, class counts
    king()
    ibs_ms, king_ms = [], []
    for _ in range(repeats):
        ms, _ = clock(ibs_sweep, multi); ibs_ms.append(ms)
        ms, mine = clock(king, multi); king_ms.append(ms)
    free = torch.cuda.mem_get_info(local)[0] / 1e9
    pairs = gather_king_pairs(mine) if multi else mine
    deg = king_degree(pairs["kinship"])
    out = {"workload": f"config 5: {n} genomes x {l} SNPs, every upper tile, king_pairs({threshold}), tiles dealt to {world} GPU(s)",
           "n_gpus": world, "tiles_rank0": int(coords.shape[0]), "tensor_cores": ctx.ibs_used_tensor_cores(),
           "ibs_sweep": spread(ibs_ms), "king_pairs": spread(king_ms), "king_over_ibs": float(np.median(king_ms) / np.median(ibs_ms)),
           "ibs_pair_loci_per_s": pair_loci / (np.median(ibs_ms) * 1e-3), "king_pair_loci_per_s": pair_loci / (np.median(king_ms) * 1e-3),
           "n_pairs": int(pairs.shape[0]), "output_bytes": int(pairs.shape[0] * KING_PAIR_DTYPE.itemsize),
           "ibs_counts_bytes_if_returned": int(n * n * 16), "pairs_by_degree": {str(k): int((deg == k).sum()) for k in (0, 1, 2, 3)},
           "max_kinship": float(pairs["kinship"].max()) if pairs.shape[0] else None, "free_hbm_gb_rank0": free}
    sorted_ok = bool(np.all(np.diff(pairs["a"].astype(np.int64) * n + pairs["b"]) > 0)) if pairs.shape[0] > 1 else True
    out["sorted_unique"] = sorted_ok
    ctx.close()
    assert sorted_ok and np.all(pairs["kinship"] >= threshold)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, choices=(4, 5), required=True)
    ap.add_argument("--n", type=int, default=None)
    ap.add_argument("--l", type=int, default=None)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--threshold", type=float, default=0.0442)
    a = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    try:
        if a.config == 4:
            out = config4(local, a.n or 2504, a.l or 20_000_000, a.repeats)
        else:
            out = config5(local, rank, world, a.n or 100_000, a.l or 1_000_000, a.repeats, a.threshold)
        out.update(gpu_info(local))
        if rank == 0:
            print(json.dumps(out), flush=True)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
