#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json on N B200s of one node.

Metric: inbreeding genotype-loci/s (BASELINE.json `metric`) on config 2, the chr22 shape: 2,504 genomes x 1.1 M biallelic
SNPs, per-locus allele counts + per-genome inbreeding (Simple estimator: class counts, expected class-frequency sums, F)
with a gnomAD-style float AF vector per super-population. One "step" = one fused pass over one batch of synthetic input:
per-locus preparation from the AF vectors, the streaming kernel k_stream_count_ct over the 2-bit matrix, counter expansion,
moment assembly and the closed-form estimator.

  value : whole-job genotype-loci/s with the inputs resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e   : the same pass through the C ABI with HOST buffers: H2D of the packed matrix, AF vectors, super-populations and
          locus selection, and D2H of the per-locus counts and LocusResults inside the timed region
  N > 1 : weak scaling, every rank owns a locus shard of the same size; per-genome partial sums are all-reduced (NCCL)
          between the streaming pass and the estimator (SURVEY 8e).

`--impl reference` times the reference's own CPU implementation (oracle/_ref/kgl_ref_harness, the reference TUs
compiled where they lie; else the oracle port) on a bounded sample of the same workload, on the host cores.

`--dump-outputs DIR` writes, after the timed steps, the per-locus counts and per-genome results of the step as
DIR/<name>.npy (see dump_outputs and run_ours). The inputs depend on the arguments only, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line. Libraries write there too (NCCL prints "NCCL version ..." to stdout from C), so
# file descriptor 1 is pointed at stderr for the life of the process and the JSON line goes to a private copy of the
# original stdout. (NCCL_DEBUG is left as the caller set it.)
_JSON_FD = None


def claim_stdout():
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)

N_GENOMES = 2504
N_LOCI = 1_100_000
SEED = 20261018
METRIC = "inbreeding genotype-loci/s"
UNIT = "genotype-loci/s"
# Bounded samples of the reference CPU path (BASELINE.md section 4 / SURVEY 8d: 2,504 genomes x 50,000 loci; the reference
# cannot materialise config 2 as a PopulationDB). --impl reference times the BASELINE sample (~25 s per repeat on 15 threads);
# the cpu_baseline object of the GPU arm uses a 20,000-locus prefix of the same population (~10 s per repeat).
REFERENCE_SAMPLE = (2504, 50_000)
CPU_SAMPLE = (2504, 20_000)
DUMP_BYTES = 64_000_000     # --dump-outputs: at most this much in all, .npy headers included
DUMP_HEADER_BYTES = 4096    # what the headers of its (at most 14) files may take


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--genomes", type=int, default=N_GENOMES)
    ap.add_argument("--loci", type=int, default=N_LOCI)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-kinship", action="store_true")
    ap.add_argument("--no-estimators", action="store_true", help="skip the RitlandLocus / HallME / Loglikelihood timings")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the per-genome partial sums of the locus shards meet -- 'peer': inside the step's own kernel over "
                         "NVLink peer memory (CUDA IPC); 'nccl': an NCCL all-reduce between the step's kernels")
    ap.add_argument("--kinship-loci", type=int, default=20_000_000,
                    help="loci of the pairwise run (default: BASELINE config 4, 20 M SNPs; 0 = the resident chr22-shape matrix)")
    ap.add_argument("--kinship-steps", type=int, default=3)
    ap.add_argument("--reference-sample", default="", help="--impl reference: GENOMESxLOCI of the CPU sample (default 2504x50000, BASELINE.md section 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the per-locus counts and per-genome results of the step as DIR/<name>.npy "
                         "(one GPU: of one more run of the step; N > 1: of the last timed step, locus counts of rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    return args


def sample_rows(n_rows: int, row_bytes: int, room: int, seed: int):
    """None if n_rows rows of row_bytes fit in room bytes; else the sorted row numbers of a fixed sample, drawn with `seed`,
    that fits there together with the row numbers themselves (8 B per row)."""
    if n_rows * row_bytes <= room:
        return None
    return np.sort(np.random.default_rng(seed).choice(n_rows, size=max(1, room // (row_bytes + 8)), replace=False))


def dump_outputs(path, locus_counts, results):
    """Writes what one step of the timed path hands its caller: the per-locus allele counts uint32 [L, 4] as locus_counts.npy
    (float32, exact below 2^24 genomes) and every LocusResults field of every genome as genome_<field>.npy (float64), at most
    DUMP_BYTES in all. The per-genome arrays get at most half of that, the per-locus counts the rest; an array that does not
    fit its share holds a fixed sample of rows, drawn with the bench seed, and genome_rows.npy / locus_rows.npy their row
    numbers."""
    os.makedirs(path, exist_ok=True)
    out = {}
    room = DUMP_BYTES - DUMP_HEADER_BYTES
    rows = sample_rows(results.shape[0], 8 * len(results.dtype.names), room // 2, SEED)
    if rows is not None:
        out["genome_rows"] = rows.astype(np.float64)
        results = results[rows]
    out.update({"genome_" + f: results[f].astype(np.float64) for f in results.dtype.names})
    room -= sum(a.nbytes for a in out.values())
    rows = sample_rows(locus_counts.shape[0], 16, room, SEED + 1)
    if rows is not None:
        out["locus_rows"] = rows.astype(np.float64)
        locus_counts = locus_counts[rows]
    out["locus_counts"] = locus_counts.astype(np.float32)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def stream_kernel_name(n_genomes: int) -> str:
    """The streaming kernel plan_stream picks for this width (kgl_gene_b200/csrc/stream_common.cuh)."""
    units = (n_genomes + 63) // 64
    if units > 56:
        units = (units + 39) // 40 * 40
    if units == 8:
        return "k_stream_count_ct<8,256>"
    if units % 40 == 0:
        return "k_stream_count_ct<40,64>" + (f" x {units // 40} slices" if units > 40 else "")
    return "k_stream_count_rt (runtime shape)"


def workload_name(n, l, world):
    base = f"1000G chr22 shape: {n} genomes x {l} biallelic SNPs, per-locus allele counts + Simple inbreeding, 6 float AF vectors"
    return base if world == 1 else base + f" per GPU (locus-sharded, {world} shards, partial sums all-reduced)"


# --------------------------------------------------------------------------------------------- CPU baseline ---------
def cpu_reference_run(repeat: int, sample=None):
    """Times the reference CPU path on the bounded sample. Returns dict(value, cores, kind, sample, seconds list)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    n, l = sample or CPU_SAMPLE
    offsets, af = make_loci(l, SEED)                      # the bench generator: the first l loci of the population the GPU arm times
    superpop, inbreeding = make_genomes(n, SEED)
    pop = FlatPopulation(offsets, af, superpop, O.synth_genotypes(SEED, n, l, af, superpop, inbreeding), n, False)
    cells = float(n) * float(l)
    if O.have_reference_harness():
        out = O.run_reference(pop, algos=("Simple",), variantdb=False, repeat=repeat, timeout=3000)
        secs = [float(s) for s in out["Simple_repeat_seconds"]]
        cores = int(out["meta"][0])
        kind = "reference"
        what = (f"reference TUs (kga_inbreed processSimple + generateFrequencies) via WorkflowThreads({cores}) on {n} genomes x {l} loci "
                f"drawn from the bench generator; fan-out/future.get() loop timed, PopulationDB construction excluded")
    else:
        sel = O.select_all_pops(pop)
        secs = []
        for _ in range(repeat):
            t0 = time.perf_counter()
            O.inbreed(pop, sel, "Simple")
            secs.append(time.perf_counter() - t0)
        cores = O.threads()
        kind = "port"
        what = f"oracle C port (OpenMP, {cores} threads) on {n} genomes x {l} loci drawn from the bench generator"
    return dict(cells=cells, seconds=secs, cores=cores, kind=kind, sample=what)


def cpu_port_run():
    """SURVEY 8d (ii), the "fair CPU" line: the flat C restatement (oracle/kgl_oracle.c, OpenMP over genomes) doing counts +
    Simple on a bounded sample of the same generator, all host threads. Reported next to the reference figure; never the
    thing measured as the product."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    from kgl_gene_b200.flatfile import FlatPopulation
    from kgl_gene_b200.synth import make_genomes, make_loci
    n, l = 2504, 40_000
    offsets, af = make_loci(l, SEED)
    superpop, inbreeding = make_genomes(n, SEED)
    pop = FlatPopulation(offsets, af, superpop, O.synth_genotypes(SEED, n, l, af, superpop, inbreeding), n, False)
    sel = O.select_all_pops(pop)
    O.inbreed(pop, sel, "Simple")
    secs = []
    for _ in range(3):
        t0 = time.perf_counter()
        O.allele_count(pop)
        O.inbreed(pop, sel, "Simple")
        secs.append(time.perf_counter() - t0)
    cores = O.threads()
    return {"value": float(n) * float(l) / float(np.median(secs)), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle C restatement on the flat 2-bit matrix (OpenMP, {cores} threads): allele counts + Simple on {n} genomes x {l} loci of the bench generator"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warm = min(args.warmup, 1)                            # at most one untimed repeat: the reference has no caches to warm
    repeats = warm + args.steps
    sample = REFERENCE_SAMPLE
    if args.reference_sample:
        sample = tuple(int(x) for x in args.reference_sample.lower().split("x"))
    r = cpu_reference_run(repeats, sample)
    secs = r["seconds"][warm:]
    mean = float(np.mean(secs))
    value = r["cells"] / mean
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(secs),
        "warmup": warm, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.genomes, args.loci, 1),
                   "note": "reference CPU path timed on a bounded sample of this workload (BASELINE.md section 4: 2,504 genomes x 50,000 loci); "
                           "value is per-unit throughput"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# --------------------------------------------------------------------------------------------------- clocks ---------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class RawCudaArray:
    def __init__(self, ptr: int, n: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


# ----------------------------------------------------------------------------------------------------- ours ---------
def run_ours(args):
    import ctypes as C

    import torch
    import torch.distributed as dist
    from kgl_gene_b200.capi import KglB200, RESULT_DTYPE
    from kgl_gene_b200.flatfile import row_bytes_for
    from kgl_gene_b200.synth import make_genomes, make_loci

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    n, l = args.genomes, args.loci
    rb = row_bytes_for(n)
    ctx = KglB200(local_rank)
    # a real (non-default) stream: the C ABI treats a NULL handle as "use the context's own stream", and CUDA events must
    # be recorded on the stream the kernels run on
    stream = torch.cuda.Stream(device=dev, priority=-1)      # the streaming kernel's stream outranks the context's side streams
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)

    # ---- synthetic shard, generated on the device (SURVEY 8d): same genomes on every rank, rank-specific loci ----
    offsets, af = make_loci(l, SEED + 1000 * rank)
    superpop, inbreeding = make_genomes(n, SEED)
    ctx.upload_loci(af, offsets)
    ctx.set_genome_superpop(superpop)
    ctx.synth_genotypes(SEED, n, l, inbreeding, missing_rate=0.001, locus_base=rank * l)
    ctx.select_loci()                      # one window = all loci (LociiCount = inf, SamplingDistance = 0, AF in [0,1])

    def allreduce_partials():
        ptr, cnt = ctx.inbreed_partials_buffer()
        t = torch.as_tensor(RawCudaArray(ptr, cnt, "<f8"), device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)

    def step_nccl():
        ctx.inbreed_begin("Simple", count_loci=True)
        ctx.inbreed_accumulate()
        allreduce_partials()
        ctx.inbreed_update()

    use_peer = world > 1 and args.exchange == "peer"
    exchange_note = args.exchange
    if use_peer:
        # exchange regions of all ranks, mapped into every rank once (CUDA IPC handles travel over the process group)
        from kgl_gene_b200.capi import KglError
        handles = [None] * world
        dist.all_gather_object(handles, ctx.peer_export())
        attached = torch.ones(1, device=dev, dtype=torch.int32)
        try:
            ctx.peer_attach(rank, world, handles)
        except KglError as ex:        # e.g. a container that forbids CUDA IPC between its processes
            attached.zero_()
            sys.stderr.write(f"bench.py: rank {rank}: peer_attach failed ({ex}); the ranks fall back to --exchange nccl\n")
        dist.all_reduce(attached, op=dist.ReduceOp.MIN)
        if int(attached.item()) == 0:
            use_peer = False
            exchange_note = "nccl (CUDA IPC peer mapping unavailable on this box)"
    if use_peer:
        # the fused exchange against the NCCL path, once, before anything is timed
        step_nccl()
        want = ctx.inbreed_fetch()
        ctx.enqueue_count_and_inbreed_peer()
        got = ctx.inbreed_fetch()
        for fld in ("major_homo_count", "major_hetero_count", "minor_homo_count", "minor_hetero_count", "total_allele_count"):
            assert np.array_equal(got[fld], want[fld]), fld
        assert np.max(np.abs(got["inbred_allele_sum"] - want["inbred_allele_sum"])) < 1e-12, "peer exchange differs from the NCCL all-reduce"

    def step_resident():
        if world == 1:
            ctx.enqueue_count_and_inbreed()
        elif use_peer:
            ctx.enqueue_count_and_inbreed_peer()
        else:
            step_nccl()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        ctx.flush()              # the tail of the last pass runs on a side stream: the closing event is ordered after it
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- resident timing ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    ctx.kernel_timer_reset()
    launches0 = ctx.launch_count()
    total_ms = timed(step_resident, args.steps, 0)
    launches = ctx.launch_count() - launches0
    kernel_ms = ctx.kernel_timer_read()
    clocks = sampler.stop() if rank == 0 else None
    cells = float(n) * float(l) * world
    value = cells * args.steps / (total_ms * 1e-3)

    # ---- parity spot check of the resident result (size-independent invariants; full parity lives in tests/) ----
    res = ctx.inbreed_fetch() if world > 1 else None
    lc = ctx.fetch_locus_counts()
    assert int(lc.sum()) == n * l and np.all(lc.sum(axis=1) == n), "per-locus counts do not add up to the genome count"
    if args.dump_outputs:
        if world == 1:
            # The C ABI hands the per-genome results of a single-GPU pass to the host only through the one-call form of the
            # same pass (kgl_b200_run_count_and_inbreed): what is written comes from one more run of the step, whose per-locus
            # counts must equal those of the last timed step.
            lc_again, res = ctx.count_and_inbreed()
            assert np.array_equal(lc_again, lc), "a repeated pass gives other per-locus counts"
        if rank == 0:
            dump_outputs(args.dump_outputs, lc, res)

    # ---- end to end through the C ABI with host buffers ----
    e2e = None
    if not args.no_e2e:
        h_packed = torch.empty((l, rb), dtype=torch.uint8, pin_memory=True)
        ctx._check(ctx.lib.kgl_b200_download_genotypes(ctx.h, C.c_uint64(l * rb), C.c_void_p(h_packed.data_ptr())), "download_genotypes")
        h_af = torch.from_numpy(af).pin_memory()
        h_lc = torch.empty((l, 4), dtype=torch.int32, pin_memory=True)
        h_res = torch.empty((n * RESULT_DTYPE.itemsize,), dtype=torch.uint8, pin_memory=True)
        af_np, off_np = h_af.numpy(), offsets

        def step_e2e():
            ctx.upload_genotypes_ptr(h_packed.data_ptr(), n, l, rb)
            ctx.upload_loci(af_np, off_np)
            ctx.set_genome_superpop(superpop)
            ctx.select_loci()
            if world == 1:
                ctx.count_and_inbreed_into(h_lc.data_ptr(), h_res.data_ptr())
            else:
                if use_peer:
                    ctx.enqueue_count_and_inbreed_peer()
                else:
                    step_nccl()
                ctx._check(ctx.lib.kgl_b200_inbreed_fetch(ctx.h, C.c_void_p(h_res.data_ptr())), "inbreed_fetch")
                ctx._check(ctx.lib.kgl_b200_fetch_locus_counts(ctx.h, C.c_void_p(h_lc.data_ptr())), "fetch_locus_counts")

        e2e_steps = max(3, min(args.steps, 10))
        e2e_ms = timed(step_e2e, e2e_steps, 2)
        h2d = l * rb + af.nbytes + offsets.nbytes + n      # matrix, AF vectors, locus offsets, super-populations (the selection is made on the device)
        d2h = 16 * l + RESULT_DTYPE.itemsize * n
        e2e = {"value": cells * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps}
        lc2 = h_lc.numpy().view(np.uint32)
        assert np.array_equal(lc2, lc), "e2e per-locus counts differ from the resident run"
        # What the host can deliver: the matrix alone, one cudaMemcpyAsync from the same pinned buffer, every rank at once (the
        # ranks of one box share its memory controllers and PCIe switches: the e2e step is this copy plus ~1 ms)
        d_tmp = torch.empty((l, rb), dtype=torch.uint8, device=dev)
        bare_ms = timed(lambda: d_tmp.copy_(h_packed, non_blocking=True), 3, 1) / 3
        e2e["bare_matrix_h2d_ms"] = bare_ms
        e2e["bare_matrix_h2d_gbs_per_gpu"] = l * rb / (bare_ms * 1e-3) / 1e9
        e2e["bare_matrix_h2d_gbs_all_gpus"] = world * l * rb / (bare_ms * 1e-3) / 1e9
        del d_tmp
        if world == 1:
            # The plugin's real shape (kga_analysis_inbreed_b200.cpp): ONE upload per iteration, then the window loop for every
            # parameter block -- here 20 windows of 55,000 loci x the four algorithms, results fetched to the host per window.
            n_windows, per = 20, l // 20
            t0 = time.perf_counter()
            ctx.upload_genotypes_ptr(h_packed.data_ptr(), n, l, rb)
            ctx.upload_loci(af_np, off_np)
            ctx.set_genome_superpop(superpop)
            ctx.synchronize()
            t_upload = time.perf_counter() - t0
            def window_loop():
                per_algo = {}
                t1 = time.perf_counter()
                for algorithm in ("Simple", "RitlandLocus", "HallME", "Loglikelihood"):
                    t2 = time.perf_counter()
                    for w in range(n_windows):
                        ctx.select_loci(lower=int(off_np[w * per]), upper=int(off_np[min(l, (w + 1) * per) - 1]))
                        ctx.inbreed(algorithm)
                    per_algo[algorithm] = (time.perf_counter() - t2) * 1e3
                return per_algo, (time.perf_counter() - t1) * 1e3
            first_algo, first_ms = window_loop()        # buffers of the context grow to the window sizes here (cudaMalloc)
            per_algo, loop_ms = window_loop()
            total = t_upload + loop_ms * 1e-3
            e2e["plugin_shape"] = {"windows": n_windows, "loci_per_window": per, "algorithms": 4, "upload_ms": t_upload * 1e3,
                                   "ms_per_algorithm": per_algo, "ms_total": total * 1e3,
                                   "ms_per_algorithm_first_pass": first_algo, "ms_total_first_pass": t_upload * 1e3 + first_ms,
                                   "genotype_loci_per_s": 4.0 * n * per * n_windows / total,
                                   "note": "one upload (matrix, AF, super-populations), then select_loci + run_inbreed with host results "
                                           "for every window and algorithm; host wall clock; the first pass over the windows also "
                                           "grows the context's buffers"}
            ctx.select_loci()                  # back to one window = all loci for what follows

    hbm_peak = 6650.0
    try:
        hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
    except Exception:
        pass
    est = None
    if not args.no_estimators:
        est = run_estimators(ctx, torch, dist, dev, stream, world, n, l, rb, allreduce_partials, hbm_peak)

    kin = None
    if not args.no_kinship:
        kin = run_kinship(args, ctx, torch, dist, dev, stream, rank, world, timed, n, l, rb, SEED, superpop, inbreeding)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        k_ms = float(np.mean(kernel_ms)) if len(kernel_ms) else None
        # algorithmic bytes of one k_stream_count launch: 2 bits per genotype + 2 B selection flags and 16 B of counts per locus
        alg_bytes = n * l / 4.0 + 2.0 * l + 16.0 * l
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms else None
        traffic = None
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "k_stream_count_traffic.json")))
            if prof.get("n_genomes") == n and prof.get("n_loci") == l:
                traffic = prof.get("dram_bytes_per_launch")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64 bit-planes + f64 sums", "data": "synthetic",
            "config": {"workload": workload_name(n, l, world), "n_genomes": n, "n_loci_per_gpu": l, "af_vectors": int(af.shape[0]),
                       "selection": "one window, all loci", "missing_rate": 0.001,
                       "l2": f"inputs ({l * rb / 1e6:.0f} MB matrix per GPU) are larger than the 126 MB L2; no flush needed",
                       "step": "k_locus_prepare (flags, dense totals, rare-major rows; side stream, next to the previous pass's streaming kernel) + k_stream_count_ct (per-locus counts, per-genome counts) + k_tail (code-3 cells, moments, Simple closed form; side stream, next to the next pass's streaming kernel)"
                               + ("" if world == 1 else (" + k_peer_exchange (signal, wait, gather the partial sums of all ranks over NVLink peer memory, fixed-order sum, closed form; no NCCL call in the step)"
                                                         if use_peer else " + NCCL all-reduce + k_finalize_closed_form")),
                       "exchange": None if world == 1 else exchange_note},
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": stream_kernel_name(n), "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                         "frac": (achieved / peak_gbs) if achieved else None, "traffic": traffic, "peak_source": peak_src,
                         "kernel_ms": k_ms, "kernel_share_of_step": (k_ms * len(kernel_ms) / total_ms) if k_ms else None,
                         "algorithmic_bytes_per_launch": alg_bytes},
            "clocks": clocks,
        }
        if est is not None:
            line["estimators"] = est
        if kin is not None:
            line["kinship"] = kin
        if not args.no_cpu_baseline and world == 1:
            try:
                r = cpu_reference_run(2)
                secs = r["seconds"][1:] or r["seconds"]
                line["cpu_baseline"] = {"value": r["cells"] / float(np.mean(secs)), "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                        "sample": r["sample"]}
            except Exception as ex:  # the baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {ex}"}
            try:
                line["cpu_baseline_port"] = cpu_port_run()
            except Exception as ex:
                line["cpu_baseline_port"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {ex}"}
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def run_estimators(ctx, torch, dist, dev, stream, world, n, l, rb, allreduce_partials, hbm_peak):
    """The other three estimators of kga_inbreed on the resident shard. `ms` is the whole estimator on a FRESH selection: the
    counting pass, the per-selection tables of the iterative estimators (terms_moments.cuh: sort, payload tiles, the tensor-core
    pass over the matrix, lists) and all sweeps. One GPU: kgl_b200_run_inbreed (all sweeps in one launch); N > 1: the
    accumulate / all-reduce / update protocol, sweep by sweep."""
    out = {}

    def timed_call(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        r = fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), r

    def protocol(algorithm, **kw):
        ctx.inbreed_begin(algorithm, **kw)
        finished, sweeps = False, 0
        while not finished:
            ctx.inbreed_accumulate()
            if world > 1:
                allreduce_partials()
            finished = ctx.inbreed_update()
            sweeps += 1
        return sweeps

    for algorithm in ("RitlandLocus", "HallME", "Loglikelihood"):
        iterative = algorithm != "RitlandLocus"
        run = (lambda **kw: ctx.inbreed(algorithm, **kw)) if world == 1 else (lambda **kw: protocol(algorithm, **kw))
        run()                                   # warm-up: buffers, derived copies
        ctx.select_loci()                       # a fresh selection (untimed): nothing of the run before is reused
        if world > 1:
            dist.barrier()
        cold, _ = timed_call(run)
        cached, _ = timed_call(run)             # same selection again: the tables are reused
        t = torch.tensor([cold, cached], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        cold, cached = float(t[0].item()), float(t[1].item())
        cells = float(n) * float(l) * world
        o = {"ms": cold, "genotype_loci_per_s": cells / (cold * 1e-3), "ms_same_selection_again": cached}
        if iterative:
            path = ctx.used_moment_tables()
            o["sweeps_from"] = {0: "exact kernels (every cell in every sweep)", 1: "moment tables, built on the CUDA cores",
                                2: "moment tables, built on the tensor cores (k_mom_mma)"}[path]
            exact, _ = timed_call(lambda: run(exact_sweeps=True))
            o["ms_exact_sweeps"] = exact          # round-1 path: k_terms_fast, N x L reciprocals per sweep
            build = max(cold - cached, 1e-6)
            matrix_bytes = float(l) * rb
            o["roofline"] = {"bound": "hbm", "kernel": "table build (k_mom_keys, radix sort, k_mom_btiles, k_mom_mma, lists): one pass over the matrix",
                             "achieved": matrix_bytes / (build * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": matrix_bytes / (build * 1e-3) / 1e9 / hbm_peak, "build_ms": build,
                             "note": "algorithmic bytes = one read of the 2-bit matrix; the sweeps read the tables only"}
        out[algorithm] = o
    return out


def timed_local(ctx, torch, stream, fn, steps):
    """CUDA-event timing of `steps` calls on this rank's stream (no cross-rank barrier)."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


KINSHIP_METRIC = "kinship sample-pair-loci/s"
LOP3_PER_CLK_SM = 62.45      # measured, profiles/r01_pipe_rates_kbench.log (kgl_gene_b200/csrc/tools/kbench.cu)
POPC_PER_CLK_SM = 15.90


def run_kinship(args, ctx, torch, dist, dev, stream, rank, world, timed, n, l, rb, seed, superpop, inbreeding):
    """BASELINE.json's second metric: pairwise IBS over all sample pairs; 64 x 64 tiles of the upper triangle dealt round-robin
    to the ranks, every rank holds the whole matrix, no collective in the data path (SURVEY 8e)."""
    from kgl_gene_b200.shards import block_tile_coords, tiles_of_rank
    from kgl_gene_b200.synth import make_loci
    kl = args.kinship_loci or l
    if world > 1 or kl != l:
        # the pairwise job needs the SAME population on every rank (the inbreeding job above holds one locus shard per rank)
        offsets, af = make_loci(kl, seed)
        ctx.upload_loci(af, offsets)
        ctx.set_genome_superpop(superpop)
        ctx.synth_genotypes(seed, n, kl, inbreeding, missing_rate=0.001, locus_base=0)
    side, n_up = ctx.ibs_tile_grid()
    SLAB = 8192
    # N > 1: whole 256 x 256 blocks of tiles are dealt to the ranks (shards.block_tile_coords), the unit of the tensor-core form
    coords = block_tile_coords(n, rank, world) if world > 1 else None
    mine = tiles_of_rank(n_up, rank, world) if coords is None else int(coords.shape[0])

    def step():
        done = 0
        while done < mine:
            k = min(SLAB, mine - done)
            if coords is None:
                ctx.enqueue_ibs_tiles(done, 1, k)
            else:
                ctx.enqueue_ibs_tile_list(coords[done:done + k])
            done += k

    step()                                   # builds the sample-major planes once (part of the upload, not of a pass)
    torch.cuda.synchronize()
    ctx.ibs_timer_reset()
    launches0 = ctx.launch_count()
    steps = max(1, args.kinship_steps)
    ms = timed(step, steps, 1)
    k_ms = ctx.ibs_timer_read()
    launches = ctx.launch_count() - launches0
    pair_loci = float(n) * (n + 1) / 2.0 * kl
    value = pair_loci * steps / (ms * 1e-3)
    # end to end: host matrix in, host tiles out
    e2e = None
    if not args.no_e2e and world == 1 and mine <= SLAB and kl * rb <= 16e9:     # 12.5 GB of pinned host memory at 20 M loci
        import ctypes as C
        try:
            h_packed = torch.empty((kl, rb), dtype=torch.uint8, pin_memory=True)
            ctx._check(ctx.lib.kgl_b200_download_genotypes(ctx.h, C.c_uint64(kl * rb), C.c_void_p(h_packed.data_ptr())), "download_genotypes")
            h_tiles = torch.empty((mine, 64, 64, 4), dtype=torch.int32, pin_memory=True)

            def step_e2e():
                # the whole job from host buffers: matrix in (PCIe), derived copies (sample-major planes, code-3 index, 2-bit code
                # matrix, class counts), the three Gram matrices, sparse repair, tiles out
                ctx.upload_genotypes_ptr(h_packed.data_ptr(), n, kl, rb)
                ctx._check(ctx.lib.kgl_b200_run_ibs_tiles(ctx.h, C.c_uint64(0), C.c_uint64(1), C.c_uint64(mine), C.c_void_p(h_tiles.data_ptr())), "run_ibs_tiles")

            e_ms = timed(step_e2e, 2, 1)
            e2e = {"value": pair_loci * 2 / (e_ms * 1e-3), "unit": "sample-pair-loci/s", "h2d_bytes_per_step": int(kl * rb),
                   "d2h_bytes_per_step": int(h_tiles.numel() * 4), "ms_per_step": e_ms / 2, "steps": 2}
            t = h_tiles.numpy().view(np.uint32)
            assert np.array_equal(t[..., :3].sum(-1), t[..., 3]), "IBS0 + IBS1 + IBS2 != valid"
            del h_packed, h_tiles
        except RuntimeError as ex:       # no room for the pinned copy of the matrix on this host
            e2e = {"value": None, "unit": "sample-pair-loci/s", "note": f"skipped: {str(ex)[:120]}"}
    # tensor-core variant (K5): the dosage Gram matrix of the same population, int8 x int8 -> int32 on tcgen05. At N > 1 the
    # 256 x 256 tiles are dealt to the ranks and the int32 matrix is assembled with one NCCL all-reduce (26 MB at 2,504 genomes).
    from kgl_gene_b200.shards import allreduce_gram

    def gram_step():
        ctx.enqueue_gram_tiles(rank, world)
        if world > 1:
            allreduce_gram(ctx, dev)

    gram_step()
    g_ms = timed(gram_step, steps, 1) / steps
    grm = None
    if rank == 0:
        gk_ms = ctx.last_gram_kernel_ms()
        ld = (n + 255) // 256 * 256
        n_tiles_all = sum(1 for ti in range(ld // 256) for tj in range(ti, ld // 256))
        n_tiles = len(range(rank, n_tiles_all, world))
        k_stages = (kl + 127) // 128
        ops = 2.0 * n_tiles * 256 * 256 * k_stages * 128
        # int8 tensor peak: MEASURED on this pool's B200s with the kernel's own MMA issue loop and epilogue, operand staging switched
        # off (tools/grambench --skip 2, profiles/r01_grambench_skip_modes.log: 3512 / 3567 TOP/s at 2504 x 1.1 M / 8192 x 400 k)
        peak_tops = 3567.3
        grm = {"metric": "kinship sample-pair-loci/s (int8 Gram matrix on tcgen05)", "value": pair_loci / (g_ms * 1e-3), "unit": "sample-pair-loci/s",
               "ms_per_step": g_ms, "n_gpus": world, "scaling": "strong",
               "kernel": "k_gram_i8 (tcgen05.mma kind::i8, TMEM accumulators, 256x256 tiles = two M128 MMAs per B operand, in-kernel 2-bit -> int8 expansion)",
               "roofline": {"bound": "tensor", "achieved": ops / (gk_ms * 1e-3) / 1e12, "peak": peak_tops, "unit": "int8 TOP/s",
                            "frac": ops / (gk_ms * 1e-3) / 1e12 / peak_tops,
                            "peak_source": "measured: tcgen05.mma kind::i8 128x256x32 issued back to back + epilogue, no operand staging (profiles/r01_grambench_skip_modes.log)",
                            "kernel_ms": gk_ms, "twice_measured_bf16_tops": 2.0 * 1608.9}}
    if rank != 0:
        return None
    clk = 1.965e9
    sms = 148
    launches_per_step = (mine + SLAB - 1) // SLAB
    k_s = float(np.mean(k_ms)) * launches_per_step * 1e-3 if len(k_ms) else None   # the timer ring also holds the warm-up step
    lop3_peak = LOP3_PER_CLK_SM * sms * clk / 5.0 * 32.0
    if ctx.ibs_used_tensor_cores():
        # dense part = three exact int8 Gram matrices (dosage, heterozygous, hom-alt indicators) over this rank's 256 x 256 blocks
        bs = ((n + 63) // 64 + 3) // 4
        n_blocks = len(range(rank, bs * (bs + 1) // 2, world))
        ops = 3 * 2.0 * n_blocks * 256 * 256 * ((kl + 127) // 128) * 128
        achieved = ops / k_s / 1e12 if k_s else None
        roof = {"bound": "tensor", "kernel": "3 x k_gram_i8 (tcgen05.mma kind::i8; dosage, heterozygous and hom-alt indicator Gram matrices) + k_ibs_from_grams "
                                             "(+ k_ibs_missing_fix, k_ibs_finalize outside the timed kernels)",
                "achieved": achieved, "peak": 3567.3, "unit": "int8 TOP/s", "frac": (achieved / 3567.3) if achieved else None,
                "peak_source": "measured: tcgen05.mma kind::i8 issued back to back + epilogue, no operand staging (profiles/r01_grambench_skip_modes.log)",
                "kernel_ms": k_s * 1e3 if k_s else None,
                "popcount_kernel_bound_pair_loci_per_s": lop3_peak,
                "note": "IBS0 / IBS1 follow exactly from the three matrices and the per-genome class counts (ibs_gram.cuh): 1.5 N^2 L int8 MACs "
                        "instead of 5 LOP3 + 1 POPC per pair-word; round 1's popcount tile kernel (8.5e13 pair-loci/s, 0.73 of its LOP3 bound on "
                        "useful pair-loci) remains for populations whose matrices do not fit or whose code-3 cells are not indexed"}
    else:
        # INT-pipe roofline of the tile kernel: 5 LOP3 + 1 POPC per executed pair-word (two-plane form: 3 for the two difference
        # vectors, 2 for the carry-save step); the ALU pipe issues 62.45 LOP3 per clk per SM (measured), POPC 15.9.
        exec_pair_loci = float(mine) * 4096 * kl                   # this rank's launches, incl. padding genomes and diagonal halves
        achieved = exec_pair_loci / k_s if k_s else None
        roof = {"bound": "int-pipe (ALU/LOP3)", "kernel": "k_ibs_tiles<false,2> (+ k_ibs_missing_fix, k_ibs_finalize)",
                "achieved": achieved, "peak": lop3_peak, "unit": "executed pair-loci/s",
                "frac": (achieved / lop3_peak) if achieved else None,
                # on USEFUL pair-loci (N (N + 1) / 2 pairs: no padding genomes, diagonal tiles counted once), whole step
                "frac_useful": value / world / lop3_peak,
                "peak_source": "62.45 LOP3/clk/SM (measured, kbench) x 148 SMs x 1.965 GHz / 5 LOP3 per 32 pair-loci",
                "survey_8d_peak_popc_bound": POPC_PER_CLK_SM * sms * clk / 3.0 * 32.0,
                "kernel_ms": k_s * 1e3 if k_s else None}
    return {"metric": KINSHIP_METRIC, "value": value, "unit": "sample-pair-loci/s", "ms_per_step": ms / steps, "steps": steps,
            "n_gpus": world, "scaling": "strong",
            "config": {"workload": f"pairwise IBS0/IBS1/IBS2/valid, {n} x {n} genomes over {kl} SNPs (BASELINE config 4 shape: 20 M SNPs), "
                                   f"upper-triangle 64x64 tiles, whole 256x256 blocks of them dealt to {world} GPU(s)",
                       "tiles": int(n_up), "tiles_this_rank": int(mine), "missing_rate": 0.001},
            "e2e": e2e, "gpu_launches": int(launches), "grm_i8": grm, "roofline": roof}


def main():
    args = parse_args()
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
