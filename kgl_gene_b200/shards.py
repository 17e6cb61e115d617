"""Partitioning of the hot path over the GPUs of one node (SURVEY 8e), host-side logic only.

* inbreeding / allele counts: loci are cut into contiguous shards, one per rank. Per-locus counts need no exchange; the
  per-genome partial sums (16 doubles per genome) are additive over shards and are all-reduced (SUM) between the
  streaming pass and the estimator -- `allreduce_partials`.
* pairwise IBS: the 64 x 64 sample-pair tiles of the upper triangle are dealt round-robin to the ranks (tile t belongs to
  rank t mod world); every rank holds the whole packed matrix; no collective in the data path. `gather_ibs` collects the
  compact tile blocks and `assemble_ibs` lays them out as the symmetric genome x genome matrix.
* KING related-pair lists: the same tiles (block_tile_coords) go to kgl_b200_run_king_pairs on each rank; `gather_king_pairs`
  joins the ranks' lists.

Everything here works on CPU tensors with the gloo backend as well (tests/test_shards_gloo.py) -- the CUDA context is only
touched through the KglB200 object the caller passes in.
"""
from __future__ import annotations

import numpy as np

TILE = 64


# ---------------------------------------------------------------------------------------------- locus shards ---------
def locus_shard(n_loci: int, rank: int, world: int, align: int = 256) -> tuple[int, int]:
    """[begin, end) of rank's contiguous locus shard; shard boundaries are multiples of `align` rows (the streaming
    kernel's stage height) except the last end."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    blocks = (n_loci + align - 1) // align
    b0 = blocks * rank // world
    b1 = blocks * (rank + 1) // world
    return min(b0 * align, n_loci), min(b1 * align, n_loci)


class _RawCudaArray:
    def __init__(self, ptr: int, n: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}


def bind_to_current_stream(ctx, device):
    """Orders the context's kernels with the collectives torch issues on `device`.

    dist.all_reduce is ordered against torch's CURRENT stream only, while a context enqueues on its own non-blocking stream
    unless told otherwise. With a real torch stream current, the context is bound to it (kgl_b200_set_stream) and stream
    order does the rest: returns None. With the legacy default stream current -- handle 0, which the C ABI reads as "the
    context's own stream" -- the two cannot share a stream: returns that stream and the helpers below synchronise explicitly
    on both sides of the collective."""
    import torch
    s = torch.cuda.current_stream(device)
    if s.cuda_stream != 0:
        ctx.set_stream(s.cuda_stream)
        return None
    return s


def _allreduce_device_buffer(ctx, ptr, count, typestr, device, group):
    import torch
    import torch.distributed as dist
    fence = bind_to_current_stream(ctx, device)
    if fence is not None:
        ctx.synchronize()                 # the buffer is complete before the collective reads it
    t = torch.as_tensor(_RawCudaArray(ptr, count, typestr), device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    if fence is not None:
        fence.synchronize()               # ... and reduced before the context's next kernel reads it


def allreduce_partials(ctx, device, group=None):
    """SUM all-reduce of the context's per-genome partial-sum buffer across the ranks (NCCL on the context's GPU), ordered
    after the kernels that fill it and before the ones that consume it (bind_to_current_stream)."""
    ptr, count = ctx.inbreed_partials_buffer()
    _allreduce_device_buffer(ctx, ptr, count, "<f8", device, group)


def run_inbreed_sharded(ctx, algorithm: str, device, group=None, **options):
    """The estimator state machine of the C ABI with the all-reduce in the middle: every rank holds a locus shard."""
    bind_to_current_stream(ctx, device)
    ctx.inbreed_begin(algorithm, **options)
    finished = False
    while not finished:
        ctx.inbreed_accumulate()
        allreduce_partials(ctx, device, group)
        finished = ctx.inbreed_update()
    return ctx.inbreed_fetch()


def allreduce_gram(ctx, device, group=None):
    """SUM all-reduce of the context's int32 Gram matrix: every rank computed the tiles rank, rank + world, ... and left
    the rest zero (kgl_b200_enqueue_gram_tiles)."""
    ptr, count, _ = ctx.gram_buffer()
    _allreduce_device_buffer(ctx, ptr, count, "<i4", device, group)


# ------------------------------------------------------------------------------------------------ IBS tiles ----------
def tile_side(n_genomes: int) -> int:
    return (n_genomes + TILE - 1) // TILE


def n_upper_tiles(n_genomes: int) -> int:
    s = tile_side(n_genomes)
    return s * (s + 1) // 2


def tiles_of_rank(n_upper: int, rank: int, world: int) -> int:
    """Number of tiles rank owns when tile t goes to rank t mod world."""
    return 0 if rank >= n_upper else (n_upper - rank + world - 1) // world


def upper_tile_coords(n_genomes: int) -> np.ndarray:
    """(ti, tj) of every upper-triangle tile in the C ABI's order (row-major, ti <= tj): int64[n_upper][2]."""
    s = tile_side(n_genomes)
    ti, tj = np.triu_indices(s)
    return np.stack([ti, tj], axis=1).astype(np.int64)


BLOCK_TILES = 4     # 64-genome tiles per side of a 256 x 256 block: the unit the tensor-core form of the dense part computes


def block_tile_coords(n_genomes: int, rank: int, world: int) -> np.ndarray:
    """(ti, tj) of the upper-triangle 64x64 tiles inside the 256 x 256 blocks rank owns when upper-triangle block b goes to rank
    b mod world (blocks row-major, bi <= bj): uint32[n][2], for kgl_b200_enqueue_ibs_tile_list. Dealing whole blocks keeps the
    tensor-core Gram work of a rank proportional to its tiles (a strided deal of single tiles touches every block on every rank)."""
    side = tile_side(n_genomes)
    bside = (side + BLOCK_TILES - 1) // BLOCK_TILES
    out = []
    b = 0
    for bi in range(bside):
        for bj in range(bi, bside):
            if b % world == rank:
                for ti in range(bi * BLOCK_TILES, min(side, (bi + 1) * BLOCK_TILES)):
                    for tj in range(bj * BLOCK_TILES, min(side, (bj + 1) * BLOCK_TILES)):
                        if ti <= tj:
                            out.append((ti, tj))
            b += 1
    return np.asarray(out, dtype=np.uint32).reshape(-1, 2)


def assemble_ibs_coords(n_genomes: int, coords_by_rank: list[np.ndarray], tiles_by_rank: list[np.ndarray]) -> np.ndarray:
    """Tiles with explicit coordinates (block_tile_coords) -> uint32[N][N][4], symmetric."""
    n = n_genomes
    out = np.zeros((n, n, 4), dtype=np.uint32)
    for coords, tiles in zip(coords_by_rank, tiles_by_rank):
        for (ti, tj), t in zip(coords.tolist(), tiles):
            a0, b0 = ti * TILE, tj * TILE
            a1, b1 = min(n, a0 + TILE), min(n, b0 + TILE)
            out[a0:a1, b0:b1] = t[: a1 - a0, : b1 - b0]
            out[b0:b1, a0:a1] = t[: a1 - a0, : b1 - b0].transpose(1, 0, 2)
    return out


def assemble_ibs(n_genomes: int, blocks_by_rank: list[np.ndarray]) -> np.ndarray:
    """blocks_by_rank[r] = uint32[tiles_of_rank(r)][64][64][4], the tiles r, r + world, ... -> uint32[N][N][4], symmetric."""
    world = len(blocks_by_rank)
    coords = upper_tile_coords(n_genomes)
    n_up = coords.shape[0]
    s = tile_side(n_genomes)
    full = np.zeros((s * TILE, s * TILE, 4), dtype=np.uint32)
    for r, blocks in enumerate(blocks_by_rank):
        want = tiles_of_rank(n_up, r, world)
        if blocks.shape[0] != want:
            raise ValueError(f"rank {r}: {blocks.shape[0]} tiles, expected {want}")
        for i in range(want):
            ti, tj = coords[r + i * world]
            blk = blocks[i]
            full[ti * TILE:(ti + 1) * TILE, tj * TILE:(tj + 1) * TILE] = blk
            if ti != tj:
                full[tj * TILE:(tj + 1) * TILE, ti * TILE:(ti + 1) * TILE] = blk.transpose(1, 0, 2)
    return full[:n_genomes, :n_genomes]


def gather_ibs(n_genomes: int, my_blocks: np.ndarray, group=None) -> np.ndarray | None:
    """Collects every rank's tile blocks on rank 0 (torch.distributed gather of equal-sized, zero-padded buffers) and
    returns the assembled matrix there; other ranks return None. Works with gloo (CPU tensors) and NCCL."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    n_up = n_upper_tiles(n_genomes)
    cap = tiles_of_rank(n_up, 0, world)
    buf = torch.zeros((cap, TILE, TILE, 4), dtype=torch.int32)
    buf[: my_blocks.shape[0]] = torch.from_numpy(my_blocks.view(np.int32))
    backend = dist.get_backend(group)
    if backend == "nccl":
        buf = buf.cuda()
    out = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(out, buf, group=group)
    if rank != 0:
        return None
    blocks = [o.cpu().numpy().view(np.uint32)[: tiles_of_rank(n_up, r, world)] for r, o in enumerate(out)]
    return assemble_ibs(n_genomes, blocks)


# ------------------------------------------------------------------------------------------------ KING pairs ---------
def gather_king_pairs(my_pairs: np.ndarray, group=None) -> np.ndarray:
    """Every rank's KING pair list (capi.KING_PAIR_DTYPE records, any length) joined and sorted by (a, b), returned on every
    rank (torch.distributed all_gather of the lengths, then of the zero-padded records). Works with gloo (CPU tensors) and NCCL."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    recs = np.ascontiguousarray(my_pairs)
    rec_bytes = recs.dtype.itemsize
    n = torch.tensor([recs.shape[0]], dtype=torch.int64, device=dev)
    counts = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(counts, n, group=group)
    counts = [int(c.item()) for c in counts]
    cap = max(max(counts), 1)
    buf = torch.zeros(cap * rec_bytes, dtype=torch.uint8)
    buf[: recs.nbytes] = torch.from_numpy(recs.view(np.uint8).reshape(-1))
    buf = buf.to(dev)
    out = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(out, buf, group=group)
    parts = [o.cpu().numpy()[: c * rec_bytes].view(recs.dtype) for o, c in zip(out, counts)]
    joined = np.concatenate(parts)
    return joined[np.lexsort((joined["b"], joined["a"]))]
