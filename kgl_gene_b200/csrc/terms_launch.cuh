// terms_launch.cuh -- host-side plans of the estimator sweeps: k_terms_fast (terms_fast.cuh) and k_genome_terms
// (sample_major.cuh).
#pragma once
#include <algorithm>

#include "sample_major.cuh"
#include "terms_fast.cuh"

namespace kgl {

// Dynamic shared memory of a k_terms_fast CTA: the tile's table, the per-slot accumulators of every thread, the RITLAND masks.
inline size_t fast_smem_bytes(int mode, uint32_t slots, int warps) {
  return (size_t)kMaxPop * fast_stride(mode) * 8 + (size_t)slots * warps * 32 * fast_n_acc(mode) * 8 + kMaxPop * kFastTileWords * 2 * 4;
}

struct FastPlan {
  bool ok;                         // false: no CTA shape fits the shared-memory limit (nothing may be launched)
  int warps, ctas_per_sm;
  uint32_t slots;                  // genome blocks per warp
  uint64_t gy;                     // rows of CTAs: gy * warps * slots >= gblocks
  uint64_t tile_begin, tile_end;   // 256-locus tiles swept (the selection window)
  uint64_t tiles_per_chunk, n_chunks;   // grid.x = n_chunks chunks of tiles_per_chunk tiles, the last one possibly shorter
  size_t smem;
};

// gblocks: genome blocks of the sweep (the compact blocks of the list in late Newton sweeps). sel_row_lo / sel_row_hi: rows that
// can be selected, [lo, hi); hi = ~0: unknown, every tile. smem_limit: the device's opt-in shared memory per block.
//
// Warps per CTA: of 16..24, the count that leaves the fewest genome-block slots empty (more warps on a tie), with
// min(8, ceil(gblocks / warps)) slots, among the shapes whose shared memory fits -- the unphased root search's three
// accumulators per slot overflow 227 KB at 8 slots and 22 or more warps. Only the tiles of the selection window are swept (a
// contig is usually analysed in many short windows), in chunks that give every CTA about one chunk.
inline FastPlan plan_fast(int mode, uint64_t gblocks, uint64_t n_words, uint64_t sel_row_lo, uint64_t sel_row_hi, int sm_count,
                          size_t smem_limit) {
  FastPlan p{};
  const auto slots_for = [&](int w) { return (uint32_t)std::min<uint64_t>(8, (gblocks + w - 1) / w); };
  int warps = 0; double best = -1.0;
  for (int w = 16; w <= kFastMaxWarps; ++w) {
    const uint64_t sl = slots_for(w);
    if (fast_smem_bytes(mode, (uint32_t)sl, w) > smem_limit) continue;
    const uint64_t rows = (gblocks + (uint64_t)w * sl - 1) / ((uint64_t)w * sl);
    const double filled = (double)gblocks / (double)(rows * sl * w);
    if (filled >= best) { best = filled; warps = w; }
  }
  // A handful of genome blocks (late Newton sweeps over the list of unfinished genomes, small populations) cannot fill 16
  // warps: small CTAs instead, four of them per SM, each with a quarter of the tiles -- the sweep is then bound by the
  // per-tile latency of a few warps, and four CTAs per SM overlap it.
  p.ctas_per_sm = 1;
  if (gblocks <= 8) { warps = gblocks <= 4 ? 4 : 8; p.ctas_per_sm = 4; }
  if (warps == 0) return p;
  p.warps = warps;
  p.slots = slots_for(warps);
  p.smem = fast_smem_bytes(mode, p.slots, warps);
  if (p.smem > smem_limit) return p;
  p.gy = (gblocks + (uint64_t)warps * p.slots - 1) / ((uint64_t)warps * p.slots);
  const uint64_t all_tiles = (n_words + kFastTileWords - 1) / kFastTileWords;
  p.tile_begin = std::min<uint64_t>(all_tiles, sel_row_lo / kFastTile);
  p.tile_end = std::max<uint64_t>(p.tile_begin, std::min<uint64_t>(all_tiles, sel_row_hi == ~0ull ? all_tiles : (sel_row_hi + kFastTile - 1) / kFastTile));
  const uint64_t n_tiles = std::max<uint64_t>(1, p.tile_end - p.tile_begin);
  const uint64_t want = std::max<uint64_t>(1, (uint64_t)sm_count * p.ctas_per_sm / p.gy);
  p.tiles_per_chunk = std::max<uint64_t>(1, (n_tiles + want - 1) / want);
  p.n_chunks = (n_tiles + p.tiles_per_chunk - 1) / p.tiles_per_chunk;
  p.ok = true;
  return p;
}

// k_genome_terms: ceil(n_gblocks / kTermWarps) CTAs per chunk of words, chunks of whole shared-memory tiles.
struct TermLaunch { dim3 grid; uint32_t words_per_chunk; uint64_t n_chunks; };

inline TermLaunch plan_terms(uint64_t n_gblocks, uint64_t n_words, int sm_count) {
  TermLaunch t;
  const uint64_t gx = (n_gblocks + kTermWarps - 1) / kTermWarps;
  // aim for ~4 waves of CTAs; chunks are multiples of the shared-memory tile
  uint64_t want_chunks = std::max<uint64_t>(1, ((uint64_t)sm_count * 8 + gx - 1) / gx);
  uint64_t wpc = (n_words + want_chunks - 1) / want_chunks;
  wpc = std::max<uint64_t>(kTermTileWords, (wpc + kTermTileWords - 1) / kTermTileWords * kTermTileWords);
  t.words_per_chunk = (uint32_t)wpc;
  t.n_chunks = (n_words + wpc - 1) / wpc;
  t.grid = dim3((unsigned)gx, (unsigned)t.n_chunks);
  return t;
}

}  // namespace kgl
