// ibs_launch.cuh -- host-side plan and launch of k_ibs_tiles.
#pragma once
#include <algorithm>

#include "ibs_tile.cuh"

namespace kgl {

constexpr uint64_t kIbsMaxTilesPerLaunch = 8192;     // 384 MB of accumulators

struct IbsPlan {
  uint32_t words_per_chunk, n_chunks, grid;
};

// 32-locus words of a genome block row that k_ibs_tiles reads: rounded up to an even count (it takes two words per step; the
// padding loci are coded 3).
inline uint32_t ibs_words_used(uint64_t n_loci) { return (uint32_t)(((n_loci + 31) / 32 + 1) / 2 * 2); }

// Segments (gridDim.y of k_ibs_missing_fix) every genome's dropped rows are cut into, so that the repair fills the GPU also
// when few tiles are dealt to it (multi-GPU): about eight 128-thread CTAs per SM, no segment shorter than ~256 rows on average,
// at most 64. With more than one segment the repair adds J atomically, into a plane the caller cleared.
inline uint32_t ibs_repair_segments(uint64_t n_dropped, uint64_t n_genomes, uint32_t n_tiles, int sm_count) {
  const uint64_t avg_rows = n_dropped / std::max<uint64_t>(1, n_genomes);
  uint32_t segs = (uint32_t)std::max<uint64_t>(1, ((uint64_t)sm_count * 8 + n_tiles - 1) / n_tiles);
  segs = (uint32_t)std::min<uint64_t>(segs, std::max<uint64_t>(1, avg_rows / 256));
  return std::min<uint32_t>(segs, 64);
}

// Units = tiles x word chunks, dealt round-robin to one persistent CTA per SM. The chunk count is chosen so that every CTA
// gets (nearly) the same number of units while a unit stays long enough (>= 256 words) to amortise its 48 adds per thread.
inline IbsPlan plan_ibs(uint32_t n_tiles, uint32_t words_used, int sm_count, uint32_t chunk_words_hint = 0) {
  IbsPlan p{};
  const uint32_t stages = (words_used + kIbsKW - 1) / kIbsKW;          // 16-word steps
  uint32_t best_chunks = 1;
  if (chunk_words_hint) {
    const uint32_t wpc = (chunk_words_hint + kIbsKW - 1) / kIbsKW * kIbsKW;
    best_chunks = (words_used + wpc - 1) / wpc;
  } else {
    const uint32_t max_chunks = stages >= 16 ? stages / 16 : 1;       // >= 256 words per chunk
    double best = -1.0;
    const uint32_t lo = 1, hi = max_chunks < 4096 ? max_chunks : 4096;
    for (uint32_t c = lo; c <= hi; ++c) {
      const uint32_t sp = (stages + c - 1) / c;                         // stages per chunk
      const uint32_t nc = (stages + sp - 1) / sp;
      const uint64_t units = (uint64_t)n_tiles * nc;
      const uint64_t grid = units < (uint64_t)sm_count ? units : (uint64_t)sm_count;
      const uint64_t rounds = (units + grid - 1) / grid;
      // time ~ rounds * stages per chunk (+ a fixed cost per unit of about 3 stage-times for the epilogue and pipeline refill)
      const double t = (double)rounds * ((double)sp + 3.0);
      const double eff = (double)n_tiles * stages / ((double)sm_count * t);
      if (eff > best + 1e-9) { best = eff; best_chunks = nc; }
    }
  }
  const uint32_t sp = (stages + best_chunks - 1) / best_chunks;
  p.words_per_chunk = sp * kIbsKW;
  p.n_chunks = (stages + sp - 1) / sp;
  const uint64_t units = (uint64_t)n_tiles * p.n_chunks;
  p.grid = (uint32_t)(units < (uint64_t)sm_count ? units : (uint64_t)sm_count);
  if (p.grid == 0) p.grid = 1;
  return p;
}

template <bool MISSING, int TJ>
inline cudaError_t launch_ibs_t(const IbsParams& P, const IbsPlan& pl, cudaStream_t stream) {
  const size_t smem = ibs_smem_bytes(MISSING);
  cudaError_t e = cudaFuncSetAttribute(k_ibs_tiles<MISSING, TJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  k_ibs_tiles<MISSING, TJ><<<pl.grid, kIbsTileCells / (4 * TJ), smem, stream>>>(P);
  return cudaGetLastError();
}

inline cudaError_t launch_ibs(const IbsParams& P, const IbsPlan& pl, bool missing, cudaStream_t stream, int tj = 2) {
  if (tj == 4) return missing ? launch_ibs_t<true, 4>(P, pl, stream) : launch_ibs_t<false, 4>(P, pl, stream);
  return missing ? launch_ibs_t<true, 2>(P, pl, stream) : launch_ibs_t<false, 2>(P, pl, stream);
}

}  // namespace kgl
