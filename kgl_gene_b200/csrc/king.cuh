// king.cuh -- KING-robust kinship (Manichaikul et al., Bioinformatics 2010; PLINK 2 --make-king) from the pairwise IBS counts.
//
// Over the loci where neither genome is coded 3:
//     kinship = 0.5 - (4 IBS0 + IBS1) / (4 min(het_a, het_b))            NaN when min(het_a, het_b) == 0
// IBS0 / IBS1 / valid come from the IBS tile accumulators (ibs_compute_tiles, any form). The rest from two Gram matrices over the
// 256 x 256 blocks under the tiles (ibs_gram.cuh):
//     HH = H H^T                     het/het loci (code 3 is 0 in the het indicator, so exact in every missing-cell mode)
//     M  = H C^T                     M[a][b] = loci where a is heterozygous and b is coded 3 (C = code-3 indicator)
//     het_a = h_a - M[a][b],   het_b = IBS1 + 2 HH - het_a               (h_a = all heterozygous loci of a, k_ibs_class_counts)
// Without code-3 cells M = 0 and het_a = h_a, het_b = h_b. For a tile below the diagonal the block list holds the mirror block,
// where the stored value is M[b][a]: there it gives het_b and the identity gives het_a.
// Numerator and denominator are exact integers; the result is one IEEE division and one subtraction in double, so it is
// bit-equal to any restatement that does the same two operations.
#pragma once
#include "ibs_gram.cuh"
#include "../../include/kgl_b200.h"

namespace kgl {

static_assert(sizeof(kgl_b200_king_pair) == 40 && offsetof(kgl_b200_king_pair, het_b) == 28 && offsetof(kgl_b200_king_pair, kinship) == 32,
              "kgl_b200_king_pair: the 40-byte layout of include/kgl_b200.h");

constexpr uint32_t kGramTableCode3 = 0x01000000u;   // operand byte of code c = byte c: 1 for code 3 (k_codes16 keeps code 3)

struct KingTiles {
  const uint32_t* acc;          // [n_tiles][3][64*64] of ibs_compute_tiles
  const uint2* tiles;
  uint32_t n_tiles;
  int valid_mode;               // the IBS missing-cell mode (k_ibs_finalize's valid_mode)
  const uint64_t* seg;          // dropped-cell segments (valid_mode 2)
  uint32_t n_loci;
  uint64_t n_genomes;
  const int32_t* hh;            // HH blocks (GramParams::compact)
  const int32_t* m;             // M blocks; null when the population has no code-3 cell
  const uint32_t* tile_block;   // per tile: block index | 1u << 31 when mirrored
  const int32_t* counts;        // {heterozygous, hom-alt} cells per genome
};

__device__ __forceinline__ double king_kinship(uint32_t ibs0, uint32_t ibs1, uint32_t het_a, uint32_t het_b) {
  const uint32_t h = min(het_a, het_b);
  if (h == 0) return __longlong_as_double(0x7FF8000000000000ll);
  return 0.5 - (double)(4ull * ibs0 + ibs1) / (double)(4ull * h);
}

// The record of cell `cell` of tile `tile` (a live pair: both genomes < n_genomes).
__device__ __forceinline__ kgl_b200_king_pair king_record(const KingTiles& K, uint32_t tile, uint32_t cell) {
  const uint32_t* a3 = K.acc + (size_t)tile * 3 * kIbsTileCells + cell;
  const uint2 tc = K.tiles[tile];
  const uint64_t a = (uint64_t)tc.x * kIbsT + cell / kIbsT, b = (uint64_t)tc.y * kIbsT + cell % kIbsT;
  kgl_b200_king_pair r;
  r.a = (uint32_t)a; r.b = (uint32_t)b;
  r.ibs0 = a3[0]; r.ibs1 = a3[kIbsTileCells];
  r.n_valid = K.n_loci;                                             // the valid-count rule of k_ibs_finalize
  if (K.valid_mode == 1) r.n_valid = a3[2 * kIbsTileCells];
  else if (K.valid_mode == 2) r.n_valid = K.n_loci - (uint32_t)(K.seg[a + 1] - K.seg[a]) - (uint32_t)(K.seg[b + 1] - K.seg[b]) + a3[2 * kIbsTileCells];
  const uint32_t tb = K.tile_block[tile];
  const bool mirrored = (tb >> 31) != 0u;
  const uint32_t ra = (uint32_t)(a % kGramM), rb = (uint32_t)(b % kGramN);
  const size_t at = (size_t)(tb & 0x7FFFFFFFu) * kGramM * kGramN + (mirrored ? (size_t)rb * kGramN + ra : (size_t)ra * kGramN + rb);
  r.het_het = (uint32_t)K.hh[at];
  const uint32_t h_a = (uint32_t)K.counts[a * 2], h_b = (uint32_t)K.counts[b * 2];
  const uint32_t het_sum = r.ibs1 + 2u * r.het_het;                 // het_a + het_b
  if (K.m == nullptr) { r.het_a = h_a; r.het_b = h_b; }
  else if (!mirrored) { r.het_a = h_a - (uint32_t)K.m[at]; r.het_b = het_sum - r.het_a; }
  else { r.het_b = h_b - (uint32_t)K.m[at]; r.het_a = het_sum - r.het_b; }
  r.kinship = king_kinship(r.ibs0, r.ibs1, r.het_a, r.het_b);
  return r;
}

// Dense writer: out[(a - row_begin)][n_genomes] for a in [row_begin, row_end); with `mirror` also the transposed cell (the
// kinship is symmetric). The layout of k_ibs_finalize mode 1.
__global__ void __launch_bounds__(256)
k_king_dense(const KingTiles K, uint64_t row_begin, uint64_t row_end, int mirror, double* __restrict__ out) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (uint64_t)K.n_tiles * kIbsTileCells) return;
  const uint32_t tile = (uint32_t)(idx / kIbsTileCells), cell = (uint32_t)(idx % kIbsTileCells);
  const uint2 tc = K.tiles[tile];
  const uint64_t a = (uint64_t)tc.x * kIbsT + cell / kIbsT, b = (uint64_t)tc.y * kIbsT + cell % kIbsT;
  if (a >= K.n_genomes || b >= K.n_genomes) return;
  const double k = king_record(K, tile, cell).kinship;
  if (a >= row_begin && a < row_end) out[(a - row_begin) * K.n_genomes + b] = k;
  if (mirror && tc.x != tc.y && b >= row_begin && b < row_end) out[(b - row_begin) * K.n_genomes + a] = k;
}

// Pair compactor: every pair a < b of the tiles with kinship >= min_kinship (NaN never qualifies) is appended at a position
// taken with one atomic per warp. The cursor keeps counting past `capacity` (records beyond it are not written), so the caller
// learns the true total. keys[i] = (a << 32) | b for the sort that makes the order independent of the schedule.
__global__ void __launch_bounds__(256)
k_king_pairs(const KingTiles K, double min_kinship, uint64_t capacity, kgl_b200_king_pair* __restrict__ pairs,
             unsigned long long* __restrict__ keys, uint32_t* __restrict__ index, unsigned long long* __restrict__ cursor) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool take = false;
  kgl_b200_king_pair r{};
  if (idx < (uint64_t)K.n_tiles * kIbsTileCells) {
    const uint32_t tile = (uint32_t)(idx / kIbsTileCells), cell = (uint32_t)(idx % kIbsTileCells);
    const uint2 tc = K.tiles[tile];
    const uint64_t a = (uint64_t)tc.x * kIbsT + cell / kIbsT, b = (uint64_t)tc.y * kIbsT + cell % kIbsT;
    if (a < b && b < K.n_genomes) {
      r = king_record(K, tile, cell);
      take = r.kinship >= min_kinship;
    }
  }
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t mask = __ballot_sync(0xFFFFFFFFu, take);
  if (mask == 0u) return;
  unsigned long long base = 0;
  if (lane == (uint32_t)(__ffs(mask) - 1)) base = atomicAdd(cursor, (unsigned long long)__popc(mask));
  base = __shfl_sync(0xFFFFFFFFu, base, __ffs(mask) - 1);
  if (!take) return;
  const uint64_t pos = base + (uint64_t)__popc(mask & ((1u << lane) - 1u));
  if (pos >= capacity) return;
  pairs[pos] = r;
  keys[pos] = ((unsigned long long)r.a << 32) | r.b;
  index[pos] = (uint32_t)pos;
}

// sorted[i] = pairs[order[i]] (the KING and LD pair lists)
template <class Pair>
__global__ void __launch_bounds__(256)
k_gather_pairs(const Pair* __restrict__ pairs, const uint32_t* __restrict__ order, uint64_t n, Pair* __restrict__ sorted) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) sorted[i] = pairs[order[i]];
}

}  // namespace kgl
