// ibs_gram.cuh -- pairwise IBS through three exact int8 Gram matrices on the tensor cores.
//
// With the indicators H ("heterozygous") and A ("homozygous alternate") of the pre-masked genotypes (code 3 counted as hom-ref,
// as the dense pass of the popcount path does; k_ibs_missing_fix repairs both the same way) and the dosage g = H + 2 A:
//     HH = H H^T,  AA = A A^T,  S = g g^T = HH + 2 (H A^T + A H^T) + 4 AA   =>   X = H A^T + A H^T = (S - HH - 4 AA) / 2
//     IBS1[a][b] = #(exactly one of the two is heterozygous)      = h_a + h_b - 2 HH[a][b]
//     IBS0[a][b] = #(one hom-ref, the other hom-alt)              = a_a + a_b - X[a][b] - 2 AA[a][b]
// h_a, a_a = the genome's heterozygous / hom-alt cells (k_ibs_class_counts, once per upload).
// Three runs of k_gram_i8 (gram_i8.cuh) with the expansion tables below instead of 5 LOP3 + 1 POPC per pair-word: 1.5 N^2 L MACs at
// ~3 PetaOP/s against the INT pipe's 1.2e14 pair-loci/s. Exact in int32 for n_loci < 2^29. The matrices exist only as the 256 x 256
// blocks under the tiles of a call (GramParams::compact), so the width of the population does not matter.
#pragma once
#include "gram_i8.cuh"
#include "ibs_tile.cuh"

namespace kgl {

constexpr uint32_t kGramTableDosage = 0x00020100u, kGramTableHet = 0x00000100u, kGramTableHomAlt = 0x00010000u;
constexpr uint32_t kIbsTilesPerBlock = kGramM / kIbsT;            // 64-genome tiles per side of a 256 x 256 Gram block

// counts[g] = {heterozygous cells, hom-alt cells} of genome g on the sample-major planes (code 3 in neither). Block = (genome
// block, chunk of words); lane = genome.
__global__ void __launch_bounds__(256)
k_ibs_class_counts(const uint32_t* __restrict__ lo, const uint32_t* __restrict__ hi, uint64_t n_words, uint32_t words_per_chunk,
                   int32_t* __restrict__ counts /* [n_gblocks * 32][2], zeroed */) {
  __shared__ int32_t s_sum[8][32][2];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t gb = blockIdx.x, w0 = (uint64_t)blockIdx.y * words_per_chunk, w1 = min(n_words, w0 + words_per_chunk);
  int32_t h = 0, a = 0;
  for (uint64_t w = w0 + warp; w < w1; w += 8) {
    const uint64_t o = (gb * n_words + w) * 32 + lane;
    const uint32_t x = lo[o], y = hi[o];
    h += __popc(x & ~y); a += __popc(y & ~x);
  }
  s_sum[warp][lane][0] = h; s_sum[warp][lane][1] = a;
  __syncthreads();
  if (warp == 0) {
    for (int k = 1; k < 8; ++k) { h += s_sum[k][lane][0]; a += s_sum[k][lane][1]; }
    atomicAdd(counts + (gb * 32 + lane) * 2, h);
    atomicAdd(counts + (gb * 32 + lane) * 2 + 1, a);
  }
}

// acc[tile][0] = IBS0, acc[tile][1] = IBS1 (the layout k_ibs_tiles leaves) of 64 x 64 tiles from the three matrices, stored block by
// block (256 x 256, GramParams::compact). tile_block[t] = index of the block that holds tile t | 1u << 31 when the tile lies below
// the diagonal (the block list holds its mirror image: rows and columns swap).
__global__ void __launch_bounds__(256)
k_ibs_from_grams(const int32_t* __restrict__ s, const int32_t* __restrict__ hh, const int32_t* __restrict__ aa,
                 const int32_t* __restrict__ counts, const uint2* __restrict__ tiles, const uint32_t* __restrict__ tile_block,
                 uint32_t n_tiles, uint32_t* __restrict__ acc) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (uint64_t)n_tiles * kIbsTileCells) return;
  const uint32_t tile = (uint32_t)(idx / kIbsTileCells), cell = (uint32_t)(idx % kIbsTileCells);
  const uint2 tc = tiles[tile];
  const uint32_t tb = tile_block[tile];
  const bool mirrored = (tb >> 31) != 0u;
  const uint64_t a = (uint64_t)tc.x * kIbsT + cell / kIbsT, b = (uint64_t)tc.y * kIbsT + cell % kIbsT;
  const uint32_t ra = (uint32_t)(a % kGramM), rb = (uint32_t)(b % kGramN);          // position inside the block
  const size_t at = (size_t)(tb & 0x7FFFFFFFu) * kGramM * kGramN + (mirrored ? (size_t)rb * kGramN + ra : (size_t)ra * kGramN + rb);
  const int32_t v_hh = hh[at], v_aa = aa[at], v_s = s[at];
  const int32_t h_a = counts[a * 2], a_a = counts[a * 2 + 1], h_b = counts[b * 2], a_b = counts[b * 2 + 1];
  const int32_t x = (v_s - v_hh - 4 * v_aa) / 2;
  uint32_t* out = acc + (size_t)tile * 3 * kIbsTileCells + cell;
  out[0] = (uint32_t)(a_a + a_b - x - 2 * v_aa);
  out[kIbsTileCells] = (uint32_t)(h_a + h_b - 2 * v_hh);
}

}  // namespace kgl
