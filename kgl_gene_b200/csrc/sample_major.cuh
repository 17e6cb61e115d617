// sample_major.cuh -- K6 bit transpose and the lane-per-genome log-likelihood kernel.
//
// Derived layout ("sample-major, warp-interleaved"): genomes are grouped in blocks of 32 (one warp), loci in words of 32.
//   sm_lo / sm_hi : uint32 [n_gblocks][n_words][32]   word (gb, w, lane) = bits of genome 32*gb+lane at loci 32w..32w+31
// A warp reading word w of its 32 genomes touches one contiguous 128-byte line. Loci beyond n_loci are coded 3 (dropped)
// so they can never be counted.
#pragma once
#include "common.cuh"

namespace kgl {

// 32x32 bit-matrix transpose across a warp: lane i holds row i on entry, column i on exit.
__device__ __forceinline__ uint32_t warp_transpose32(uint32_t x, int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    // m: bit positions j with (j & s) == 0
    const uint32_t m = (s == 16) ? 0x0000FFFFu : (s == 8) ? 0x00FF00FFu : (s == 4) ? 0x0F0F0F0Fu : (s == 2) ? 0x33333333u : 0x55555555u;
    const uint32_t y = __shfl_xor_sync(kFull, x, s);
    x = (lane & s) ? ((x & ~m) | ((y & ~m) >> s)) : ((x & m) | ((y & m) << s));
  }
  return x;
}

// grid: (n_words, ceil(n_gblocks / 8)); block: 256 threads = 8 warps, warp = one genome block, lane = one locus row.
__global__ void __launch_bounds__(256)
k_to_sample_major(const uint32_t* __restrict__ packed32 /* loci-major as u32 words */, uint64_t row_words,
                  uint64_t n_loci, uint64_t n_gblocks, uint64_t n_words,
                  uint32_t* __restrict__ sm_lo, uint32_t* __restrict__ sm_hi) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t w = blockIdx.x;
  const uint64_t gb = (uint64_t)blockIdx.y * 8 + warp;
  if (gb >= n_gblocks) return;
  const uint64_t l = w * 32 + lane;
  // unit = gb/2; inside the unit the u32 words are {lo[0], lo[1], hi[0], hi[1]}
  const uint64_t word_in_row = (gb >> 1) * 4 + (gb & 1);
  uint32_t lo = 0xFFFFFFFFu, hi = 0xFFFFFFFFu;   // padding loci: code 3
  if (l < n_loci) {
    lo = packed32[l * row_words + word_in_row];
    hi = packed32[l * row_words + word_in_row + 2];
  }
  lo = warp_transpose32(lo, lane);
  hi = warp_transpose32(hi, lane);
  const uint64_t o = (gb * n_words + w) * 32 + lane;
  sm_lo[o] = lo;
  sm_hi[o] = hi;
}

// ---------------------------------------------------------------------------------------------------------------------
// Lane-per-genome term accumulation. A warp owns 32 genomes and walks the selected loci of each lane's super-population;
// per-locus allele frequencies of the current 128-locus tile sit in shared memory (one row per population).
//   NEWTON  : d/df, d2/df2 of logLikelihood over the unclamped terms, and the numbers of clamped homozygous and
//             heterozygous terms (calc.cpp:94-129; a clamped term is constant in f, so it contributes no derivative)
//   GRID    : logLikelihood at up to kGridMax shared f values                (calc.cpp:94-129)
enum { TERM_NEWTON, TERM_GRID };
constexpr int kTermWarps = 8;          // genome blocks per CTA
constexpr int kTermTileWords = 4;      // 128 loci per shared-memory tile
constexpr int kGridMax = 8;            // grid points per launch in GRID mode

struct TermParams {
  const uint32_t* sm_lo; const uint32_t* sm_hi;
  uint64_t n_gblocks, n_words, n_loci, n_genomes;
  const uint32_t* selw;        // [n_pop][n_words] selected & valid
  const float* af;             // [n_pop][n_loci]
  const uint8_t* superpop;     // [n_genomes]
  int n_pop;
  int unphased;
  uint32_t words_per_chunk;    // multiple of kTermTileWords
  const double* f;             // [n_genomes_padded] current iterate (NEWTON)
  const double* grid; int n_grid;
  double* out;                 // [n_chunks][n_genomes_padded][n_out]
  int n_out;
  uint64_t n_genomes_padded;
  // NEWTON as the exact fallback of k_terms_fast (terms_fast.cuh): only genomes with lane_state == 2 are evaluated, and
  // nothing at all when *n_slow == 0. Both null: every genome.
  const uint8_t* lane_state;
  const uint32_t* n_slow;
};

template <int MODE>
__global__ void __launch_bounds__(kTermWarps * 32)
k_genome_terms(const TermParams P) {
  __shared__ double s_p[kMaxPop][kTermTileWords * 32];     // alt-allele frequency per (population, locus of the tile)
  __shared__ uint32_t s_sel[kMaxPop][kTermTileWords];

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t gb = (uint64_t)blockIdx.x * kTermWarps + warp;
  const uint64_t g = gb * 32 + lane;
  if (P.n_slow && *P.n_slow == 0) return;
  const bool live = gb < P.n_gblocks && g < P.n_genomes && (!P.lane_state || P.lane_state[g] == 2);
  const int k = live ? P.superpop[g] : 0;
  const double f = (MODE == TERM_NEWTON) ? (live ? P.f[g] : 0.0) : 0.0;

  constexpr int NACC = (MODE == TERM_GRID) ? kGridMax : 4;
  double acc[NACC];
#pragma unroll
  for (int j = 0; j < NACC; ++j) acc[j] = 0.0;
  double gridv[kGridMax];
  if (MODE == TERM_GRID) {
#pragma unroll
    for (int j = 0; j < kGridMax; ++j) gridv[j] = (j < P.n_grid) ? P.grid[j] : 0.0;
  }

  const uint64_t w_begin = (uint64_t)blockIdx.y * P.words_per_chunk;
  const uint64_t w_end = min(w_begin + (uint64_t)P.words_per_chunk, P.n_words);

  for (uint64_t wt = w_begin; wt < w_end; wt += kTermTileWords) {
    __syncthreads();
    for (int i = threadIdx.x; i < kMaxPop * kTermTileWords * 32; i += kTermWarps * 32) {
      const int kk = i / (kTermTileWords * 32), j = i % (kTermTileWords * 32);
      const uint64_t l = wt * 32 + j;
      double p = 0.0;
      if (kk < P.n_pop && l < P.n_loci) p = locus_freq(P.af[(uint64_t)kk * P.n_loci + l]).p;
      s_p[kk][j] = p;
    }
    if (threadIdx.x < kMaxPop * kTermTileWords) {
      const int kk = threadIdx.x / kTermTileWords, j = threadIdx.x % kTermTileWords;
      s_sel[kk][j] = (kk < P.n_pop && wt + j < w_end) ? P.selw[(uint64_t)kk * P.n_words + wt + j] : 0u;
    }
    __syncthreads();
    if (!live) continue;

    for (int tw = 0; tw < kTermTileWords && wt + tw < w_end; ++tw) {
      const uint32_t sel = s_sel[k][tw];
      if (sel == 0) continue;
      const uint64_t o = (gb * P.n_words + wt + tw) * 32 + lane;
      const uint32_t lo = P.sm_lo[o], hi = P.sm_hi[o];
      // every classified cell (code 3 is not)
      uint32_t todo = sel & ~(lo & hi);
      while (todo) {
        const int i = __ffs(todo) - 1;
        todo &= todo - 1;
        const double p = s_p[k][tw * 32 + i];
        double q = __dsub_rn(1.0, p);
        q = q < 0.0 ? 0.0 : (q > 1.0 ? 1.0 : q);
        const int code = ((lo >> i) & 1) | (((hi >> i) & 1) << 1);
        if (code == 0 && !(q > kMinMajorFreq)) continue;     // freq.cpp:532: rare major allele -> locus dropped
        const bool hom = (code == 0) || (code == 2 && !P.unphased);
        const double a = (code == 0) ? q : p;               // first allele frequency
        const double a2 = (code == 1) ? q : p;              // second allele (het): major for code 1, p for an unphased hom-alt pair
        if (MODE == TERM_NEWTON) {
          if (hom) {
            // prob = f*a + (1-f)*a^2 = a*(a + f*(1-a)); d/df log prob = (1-a)/(a + f(1-a)) while prob is not clamped
            const double prob = __dadd_rn(__dmul_rn(f, a), __dmul_rn(__dsub_rn(1.0, f), __dmul_rn(a, a)));
            if (prob >= kSmallProb) {
              if (prob <= 1.0) {
                const double t = (1.0 - a) / (a + f * (1.0 - a));
                acc[0] += t;
                acc[1] -= t * t;
              }
            } else {
              acc[2] += 1.0;
            }
          } else {
            const double prob = 2 * (1.0 - f) * a * a2;
            if (prob >= kSmallProb && prob <= 1.0) {
              const double t = 1.0 / (1.0 - f);
              acc[0] -= t;
              acc[1] -= t * t;
            } else {
              acc[3] += 1.0;
            }
          }
        } else {  // TERM_GRID: logLikelihood, operation order of calc.cpp:100-125
#pragma unroll
          for (int j = 0; j < kGridMax; ++j) {
            const double fj = gridv[j];
            double prob;
            if (hom) {
              const double freq_sqd = __dmul_rn(a, a);
              prob = __dadd_rn(__dmul_rn(fj, a), __dmul_rn(__dsub_rn(1.0, fj), freq_sqd));
            } else {
              prob = __dmul_rn(__dmul_rn(__dmul_rn(2.0, __dsub_rn(1.0, fj)), a), a2);
            }
            prob = prob < kSmallProb ? kSmallProb : (prob > 1.0 ? 1.0 : prob);
            acc[j] += log(prob);
          }
        }
      }
    }
  }

  if (gb < P.n_gblocks) {
    double* out = P.out + ((uint64_t)blockIdx.y * P.n_genomes_padded + g) * P.n_out;
#pragma unroll
    for (int j = 0; j < NACC; ++j) if (j < P.n_out) out[j] = acc[j];
  }
}

}  // namespace kgl
