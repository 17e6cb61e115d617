// tail_kernels.cuh -- everything that follows the streaming kernel of a pass, in ONE launch without atomics or tickets.
//
// Round 1 ended a pass with k_post (three block roles: counter expansion, indexed code-3 cells, rare-major rows) and
// k_moment_partials: 39 + 7 us behind a 114 us streaming kernel on the chr22 shape. Now
//   * the streaming kernel expands its own bit-sliced counters (stream_common.cuh: vc_flush_counts) and leaves plain
//     per-CTA counts [cta][plane][genome],
//   * rare-major rows depend on the selection only and run behind k_locus_prepare on the preparation stream,
//   * the side list of code-3 cells carries the cell's own frequency float (k_dropped_cells), so a pass reads 8 sequential
//     bytes per cell instead of gathering one 32-byte sector of the frequency table per cell,
// and k_tail does the rest per genome: sums the CTA counts, walks the genome's code-3 cells (two warps per genome, fixed
// summation order), and assembles the partial sums / the Simple closed form (generateFrequencies' statistics block,
// kga_analysis_inbreed_freq.cpp:549-579; processSimple, kga_analysis_inbreed_calc.cpp:333-359). Launched with programmatic
// stream serialisation: its blocks are scheduled while the streaming kernel drains and do the code-3 walk, which does not depend
// on that kernel, before they wait for it (griddepcontrol.wait).
#pragma once
#include "misc_kernels.cuh"
#include "sparse_events.cuh"
#include "stream_common.cuh"

namespace kgl {

struct TailParams {
  const uint32_t* cta_counts; uint32_t n_ctas; uint64_t n_genomes_padded;      // [n_ctas][2][n_genomes_padded]
  // side list of code-3 cells, genome-major and row-sorted: {row, frequency float of the genome's population}; seg[g] = first
  // cell of genome g ([n_genomes_padded + 1]); null: the population has no code-3 cell
  const uint2* cells; const uint64_t* seg;
  uint32_t row_lo, row_hi;                 // rows outside [row_lo, row_hi) cannot be selected (the window of kgl_b200_select_loci)
  uint64_t n_genomes;
  const uint16_t* flags16;                 // null: raw mode (every row counts, no frequency corrections)
  const uint32_t* unselected_blocks;       // non-null and 0: every row is selected and valid for every population (skip the flag gather)
  const uint8_t* superpop;
  int want_moments;                        // 1: partial sums (+ Simple closed form when results != null); 0: counts only
  int unphased;
  const uint32_t* nz_rare; const unsigned long long* ecorr_rare_fx; double fx_inv;   // k_locus_prepare (null with want_moments == 0)
  DenseTotals totals; double* partials; kgl_b200_locus_results* results;
  uint32_t* gcounts; uint32_t* n3;         // counts-only consumers (raw / AF-bin passes): [g]{lo, hi}, [g]
};

constexpr int kTailGenomesPerBlock = 4;    // 64 threads (two warps) per genome: N / 4 blocks fit the machine in one wave

__global__ void __launch_bounds__(256)
k_tail(const TailParams P) {
  constexpr int GPB = kTailGenomesPerBlock, TPG = 256 / GPB, WPG = TPG / 32;
  __shared__ double s_sum[GPB][WPG][2];
  __shared__ uint32_t s_n[GPB][WPG];
  __shared__ uint32_t s_cnt[8][GPB * 2];
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, gi = tid / TPG, wi = (tid % TPG) >> 5, tl = tid % TPG;
  const uint64_t g0 = (uint64_t)blockIdx.x * GPB, g = g0 + gi;
  const bool raw = P.flags16 == nullptr;

  // ---- code-3 cells of the genome (independent of the streaming kernel) ----
  uint32_t n = 0;
  double sa = 0.0, sm = 0.0;
  if (g < P.n_genomes && P.cells != nullptr) {
    uint64_t i0 = P.seg[g], i1 = P.seg[g + 1];
    if (raw) {
      n = (tl == 0) ? (uint32_t)(i1 - i0) : 0u;
    } else {
      // a genome with many cells and a proper window: two binary searches on the rows find its cells inside the window (for a
      // short list the ~2 log2(n) dependent loads cost more than walking it -- cells outside the window fail the flag test)
      if ((P.row_lo != 0 || P.row_hi != 0xFFFFFFFFu) && i1 - i0 > 4096) {
        uint64_t lo = i0, hi = i1;
        while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (P.cells[mid].x < P.row_lo) lo = mid + 1; else hi = mid; }
        const uint64_t b = lo;
        hi = i1;
        while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (P.cells[mid].x < P.row_hi) lo = mid + 1; else hi = mid; }
        i0 = b; i1 = lo;
      }
      const int k = P.superpop[g];
      const bool all_sel = P.unselected_blocks != nullptr && __ldcg(P.unselected_blocks) == 0;
      // four cells per thread and trip: the loads of a trip are independent and overlap
      for (uint64_t i = i0 + tl; i < i1; i += 4 * TPG) {
        uint2 c[4];
        uint32_t fl[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) c[j] = (i + TPG * j < i1) ? __ldg(P.cells + i + TPG * j) : make_uint2(0xFFFFFFFFu, 0u);
#pragma unroll
        for (int j = 0; j < 4; ++j) fl[j] = (c[j].x == 0xFFFFFFFFu) ? 0u : (all_sel ? 0xFFu : (uint32_t)P.flags16[c[j].x]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if ((fl[j] >> k) & 1u) {
            ++n;
            if (P.want_moments) {
              double a, h, m;
              class_freqs(locus_freq(__uint_as_float(c[j].y)).p, a, h, m);
              sa += a; sm += m;
            }
          }
        }
      }
    }
  }
  n = __reduce_add_sync(kFull, n);
  sa = warp_sum(sa); sm = warp_sum(sm);
  if (lane == 0) { s_n[gi][wi] = n; s_sum[gi][wi][0] = sa; s_sum[gi][wi][1] = sm; }

  // ---- everything below reads what the streaming kernel (and, on the preparation stream, k_locus_prepare) wrote ----
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // per-genome counts: thread t adds the CTAs t, t + 256, ... for the block's four genomes and both planes (16-byte loads)
  uint32_t c8[GPB * 2];
#pragma unroll
  for (int j = 0; j < GPB * 2; ++j) c8[j] = 0;
  if (g0 + GPB <= P.n_genomes_padded) {
    for (uint32_t c = tid; c < P.n_ctas; c += 256) {
      const uint4 a = __ldcg(reinterpret_cast<const uint4*>(P.cta_counts + ((size_t)c * 2 + 0) * P.n_genomes_padded + g0));
      const uint4 b = __ldcg(reinterpret_cast<const uint4*>(P.cta_counts + ((size_t)c * 2 + 1) * P.n_genomes_padded + g0));
      c8[0] += a.x; c8[1] += a.y; c8[2] += a.z; c8[3] += a.w;
      c8[4] += b.x; c8[5] += b.y; c8[6] += b.z; c8[7] += b.w;
    }
  }
#pragma unroll
  for (int j = 0; j < GPB * 2; ++j) {
    const uint32_t v = __reduce_add_sync(kFull, c8[j]);
    if (lane == 0) s_cnt[warp][j] = v;
  }
  __syncthreads();
  if (tl != 0 || g >= P.n_genomes) return;
  uint32_t n_lo = 0, n_hi = 0, n3 = 0;
  double ta = 0.0, tm = 0.0;
#pragma unroll
  for (int w = 0; w < 8; ++w) { n_lo += s_cnt[w][gi]; n_hi += s_cnt[w][GPB + gi]; }
#pragma unroll
  for (int w = 0; w < WPG; ++w) { n3 += s_n[gi][w]; ta += s_sum[gi][w][0]; tm += s_sum[gi][w][1]; }   // fixed order
  if (!P.want_moments) {
    P.gcounts[g * 2 + 0] = n_lo; P.gcounts[g * 2 + 1] = n_hi; P.n3[g] = n3;
    return;
  }
  const double da = ta + (double)(long long)__ldcg(&P.ecorr_rare_fx[g * 2 + 0]) * P.fx_inv;
  const double dm = tm + (double)(long long)__ldcg(&P.ecorr_rare_fx[g * 2 + 1]) * P.fx_inv;
  moment_partials_from(g, (double)n_lo, (double)n_hi, (double)n3, (double)__ldcg(&P.nz_rare[g]), da, dm, P.totals, P.superpop[g],
                       P.unphased, P.partials, P.results);
}

}  // namespace kgl
