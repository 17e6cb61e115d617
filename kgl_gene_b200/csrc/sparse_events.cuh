// sparse_events.cuh -- the sparse side of the fused pass: code-3 ("dropped") cells and rare-major rows.
//
// The streaming kernel (stream_count.cuh) only counts set lo / hi bits. Two kinds of cells need more than a count, and
// both are sparse in real data:
//   * code-3 cells (first variant not in the AF list, >2 variants, missing ...; SURVEY flattener contract): they are not
//     classified, so the locus' class frequencies leave the genome's expected sums (kga_analysis_inbreed_freq.cpp:462-543)
//   * rows whose major allele is rare for a population (q <= 0.01): a hom-ref genome is dropped there (freq.cpp:532-539)
// Dropped cells are indexed ONCE per uploaded matrix (k_dropped_count / k_dropped_index + a key sort, part of the upload:
// the index is the "side list" of the flattener contract in device form, genome-major and row-sorted; k_dropped_cells adds
// the cell's own allele frequency, so that a pass reads 8 sequential bytes per cell instead of gathering a 32-byte sector
// from the frequency table); every pass then visits only the indexed cells, two warps per genome, without atomics and in a
// fixed summation order (k_tail, tail_kernels.cuh). Populations with too many code-3 cells for an index fall back to
// k_dropped_scan, which re-reads the matrix.
// Sums that ARE accumulated with atomics (rare-major rows, the scan fallback) are kept in 64-bit fixed point: integer adds
// commute, so every result is independent of the schedule (the scale leaves room for n_loci terms below 1).
#pragma once
#include "common.cuh"

namespace kgl {

typedef unsigned long long DroppedKey;     // (genome << 32) | row

// ---- index construction (upload time) ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_dropped_count(const uint4* __restrict__ packed, uint64_t n_cells128, unsigned long long* __restrict__ total) {
  uint32_t c = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cells128; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint4 v = ld_stream_u4(packed + i);
    c += __popc(v.x & v.z) + __popc(v.y & v.w);
  }
  c = __reduce_add_sync(kFull, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(total, (unsigned long long)c);
}

// Appends one key per code-3 cell of a range of units (any order; sorted afterwards). The cursor keeps counting past the
// capacity, so the caller learns the true total and can retry with an exact allocation.
__global__ void __launch_bounds__(256)
k_dropped_index(const uint4* __restrict__ packed /* first unit of the range */, uint64_t n_cells128, uint64_t cell0 /* its global unit index */,
                uint32_t units, unsigned long long* __restrict__ cursor, DroppedKey* __restrict__ cells, uint64_t capacity) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  const uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (uint64_t base = i0 - lane; base < n_cells128; base += stride) {   // whole warps iterate together
    const uint64_t i = base + lane;
    uint64_t both = 0;
    if (i < n_cells128) {
      const uint4 v = ld_stream_u4(packed + i);
      both = (uint64_t)(v.x & v.z) | ((uint64_t)(v.y & v.w) << 32);
    }
    const uint32_t n = (uint32_t)__popcll(both);
    if (__any_sync(kFull, n != 0)) {
      // warp-level exclusive scan of n, one atomic per warp
      uint32_t incl = n;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(kFull, incl, o);
        if ((int)lane >= o) incl += t;
      }
      const uint32_t warp_total = __shfl_sync(kFull, incl, 31);
      unsigned long long start = 0;
      if (lane == 0) start = atomicAdd(cursor, (unsigned long long)warp_total);
      start = __shfl_sync(kFull, start, 0);
      uint64_t o = start + (incl - n);
      const uint32_t row = (uint32_t)((cell0 + i) / units), unit = (uint32_t)((cell0 + i) % units);
      while (both) {
        const int b = __ffsll((long long)both) - 1;
        both &= both - 1;
        if (o < capacity) cells[o] = ((DroppedKey)(unit * 64 + (uint32_t)b) << 32) | row;
        ++o;
      }
    }
  }
}

// ---- per pass ---------------------------------------------------------------------------------------------------------------
// Fixed-point scale of the atomically accumulated class-frequency sums: terms lie in [0, 1], at most n_loci of them per genome.
inline double fx_scale_for(uint64_t n_loci) {
  int bits = 1;
  while (bits < 40 && (n_loci >> bits) != 0) ++bits;
  return (double)(1ull << (62 - bits));
}
__device__ __forceinline__ void fx_add(unsigned long long* acc, double v, double fx) {
  atomicAdd(acc, (unsigned long long)__double2ll_rn(v * fx));
}

// Side list entry of a code-3 cell: its row and the frequency float of the GENOME'S population at that row.
__global__ void __launch_bounds__(256)
k_dropped_cells(const DroppedKey* __restrict__ keys, uint64_t n_keys, const uint8_t* __restrict__ superpop /* nullable: rows only */,
                const float* __restrict__ af, uint64_t n_loci, uint2* __restrict__ cells) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_keys) return;
  const DroppedKey key = keys[i];
  const uint32_t row = (uint32_t)key, g = (uint32_t)(key >> 32);
  float a = 0.0f;
  if (superpop) a = af[(uint64_t)superpop[g] * n_loci + row];
  cells[i] = make_uint2(row, __float_as_uint(a));
}

// seg[g] = first key of genome g in the sorted key array (g = 0 .. n_genomes_padded inclusive).
__global__ void __launch_bounds__(256)
k_dropped_segments(const DroppedKey* __restrict__ keys, uint64_t n_keys, uint64_t n_genomes_padded, uint64_t* __restrict__ seg) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g > n_genomes_padded) return;
  const DroppedKey want = (DroppedKey)g << 32;
  uint64_t lo = 0, hi = n_keys;
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if (keys[mid] < want) lo = mid + 1; else hi = mid;
  }
  seg[g] = lo;
}

// Fallback without an index: one thread per 128-bit unit-row. n3[g] += code-3 cells in rows selected for the genome;
// ecorr_fx[g][2] += their {majHom, minHom} class frequencies (fixed point). flags16 == null: raw mode, every cell counts.
__global__ void __launch_bounds__(256)
k_dropped_scan(const uint4* __restrict__ packed, uint64_t n_cells128, uint32_t units, const uint16_t* __restrict__ flags16,
               const uint8_t* __restrict__ superpop, const float* __restrict__ af, uint64_t n_loci, uint32_t* __restrict__ n3,
               unsigned long long* __restrict__ ecorr_fx, double fx) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cells128; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint4 v = ld_stream_u4(packed + i);
    uint64_t both = (uint64_t)(v.x & v.z) | ((uint64_t)(v.y & v.w) << 32);
    if (both == 0) continue;
    const uint32_t row = (uint32_t)(i / units), unit = (uint32_t)(i % units);
    const uint32_t fl = flags16 ? flags16[row] : 0u;
    while (both) {
      const int b = __ffsll((long long)both) - 1;
      both &= both - 1;
      const uint32_t g = unit * 64 + (uint32_t)b;
      if (flags16 == nullptr) { atomicAdd(&n3[g], 1u); continue; }
      const int k = superpop[g];
      if (!((fl >> k) & 1u)) continue;
      atomicAdd(&n3[g], 1u);
      double a, h, m;
      class_freqs(locus_freq(af[(uint64_t)k * n_loci + row]).p, a, h, m);
      fx_add(&ecorr_fx[(uint64_t)g * 2 + 0], a, fx);
      fx_add(&ecorr_fx[(uint64_t)g * 2 + 1], m, fx);
    }
  }
}

}  // namespace kgl
