// hwe.cuh -- Hardy-Weinberg equilibrium per (locus, group) from the per-group counts of k_group_counts (fst.cuh): the exact test
// of Wigginton, Cutler & Abecasis 2005 (kgl_b200_run_hardy), its mid-p, the per-locus F = 1 - H_obs / H_exp, and the variant QC
// mask built from the test, the call rate and the minor allele frequency (kgl_b200_run_variant_qc). The contract -- the recurrence,
// the summation order, the tie margin -- is stated in include/kgl_b200.h; tests/hwe_oracle.py restates it term by term.
//
// The walk. One thread takes one (locus, group) cell. It walks from the mode m down to P(obs) (or up), then sums the support from
// the mode: S over every term, N over the terms with P(h) <= P(obs) (1 + 2^-40), the terms below the mode first (m-2, m-4, ..),
// then those above. A side stops early, with the same bits, once its exact ratio to the next term is below 1 (the distribution is
// log-concave, so every later term on the side is smaller still) and the current term t is 0 or below 2^-54 of both S and N: a
// smaller term is under half an ulp of either accumulator, so round to nearest returns it unchanged, qualifying or not. Testing t
// against S alone would be wrong: terms that fail the tie test join S only, and the smaller ones after them do qualify for N.
//
// Load balance. A walk costs from 1 term (monomorphic) to thousands (common allele, tens of thousands of genomes), and a warp waits
// for its longest lane. k_hwe_keys keys every cell by the bit length of its rare-allele count n_r (the walk's width grows with
// sqrt(n_r)), longest first; one radix pass over those 5 bits (cub, stable) orders the cells, and k_hwe scatters p and F back.
#pragma once
#include "common.cuh"

#include <cstdint>

namespace kgl {

constexpr uint32_t kHweThreads = 128;
constexpr int kHweKeyShift = 40;                     // sort key = (31 - bit length of n_r) << 40 | cell
constexpr uint64_t kHweCellMask = (1ull << kHweKeyShift) - 1;
constexpr uint32_t kHweMaxGenomes = 1u << 25;        // every integer of the recurrence is exact in double below this group size

// The margin that makes rounding-level near-ties count as ties: a term qualifies for N when P(h) <= P(obs) * (1 + 2^-40).
#define KGL_HWE_TIE_FACTOR (1.0 + 0x1p-40)
#define KGL_HWE_ABSORB 0x1p-54

__device__ __forceinline__ double hwe_nan() { return __longlong_as_double(0x7FF8000000000000ll); }

// rows[n_rows] -> flag[row] = 1 (the multi-allelic rows; flag cleared by the caller).
__global__ void k_hwe_mark_rows(const uint32_t* __restrict__ rows, uint64_t n_rows, uint8_t* __restrict__ flag) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_rows) flag[rows[i]] = 1;
}

// Rare-allele copies of a cell's counts (0 where the cell has no test: no valid call, or a multi-allelic row).
__device__ __forceinline__ uint64_t hwe_rare(uint4 c, bool multi) {
  const uint64_t v = (uint64_t)c.x + c.y + c.z;
  if (multi || v == 0) return 0;
  const uint64_t a = (uint64_t)c.y + 2ull * c.z, b = (uint64_t)c.y + 2ull * c.x;
  return a < b ? a : b;
}

__global__ void __launch_bounds__(256) k_hwe_keys(const uint4* __restrict__ counts, const uint8_t* __restrict__ multi, uint64_t n_cells,
                                                  uint32_t n_groups, unsigned long long* __restrict__ keys) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_cells) return;
  const uint64_t nr = hwe_rare(__ldg(counts + i), multi && multi[i / n_groups]);
  const uint32_t len = nr ? 64 - __clzll((long long)nr) : 0;
  keys[i] = (unsigned long long)(31 - len) << kHweKeyShift | i;
}

struct HweParams {
  const uint4* counts;                  // [n_loci][n_groups] = {n0, n1, n2, n3}
  const unsigned long long* order;      // [n_cells] sort keys (low 40 bits: the cell)
  const uint8_t* multi;                 // [n_loci] 1 = multi-allelic row, or null
  uint64_t n_cells;
  uint32_t n_groups, midp;
  double* p;                            // [n_cells]
  double* f;                            // [n_cells] or null
  unsigned long long* terms;            // terms walked, all cells (instrumentation)
};

// The exact test of one cell; `walked` receives the terms computed.
__device__ __forceinline__ double hwe_exact(uint64_t n1, uint64_t nr, uint64_t nc, uint64_t v, uint32_t midp, uint32_t& walked) {
  if (nr == 0) return 1.0;
  uint64_t m = nr * nc / (2 * v);
  if ((m ^ nr) & 1) ++m;
  // P(obs): from the mode towards the observed heterozygote count. A term that underflows to 0 stays 0.
  double pobs = 1.0;
  if (n1 < m) {
    for (uint64_t h = m; h > n1 && pobs != 0.0; h -= 2) {
      const uint64_t r = (nr - h) / 2, c = (nc - h) / 2;
      pobs = __ddiv_rn(__dmul_rn(pobs, (double)(h * (h - 1))), (double)(4 * (r + 1) * (c + 1)));
      ++walked;
    }
  } else {
    for (uint64_t h = m; h < n1 && pobs != 0.0; h += 2) {
      const uint64_t r = (nr - h) / 2, c = (nc - h) / 2;
      pobs = __ddiv_rn(__dmul_rn(pobs, (double)(4 * r * c)), (double)((h + 2) * (h + 1)));
      ++walked;
    }
  }
  if (pobs == 0.0) return 0.0;                        // N = 0: no term is <= 0 (the floor of the test)
  const double thr = __dmul_rn(pobs, KGL_HWE_TIE_FACTOR);
  double S = 1.0, N = 1.0 <= thr ? 1.0 : 0.0;
  double t = 1.0;
  for (uint64_t h = m; h >= 2; h -= 2) {              // below the mode
    const uint64_t r = (nr - h) / 2, c = (nc - h) / 2;
    const uint64_t a = h * (h - 1), b = 4 * (r + 1) * (c + 1);
    if (a < b && __dmul_rn(S, KGL_HWE_ABSORB) > t && __dmul_rn(N, KGL_HWE_ABSORB) > t) break;
    t = __ddiv_rn(__dmul_rn(t, (double)a), (double)b);
    ++walked;
    S = __dadd_rn(S, t);
    if (t <= thr) N = __dadd_rn(N, t);
    if (t == 0.0) break;
  }
  t = 1.0;
  for (uint64_t h = m; h + 2 <= nr; h += 2) {         // above the mode
    const uint64_t r = (nr - h) / 2, c = (nc - h) / 2;
    const uint64_t a = 4 * r * c, b = (h + 2) * (h + 1);
    if (a < b && __dmul_rn(S, KGL_HWE_ABSORB) > t && __dmul_rn(N, KGL_HWE_ABSORB) > t) break;
    t = __ddiv_rn(__dmul_rn(t, (double)a), (double)b);
    ++walked;
    S = __dadd_rn(S, t);
    if (t <= thr) N = __dadd_rn(N, t);
    if (t == 0.0) break;
  }
  return midp ? __ddiv_rn(__dsub_rn(N, __dmul_rn(0.5, pobs)), S) : __ddiv_rn(N, S);
}

__global__ void __launch_bounds__(kHweThreads) k_hwe(HweParams P) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t walked = 0;
  if (i < P.n_cells) {
    const uint64_t cell = __ldg(P.order + i) & kHweCellMask;
    const uint4 cn = __ldg(P.counts + cell);
    const bool multi = P.multi && P.multi[cell / P.n_groups];
    const uint64_t v = (uint64_t)cn.x + cn.y + cn.z;
    double p = hwe_nan(), f = hwe_nan();
    if (!multi && v > 0) {
      const uint64_t s = (uint64_t)cn.y + 2ull * cn.z, nr = hwe_rare(cn, false);
      p = hwe_exact(cn.y, nr, 2 * v - nr, v, P.midp, walked);
      if (s != 0 && s != 2 * v) f = __dsub_rn(1.0, __ddiv_rn((double)(2 * v * cn.y), (double)(s * (2 * v - s))));
    }
    P.p[cell] = p;
    if (P.f) P.f[cell] = f;
  }
  unsigned long long w = walked;
  for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xFFFFFFFFu, w, o);
  if ((threadIdx.x & 31) == 0 && w) atomicAdd(P.terms, w);
}

struct QcParams {
  const uint32_t* pooled;               // [n_loci][4] raw counts over all genomes
  const double* p;                      // [n_loci][n_groups] or null (no HWE filter)
  const uint8_t* keep;                  // [n_loci] or null
  const uint8_t* multi;                 // [n_loci] or null
  uint64_t n_loci, n_genomes;
  uint32_t n_groups;
  double min_call_rate, min_maf, min_hwe_p;
  uint8_t* keep_out;
  unsigned long long* n_kept;
};

// One thread per locus: the QC rule of include/kgl_b200.h, and the number kept.
__global__ void __launch_bounds__(256) k_variant_qc(QcParams P) {
  const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool k = false;
  if (l < P.n_loci) {
    k = (!P.keep || P.keep[l]) && !(P.multi && P.multi[l]);
    const uint32_t n0 = P.pooled[4 * l], n1 = P.pooled[4 * l + 1], n2 = P.pooled[4 * l + 2], n3 = P.pooled[4 * l + 3];
    if (k && P.min_call_rate != 0.0) k = __ddiv_rn((double)(P.n_genomes - n3), (double)P.n_genomes) >= P.min_call_rate;
    if (k && P.min_maf != 0.0) {
      const uint64_t v2 = 2 * ((uint64_t)n0 + n1 + n2), s = (uint64_t)n1 + 2ull * n2;
      k = v2 != 0 && __ddiv_rn((double)(s < v2 - s ? s : v2 - s), (double)v2) >= P.min_maf;
    }
    if (k && P.p)
      for (uint32_t g = 0; g < P.n_groups; ++g)
        if (P.p[l * P.n_groups + g] < P.min_hwe_p) { k = false; break; }      // NaN (a group without calls) never drops
    P.keep_out[l] = k ? 1 : 0;
  }
  const uint32_t mask = __ballot_sync(0xFFFFFFFFu, k);
  if ((threadIdx.x & 31) == 0 && mask) atomicAdd(P.n_kept, (unsigned long long)__popc(mask));
}

}  // namespace kgl
