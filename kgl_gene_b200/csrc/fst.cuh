// fst.cuh -- population differentiation: per-group genotype counts of every locus from one streaming read of the resident
// loci-major matrix (kgl_b200_run_group_counts), and Hudson / Weir-Cockerham F_ST between pairs of groups from those counts
// (kgl_b200_run_fst). The formulas, the locus rule and the summation order are stated in include/kgl_b200.h.
//
// Counting. A group's genomes inside one 32-bit half of a 128-bit unit are a 32-bit mask m; with lo / hi the code planes of that
// half, the group's cells there hold code 1 on popc(lo & ~hi & m), code 2 on popc(~lo & hi & m) and code 3 on popc(lo & hi & m)
// (one LOP3 and one POPC each); code 0 follows from the group's size. The host lists, per chunk of kGcChunkUnits units, every
// (half, group) with a non-empty mask, ordered by group (build_group_table): one entry per group present, so a unit of genomes in
// 1000 Genomes order (groups in runs) costs a few entries and a fully interleaved one at most 2 x n_groups.
// k_group_counts takes tiles of 32 rows (one per lane). Per chunk its threads stage the tile's units in shared memory with
// coalesced 128-bit streaming loads (the discipline of the streaming pass: every byte of the matrix is read once), then each warp
// walks a contiguous eighth of the chunk's entry list for its 32 rows, keeping the running group's three counts in registers.
// Only when the group changes along the slice are they added into the tile's shared counters (lane-private addresses, so the
// adds of a warp never collide), i.e. at most once per group and warp per chunk however the groups interleave.
#pragma once
#include "common.cuh"

#include <algorithm>
#include <cstdint>
#include <vector>

namespace kgl {

constexpr uint32_t kGcRows = 32;                          // rows of a tile, one per lane
constexpr uint32_t kGcChunkUnits = 32;                    // 128-bit units staged per chunk
constexpr uint32_t kGcThreads = 256;
constexpr uint32_t kGcWarps = kGcThreads / 32;
constexpr uint32_t kGcPitch = kGcChunkUnits * 4 + 1;      // words per staged row: odd, so the 32 lanes read 32 different banks
constexpr uint32_t kGcMaxGroups = 64;
constexpr uint32_t kFstBlock = 256;                       // loci per fixed summation block (include/kgl_b200.h)

inline size_t group_counts_smem(uint32_t n_groups) { return (size_t)kGcRows * kGcPitch * 4 + (size_t)n_groups * 3 * kGcRows * 4; }

// The entry lists of one labelling: entries {mask, group | lo word << 16} per chunk, ordered by group (then word), with
// chunk_begin[c] the first entry of chunk c (n_chunks + 1 values); size[k] = genomes of group k.
struct GroupTable {
  std::vector<uint2> entries;
  std::vector<uint32_t> chunk_begin, size;
};

// label[g] in 0..n_groups-1 or 0xFF (checked by the caller); units = 128-bit units of a row that hold genomes.
inline GroupTable build_group_table(const uint8_t* label, uint64_t n_genomes, uint64_t units, uint32_t n_groups) {
  GroupTable T;
  T.size.assign(n_groups, 0);
  const uint64_t halves = units * 2;
  std::vector<uint32_t> mask(halves * n_groups, 0);            // [group][half]
  for (uint64_t g = 0; g < n_genomes; ++g) {
    if (label[g] == 0xFF) continue;
    mask[(uint64_t)label[g] * halves + (g >> 5)] |= 1u << (g & 31);
    ++T.size[label[g]];
  }
  const uint64_t n_chunks = (units + kGcChunkUnits - 1) / kGcChunkUnits;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    T.chunk_begin.push_back((uint32_t)T.entries.size());
    const uint64_t h0 = c * kGcChunkUnits * 2, h1 = std::min<uint64_t>(halves, h0 + kGcChunkUnits * 2);
    for (uint32_t k = 0; k < n_groups; ++k)
      for (uint64_t h = h0; h < h1; ++h) {
        const uint32_t m = mask[(uint64_t)k * halves + h];
        // half h of unit u: its lo plane is word 4 u' + (h & 1) of the staged row (u' = unit within the chunk), its hi plane 2 later
        const uint32_t word = (uint32_t)((h - h0) >> 1) * 4 + (uint32_t)(h & 1);
        if (m) T.entries.push_back(make_uint2(m, k | word << 16));
      }
  }
  T.chunk_begin.push_back((uint32_t)T.entries.size());
  return T;
}

struct GroupCountParams {
  const uint4* packed;            // resident matrix, row pitch `pitch` units, rows padded to a multiple of 256
  uint64_t pitch, n_loci, n_tiles;
  uint32_t units;                 // units that hold genomes
  uint32_t n_groups, n_chunks;
  const uint2* entries;
  const uint32_t* chunk_begin;
  const uint32_t* size;
  uint4* counts;                  // [n_loci][n_groups] = {n0, n1, n2, n3}
};

__global__ void __launch_bounds__(kGcThreads) k_group_counts(GroupCountParams P) {
  extern __shared__ uint32_t gc_smem[];
  uint32_t* tile = gc_smem;                                   // [kGcRows][kGcPitch]
  uint32_t* acc = gc_smem + kGcRows * kGcPitch;               // [n_groups][3][kGcRows]
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t* row = tile + lane * kGcPitch;
  for (uint64_t t = blockIdx.x; t < P.n_tiles; t += gridDim.x) {
    const uint64_t row0 = t * kGcRows;
    __syncthreads();                                          // the previous tile's counters have been written out
    for (uint32_t i = threadIdx.x; i < P.n_groups * 3 * kGcRows; i += kGcThreads) acc[i] = 0;
    for (uint32_t c = 0; c < P.n_chunks; ++c) {
      const uint32_t u0 = c * kGcChunkUnits, nu = min(kGcChunkUnits, P.units - u0);
      __syncthreads();                                        // the previous chunk's readers are done
      for (uint32_t i = threadIdx.x; i < kGcRows * kGcChunkUnits; i += kGcThreads) {
        const uint32_t r = i / kGcChunkUnits, u = i % kGcChunkUnits;
        if (u < nu) {
          const uint4 v = ld_stream_u4(P.packed + (row0 + r) * P.pitch + u0 + u);
          uint32_t* d = tile + r * kGcPitch + u * 4;
          d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        }
      }
      __syncthreads();
      const uint32_t e0 = __ldg(P.chunk_begin + c), n = __ldg(P.chunk_begin + c + 1) - e0;
      const uint32_t b = e0 + (uint32_t)((uint64_t)n * warp / kGcWarps), e = e0 + (uint32_t)((uint64_t)n * (warp + 1) / kGcWarps);
      uint32_t cur = 0xFFFFFFFFu, n1 = 0, n2 = 0, n3 = 0;
      for (uint32_t i = b; i < e; ++i) {
        const uint2 en = __ldg(P.entries + i);
        const uint32_t k = en.y & 0xFFFFu, w = en.y >> 16;
        if (k != cur) {
          if (cur != 0xFFFFFFFFu) {
            uint32_t* a = acc + cur * 3 * kGcRows + lane;
            atomicAdd(a, n1); atomicAdd(a + kGcRows, n2); atomicAdd(a + 2 * kGcRows, n3);
          }
          cur = k; n1 = n2 = n3 = 0;
        }
        const uint32_t lo = row[w], hi = row[w + 2], m = en.x;
        n1 += __popc(lo & ~hi & m);
        n2 += __popc(~lo & hi & m);
        n3 += __popc(lo & hi & m);
      }
      if (cur != 0xFFFFFFFFu) {
        uint32_t* a = acc + cur * 3 * kGcRows + lane;
        atomicAdd(a, n1); atomicAdd(a + kGcRows, n2); atomicAdd(a + 2 * kGcRows, n3);
      }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kGcRows * P.n_groups; i += kGcThreads) {
      const uint32_t r = i / P.n_groups, k = i % P.n_groups;
      const uint64_t l = row0 + r;
      if (l >= P.n_loci) continue;
      const uint32_t* a = acc + k * 3 * kGcRows + r;
      const uint32_t c1 = a[0], c2 = a[kGcRows], c3 = a[2 * kGcRows];
      P.counts[l * P.n_groups + k] = make_uint4(__ldg(P.size + k) - c1 - c2 - c3, c1, c2, c3);
    }
  }
}

// ---- F_ST -------------------------------------------------------------------------------------------------------------------
// One locus' (numerator, denominator) for groups with counts ca, cb, as the fixed sequence of IEEE round-to-nearest operations of
// include/kgl_b200.h (explicit intrinsics: no FMA contraction). False when the locus is not used for the pair.
__device__ __forceinline__ bool fst_term(uint4 ca, uint4 cb, uint32_t method, double& num, double& den) {
  const uint32_t va = ca.x + ca.y + ca.z, vb = cb.x + cb.y + cb.z;
  const uint64_t sa = (uint64_t)ca.y + 2ull * ca.z, sb = (uint64_t)cb.y + 2ull * cb.z;
  if (va == 0 || vb == 0) return false;
  if (method == 0) {                                                            // Hudson
    const double pa = __ddiv_rn((double)sa, (double)(2ull * va)), pb = __ddiv_rn((double)sb, (double)(2ull * vb));
    const double d = __dsub_rn(pa, pb);
    const double ta = __ddiv_rn(__dmul_rn(pa, __dsub_rn(1.0, pa)), (double)(2ull * va - 1));
    const double tb = __ddiv_rn(__dmul_rn(pb, __dsub_rn(1.0, pb)), (double)(2ull * vb - 1));
    num = __dsub_rn(__dsub_rn(__dmul_rn(d, d), ta), tb);
    den = __dadd_rn(__dmul_rn(pa, __dsub_rn(1.0, pb)), __dmul_rn(pb, __dsub_rn(1.0, pa)));
  } else {                                                                      // Weir & Cockerham, r = 2
    if ((uint64_t)va + vb < 3) return false;                                    // n_bar = 1
    const double na = (double)va, nb = (double)vb, nt = (double)((uint64_t)va + vb);
    const double nbar = __dmul_rn(nt, 0.5);
    const double nc = __ddiv_rn(__dmul_rn((double)((uint64_t)va * vb), 2.0), nt);
    const double pa = __ddiv_rn((double)sa, __dmul_rn(na, 2.0)), pb = __ddiv_rn((double)sb, __dmul_rn(nb, 2.0));
    const double pbar = __ddiv_rn((double)(sa + sb), __dmul_rn(nt, 2.0));
    const double da = __dsub_rn(pa, pbar), db = __dsub_rn(pb, pbar);
    const double s2 = __ddiv_rn(__dadd_rn(__dmul_rn(na, __dmul_rn(da, da)), __dmul_rn(nb, __dmul_rn(db, db))), nbar);
    const double hbar = __ddiv_rn((double)((uint64_t)ca.y + cb.y), nt);
    const double pq = __dmul_rn(pbar, __dsub_rn(1.0, pbar));
    const double nbar1 = __dsub_rn(nbar, 1.0);
    const double inner = __dsub_rn(__dsub_rn(pq, __dmul_rn(s2, 0.5)), __dmul_rn(hbar, 0.25));
    const double a = __dmul_rn(__ddiv_rn(nbar, nc), __dsub_rn(s2, __ddiv_rn(inner, nbar1)));
    const double q = __ddiv_rn(__dsub_rn(__dmul_rn(nbar, 2.0), 1.0), __dmul_rn(nbar, 4.0));
    const double bb = __dmul_rn(__ddiv_rn(nbar, nbar1), __dsub_rn(__dsub_rn(pq, __dmul_rn(s2, 0.5)), __dmul_rn(q, hbar)));
    const double cc = __dmul_rn(hbar, 0.5);
    num = a;
    den = __dadd_rn(__dadd_rn(a, bb), cc);
  }
  return den != 0.0;
}

struct FstParams {
  const uint4* counts;            // [n_loci][n_groups]
  uint64_t n_loci, n_blocks;
  uint32_t n_groups, method, n_pairs;
  const uint8_t* keep;            // [n_loci] or null
  const uint2* pairs;             // [n_pairs] = (a, b)
  double2* terms;                 // [n_pairs][n_loci] or null: (num, den), (0, 0) where not used
  double2* block_sums;            // [n_pairs][n_blocks]
  uint32_t* block_used;           // [n_pairs][n_blocks]
};

// Block (x, pair): the terms of loci [x kFstBlock, (x + 1) kFstBlock) and their sum as a fixed halving tree (0 past the last locus).
__global__ void __launch_bounds__(kFstBlock) k_fst_blocks(FstParams P) {
  __shared__ double s_num[kFstBlock], s_den[kFstBlock];
  const uint32_t p = blockIdx.y;
  const uint64_t l = (uint64_t)blockIdx.x * kFstBlock + threadIdx.x;
  double num = 0.0, den = 0.0;
  int used = 0;
  if (l < P.n_loci && (!P.keep || P.keep[l])) {
    const uint2 pr = __ldg(P.pairs + p);
    const uint4 ca = __ldg(P.counts + l * P.n_groups + pr.x), cb = __ldg(P.counts + l * P.n_groups + pr.y);
    double n_, d_;
    if (fst_term(ca, cb, P.method, n_, d_)) { num = n_; den = d_; used = 1; }
  }
  if (P.terms && l < P.n_loci) P.terms[p * P.n_loci + l] = make_double2(num, den);
  s_num[threadIdx.x] = num; s_den[threadIdx.x] = den;
  const int n_used = __syncthreads_count(used);
  for (uint32_t s = kFstBlock / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      s_num[threadIdx.x] = __dadd_rn(s_num[threadIdx.x], s_num[threadIdx.x + s]);
      s_den[threadIdx.x] = __dadd_rn(s_den[threadIdx.x], s_den[threadIdx.x + s]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    P.block_sums[(uint64_t)p * P.n_blocks + blockIdx.x] = make_double2(s_num[0], s_den[0]);
    P.block_used[(uint64_t)p * P.n_blocks + blockIdx.x] = (uint32_t)n_used;
  }
}

// One thread per pair: the block sums in block order, F_ST = sum num / sum den, NaN without a used locus.
__global__ void k_fst_total(const double2* block_sums, const uint32_t* block_used, uint64_t n_blocks, uint32_t n_pairs, double* fst) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pairs) return;
  double num = 0.0, den = 0.0;
  uint64_t used = 0;
  for (uint64_t x = 0; x < n_blocks; ++x) {
    const double2 s = block_sums[(uint64_t)p * n_blocks + x];
    num = __dadd_rn(num, s.x); den = __dadd_rn(den, s.y);
    used += block_used[(uint64_t)p * n_blocks + x];
  }
  fst[p] = used ? __ddiv_rn(num, den) : __longlong_as_double(0x7FF8000000000000ll);
}

// One thread per (pair, window): the used loci of rows [range.x, range.y) added in row order, and their number.
__global__ void k_fst_windows(FstParams P, const uint2* range, uint64_t n_windows, double* out /* [n_pairs][n_windows][3] */) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (uint64_t)P.n_pairs * n_windows) return;
  const uint32_t p = (uint32_t)(i / n_windows);
  const uint2 pr = __ldg(P.pairs + p), rg = __ldg(range + i % n_windows);
  double num = 0.0, den = 0.0;
  uint32_t used = 0;
  for (uint64_t l = rg.x; l < rg.y; ++l) {
    if (P.keep && !P.keep[l]) continue;
    double n_, d_;
    if (!fst_term(__ldg(P.counts + l * P.n_groups + pr.x), __ldg(P.counts + l * P.n_groups + pr.y), P.method, n_, d_)) continue;
    num = __dadd_rn(num, n_); den = __dadd_rn(den, d_);
    ++used;
  }
  out[i * 3] = num; out[i * 3 + 1] = den; out[i * 3 + 2] = (double)used;
}

}  // namespace kgl
