// ld.cuh -- linkage disequilibrium: the genotypic r^2 of locus pairs inside a window, from exact int8 Gram runs over the loci
// (kgl_b200_run_ld_pairs, kgl_b200_run_ld_prune).
//
// For loci i, j and the genomes where neither cell is coded 3, with g the dosage {0,1,2} (code 3 -> 0), q = g^2 and c the code-3
// indicator, every sum r^2 needs is a dot product over genomes of two rows of the loci-major codes (pca.cuh) under a byte table:
//     GG = sum g_i g_j,  CC = sum c_i c_j,  GC_ij = sum g_i c_j,  QC_ij = sum q_i c_j
// and the per-locus totals s = n1 + 2 n2, q = n1 + 4 n2, c = n3 come from the raw counts. Then, in int64,
//     n = N - c_i - c_j + CC   S_i = s_i - GC_ij   S_j = s_j - GC_ji   Q_i = q_i - QC_ij   Q_j = q_j - QC_ji
//     cov = n GG - S_i S_j     var_i = n Q_i - S_i^2     var_j = n Q_j - S_j^2
//     r^2 = cov^2 / (var_i var_j)         one rounded product each side and one rounded division; NaN when a variance is 0
// Padding genomes (K positions >= N) hold code 0, which every table reads as 0: they add to no product, which is why n is formed
// from N and the code-3 counts rather than from a "valid" indicator (that would count the padding). Every term is below 4 N^2 <
// 2^53 for N < 2^25, so each int64 converts to double exactly and the result is bit-reproducible (tests/ld_oracle.py).
// Without code-3 cells only the GG run is needed (n = N, S = s, Q = q).
#pragma once
#include "king.cuh"

#include <algorithm>
#include <vector>

namespace kgl {

static_assert(sizeof(kgl_b200_ld_pair) == 24 && offsetof(kgl_b200_ld_pair, r2) == 16, "kgl_b200_ld_pair: the 24-byte layout of include/kgl_b200.h");

constexpr uint32_t kGramTableSquare = 0x00040100u;      // squared dosage {0,1,4}, code 3 read as 0
constexpr uint32_t kLdNotEligible = 0xFFFFFFFFu;        // rank of a locus outside the eligible set
constexpr uint64_t kLdBlockBytes = (uint64_t)kGramM * kGramN * 4;

// Compact int32 blocks one band tile costs in a slab: GG alone, or GG, CC, GC and QC, the last two also over the mirror tile (J, I)
// when the tile is off the diagonal (a diagonal block holds both GC_ij and GC_ji).
inline uint64_t ld_tile_blocks(bool code3, bool diagonal) { return code3 ? (diagonal ? 4 : 6) : 1; }

// The band: every 256 x 256 locus tile (I, J), I <= J, that holds at least one in-window pair of eligible loci, ascending, cut into
// slabs whose int32 blocks stay within budget_bytes (a slab holds at least one tile). slab_begin[s] = first tile of slab s, with
// tiles.size() at the end.
struct LdBand {
  std::vector<uint2> tiles;
  std::vector<uint32_t> slab_begin;
};

// rank[l] = index of locus l among the eligible loci, kLdNotEligible outside them. offsets (sorted) are read only with a bp limit.
// Pair i < j is in the window iff (window_loci == 0 || rank j - rank i < window_loci) and (window_bp == 0 || off j - off i <=
// window_bp); both limits are monotone in j, so the partners of eligible i are exactly the eligible loci after it up to a last
// one, jmax(i), which never decreases with i. The tiles of block row I are then the blocks J with an eligible locus between the
// first partner of any i in I and the largest jmax of I.
inline LdBand ld_band(const uint32_t* rank, const uint32_t* offsets, uint64_t n_loci, uint32_t window_loci, uint32_t window_bp,
                      bool code3, uint64_t budget_bytes) {
  const uint64_t n_blocks = (n_loci + kGramM - 1) / kGramM;
  std::vector<uint64_t> elig;
  std::vector<uint32_t> count(n_blocks, 0);
  for (uint64_t l = 0; l < n_loci; ++l)
    if (rank[l] != kLdNotEligible) { elig.push_back(l); ++count[l / kGramM]; }
  const uint64_t none = ~0ull;
  std::vector<uint64_t> lo(n_blocks, none), hi(n_blocks, 0);
  const uint64_t m = elig.size();
  uint64_t h = 0;
  for (uint64_t r = 0; r < m; ++r) {
    h = std::max(h, r);
    while (h + 1 < m && (window_loci == 0 || h + 1 - r < window_loci) &&
           (window_bp == 0 || (uint64_t)offsets[elig[h + 1]] - offsets[elig[r]] <= window_bp))
      ++h;
    if (h == r) continue;
    const uint64_t I = elig[r] / kGramM;
    lo[I] = std::min(lo[I], elig[r + 1] / kGramM);
    hi[I] = std::max(hi[I], elig[h] / kGramM);
  }
  LdBand band;
  const uint64_t budget = std::max<uint64_t>(budget_bytes / kLdBlockBytes, ld_tile_blocks(code3, false));
  uint64_t used = 0;
  for (uint64_t I = 0; I < n_blocks; ++I) {
    if (lo[I] == none) continue;
    for (uint64_t J = lo[I]; J <= hi[I]; ++J) {
      if (count[J] == 0) continue;
      const uint64_t cost = ld_tile_blocks(code3, I == J);
      if (band.slab_begin.empty() || used + cost > budget) { band.slab_begin.push_back((uint32_t)band.tiles.size()); used = 0; }
      used += cost;
      band.tiles.push_back(make_uint2((uint32_t)I, (uint32_t)J));
    }
  }
  band.slab_begin.push_back((uint32_t)band.tiles.size());
  return band;
}

struct LdTiles {
  const int32_t* gg;            // compact blocks of the band tiles
  const int32_t* cc;            // the same tiles; cc, gc and qc are null when the population has no code-3 cell
  const int32_t* gc;            // band tiles, then the mirror tiles of the off-diagonal ones
  const int32_t* qc;
  const uint2* tiles;
  const uint32_t* mirror;       // per band tile: the gc / qc block of (J, I) (the tile itself on the diagonal)
  uint32_t n_tiles;
  const uint32_t* counts;       // raw per-locus counts n0..n3
  const uint32_t* rank;
  const uint32_t* offsets;      // null without a bp limit
  uint64_t n_loci;
  uint64_t n_genomes;
  uint32_t window_loci, window_bp;
};

// Cell `cell` of band tile `tile`: false unless it is an in-window pair a < b of eligible loci; then n and r^2 by the sequence above.
__device__ __forceinline__ bool ld_cell(const LdTiles& T, uint32_t tile, uint32_t cell, uint32_t& a, uint32_t& b, uint32_t& n_valid,
                                        double& r2) {
  const uint2 tc = T.tiles[tile];
  const uint32_t ia = cell / kGramN, ib = cell % kGramN;
  a = tc.x * kGramM + ia; b = tc.y * kGramN + ib;
  if (a >= b || b >= T.n_loci) return false;
  const uint32_t rank_a = T.rank[a], rank_b = T.rank[b];
  if (rank_a == kLdNotEligible || rank_b == kLdNotEligible) return false;
  if (T.window_loci != 0 && rank_b - rank_a >= T.window_loci) return false;
  if (T.window_bp != 0 && T.offsets[b] - T.offsets[a] > T.window_bp) return false;
  const uint4 ca = reinterpret_cast<const uint4*>(T.counts)[a], cb = reinterpret_cast<const uint4*>(T.counts)[b];
  const size_t at = (size_t)tile * kGramM * kGramN + cell;
  long long n = (long long)T.n_genomes - ca.w - cb.w;
  long long s_a = ca.y + 2ll * ca.z, s_b = cb.y + 2ll * cb.z, q_a = ca.y + 4ll * ca.z, q_b = cb.y + 4ll * cb.z;
  if (T.cc) {
    const size_t mt = (size_t)T.mirror[tile] * kGramM * kGramN + (size_t)ib * kGramN + ia;
    n += T.cc[at];
    s_a -= T.gc[at]; q_a -= T.qc[at];
    s_b -= T.gc[mt]; q_b -= T.qc[mt];
  }
  const long long cov = n * T.gg[at] - s_a * s_b, var_a = n * q_a - s_a * s_a, var_b = n * q_b - s_b * s_b;
  n_valid = (uint32_t)n;
  r2 = (var_a == 0 || var_b == 0) ? __longlong_as_double(0x7FF8000000000000ll)
                                  : __ddiv_rn(__dmul_rn((double)cov, (double)cov), __dmul_rn((double)var_a, (double)var_b));
  return true;
}

// Pair compactor over the cells of a slab's band tiles, the cursor protocol of k_king_pairs. Pairs mode (prune == 0): every pair
// with r^2 >= threshold as a record, keys[i] = (a << 32) | b. Prune mode: only keys[i] = (b << 32) | a of the pairs with r^2 >
// threshold, the order the greedy scan walks them in. NaN never qualifies.
__global__ void __launch_bounds__(256)
k_ld_pairs(const LdTiles T, double threshold, int prune, uint64_t capacity, kgl_b200_ld_pair* __restrict__ pairs,
           unsigned long long* __restrict__ keys, uint32_t* __restrict__ index, unsigned long long* __restrict__ cursor) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool take = false;
  uint32_t a = 0, b = 0, n_valid = 0;
  double r2 = 0.0;
  if (idx < (uint64_t)T.n_tiles * kGramM * kGramN && ld_cell(T, (uint32_t)(idx / (kGramM * kGramN)), (uint32_t)(idx % (kGramM * kGramN)), a, b, n_valid, r2))
    take = prune ? r2 > threshold : r2 >= threshold;
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t mask = __ballot_sync(0xFFFFFFFFu, take);
  if (mask == 0u) return;
  unsigned long long base = 0;
  if (lane == (uint32_t)(__ffs(mask) - 1)) base = atomicAdd(cursor, (unsigned long long)__popc(mask));
  base = __shfl_sync(0xFFFFFFFFu, base, __ffs(mask) - 1);
  if (!take) return;
  const uint64_t pos = base + (uint64_t)__popc(mask & ((1u << lane) - 1u));
  if (pos >= capacity) return;
  if (prune) {
    keys[pos] = ((unsigned long long)b << 32) | a;
  } else {
    kgl_b200_ld_pair r;
    r.a = a; r.b = b; r.n_valid = n_valid; r.reserved = 0; r.r2 = r2;
    pairs[pos] = r;
    keys[pos] = ((unsigned long long)a << 32) | b;
  }
  index[pos] = (uint32_t)pos;
}

}  // namespace kgl
