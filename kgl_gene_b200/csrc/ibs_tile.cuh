// ibs_tile.cuh -- K4: pairwise identity-by-state over 64x64 sample-pair tiles (sm_100a, integer pipes).
//
// No reference routine exists (SURVEY 8c: parity unpinned); the matrix is the {0,1,2} genome x variant matrix that
// VariantDBVariant::genomeData() describes (kgl_variant_db_variant.h:49-51), IBS2: g_a == g_b, IBS1: |g_a - g_b| == 1,
// IBS0: |g_a - g_b| == 2, over the loci where neither genome is coded 3.
//
// Input: the sample-major, warp-interleaved bit planes of sample_major.cuh
//   lo, hi, valid : uint32 [n_gblocks][n_words][32]      (valid = ~(lo & hi); word (gb, w, lane) = genome 32*gb + lane, loci 32w..)
// With the raw code planes (0 = 00, 1 = lo, 2 = hi, 3 = both) a pair differs by one  <=> exactly one of them is het
// <=> lo_a ^ lo_b, and by two <=> hi_a ^ hi_b without lo_a ^ lo_b. Per pair and 32-locus word:
//     v  = V_a & V_b                    t1 = (lo_a ^ lo_b) & v                    t0 = (hi_a ^ hi_b) & ~t1 & v
// i.e. 4 LOP3 for the three bit vectors {t0, t1, v} (3 LOP3 and two vectors when the population has no code-3 cell).
// POPC issues at 1/4 of the LOP3 rate on this chip (15.9 vs 62.5 per clk per SM, tools/kbench.cu), so the vectors of two
// consecutive words and a per-pair "ones" register first go through a carry-save adder (2 LOP3) and only the carry word
// is counted: per pair-word 7 LOP3 + 1.5 POPC + 1.5 IADD instead of 4 LOP3 + 3 POPC + 3 IADD, which balances the ALU
// pipe (7/64 clk) against the POPC pipe (1.5/16 clk).
//
// Structure: persistent CTAs, one per SM. Work unit = (tile, chunk of words), units are dealt round-robin in chunk-major
// order so that the CTAs running at the same time read the same words of different genome blocks (L2 reuse). A producer
// warp streams the two 64-genome strips of a unit through a 4-deep shared-memory ring with 1-D TMA bulk copies
// (2 KB per (side, plane, genome block)); 8 consumer warps hold a 4x4 pair block per thread: 48 accumulators + 48 carry-save
// registers. A unit ends with 48 (atomic, when the words are split over several chunks) adds per thread into
// acc[tile][3][64*64]; integer adds commute, so the result does not depend on the schedule.
#pragma once
#include "stream_common.cuh"

namespace kgl {

constexpr int kIbsT = 64;                       // genomes per tile side
constexpr int kIbsKW = 16;                      // 32-locus words per stage
constexpr int kIbsStages = 6;
constexpr int kIbsPrefetch = 3;                 // stages in flight ahead of the consumers; a refilled slot was drained kIbsStages - kIbsPrefetch steps ago
constexpr uint32_t kIbsStripBytes = kIbsKW * 128;          // one (side, plane, genome block) strip of a stage
constexpr uint32_t kIbsTileCells = kIbsT * kIbsT;

__host__ __device__ constexpr uint32_t ibs_stage_bytes(bool missing) { return 2u * (missing ? 3u : 2u) * 2u * kIbsStripBytes; }
__host__ __device__ constexpr size_t ibs_smem_bytes(bool missing) { return (size_t)kIbsStages * ibs_stage_bytes(missing) + 2 * kIbsStages * 8 + 128; }

struct IbsParams {
  const uint32_t* plane[3];   // lo, hi, valid
  uint64_t n_words;           // words per genome-block row (pitch of the planes)
  uint32_t words_used;        // words that hold loci; even (padding loci are coded 3)
  const uint2* tiles;         // tile coordinates (ta, tb) in units of 64 genomes
  uint32_t n_tiles;
  uint32_t words_per_chunk;   // multiple of kIbsKW
  uint32_t n_chunks;
  uint32_t* acc;              // [n_tiles][3][64*64] = {IBS0, IBS1, valid}; zeroed by the caller when n_chunks > 1
};

// Producer side of the ring: walks the CTA's units in order and issues one stage (16 words of both strips) per call.
// All lanes of the calling warp execute it; lane l < 4*NP owns the (side, plane, genome block) strip l.
template <int NP>
struct IbsProducer {
  uint32_t u, w, w1, it, s, ph;
  const uint32_t* src_row;
  bool owner;
  uint32_t side, plane, gbl, strip;

  __device__ __forceinline__ void open_unit(const IbsParams& P, uint32_t n_units) {
    if (u >= n_units) return;
    const uint32_t chunk = u / P.n_tiles, tile = u - chunk * P.n_tiles;
    const uint2 tc = P.tiles[tile];
    const uint64_t gb = (uint64_t)(side ? tc.y : tc.x) * 2 + gbl;
    const uint32_t* pl = plane == 0 ? P.plane[0] : (plane == 1 ? P.plane[1] : P.plane[2]);
    src_row = pl + gb * P.n_words * 32;
    w = chunk * P.words_per_chunk;
    w1 = min(w + P.words_per_chunk, P.words_used);
  }
  __device__ __forceinline__ void init(const IbsParams& P, uint32_t n_units, uint32_t lane) {
    strip = lane; owner = strip < 4u * NP;
    side = strip / (2 * NP); plane = (strip / 2) % NP; gbl = strip & 1;
    u = blockIdx.x; it = 0; s = 0; ph = 0; w = 0; w1 = 0; src_row = nullptr;
    open_unit(P, n_units);
  }
  __device__ __forceinline__ bool done(uint32_t n_units) const { return u >= n_units; }
  // Issues the next stage; waits for its slot to be drained first (not needed for the first kIbsStages stages).
  __device__ __forceinline__ void issue(const IbsParams& P, uint32_t n_units, unsigned char* smem_raw, uint32_t stage_bytes,
                                        uint32_t bar_full, uint32_t bar_empty, uint32_t lane) {
    if (it >= (uint32_t)kIbsStages) mbar_wait(bar_empty + 8 * s, ph ^ 1);
    const uint32_t bytes = min((uint32_t)kIbsKW, w1 - w) * 128u;
    if (lane == 0) mbar_expect_tx(bar_full + 8 * s, bytes * 4u * NP);
    __syncwarp();
    if (owner) tma_bulk_g2s(smem_u32(smem_raw + (size_t)s * stage_bytes + strip * kIbsStripBytes), src_row + (size_t)w * 32, bytes, bar_full + 8 * s);
    ++it;
    if (++s == kIbsStages) { s = 0; ph ^= 1; }
    w += kIbsKW;
    if (w >= w1) { u += gridDim.x; open_unit(P, n_units); }
  }
};

// TJ = pairs per thread along B (4 -> 8 warps of 4x4 pair blocks, 2 -> 16 warps of 4x2). There is no producer warp: an odd
// warp count would leave three (five) warps on one SM sub-partition and cap every thread at 168 (96) registers. Warp 0
// refills, at the end of every step, the slot drained kIbsStages - kIbsPrefetch steps earlier, so it practically never waits.
template <bool MISSING, int TJ>
__global__ void __launch_bounds__(kIbsTileCells / (4 * TJ), 1)
k_ibs_tiles(const IbsParams P) {
  constexpr int NP = MISSING ? 3 : 2;
  constexpr int NQ = MISSING ? 3 : 2;           // counted vectors per pair: t0, t1 (, v)
  constexpr int NWARPS = kIbsTileCells / (4 * TJ) / 32;
  constexpr int TXN = kIbsT / TJ;               // threads along B
  constexpr uint32_t STAGE = ibs_stage_bytes(MISSING);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kIbsStages * STAGE);
  const uint32_t bar_full = smem_u32(s_bar), bar_empty = smem_u32(s_bar + kIbsStages);
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    for (int s = 0; s < kIbsStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, NWARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  const uint32_t n_units = P.n_tiles * P.n_chunks;
  IbsProducer<NP> prod;
  if (warp == 0) {
    prod.init(P, n_units, lane);
    for (int i = 0; i < kIbsPrefetch && !prod.done(n_units); ++i) prod.issue(P, n_units, smem_raw, STAGE, bar_full, bar_empty, lane);
  }

  // ===== consumers: thread = 4 x TJ pairs; A genomes ty*4.., B genomes tx*TJ.. =====
  const uint32_t tx = tid % TXN, ty = tid / TXN;
  // word offset of the thread's genomes inside a strip row: strip (gbl) then lane group
  const uint32_t a_off = (ty >> 3) * (kIbsStripBytes / 4) + (ty & 7) * 4;
  const uint32_t b_off = ((tx * TJ) >> 5) * (kIbsStripBytes / 4) + ((tx * TJ) & 31);
  uint32_t s = 0, ph = 0;

  for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x) {
    const uint32_t chunk = u / P.n_tiles, tile = u - chunk * P.n_tiles;
    const uint32_t w0 = chunk * P.words_per_chunk, w1 = min(w0 + P.words_per_chunk, P.words_used);
    uint32_t acc[NQ][4][TJ], ones[NQ][4][TJ];
#pragma unroll
    for (int q = 0; q < NQ; ++q)
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TJ; ++j) { acc[q][i][j] = 0; ones[q][i][j] = 0; }

    for (uint32_t w = w0; w < w1; w += kIbsKW) {
      const uint32_t nw = min((uint32_t)kIbsKW, w1 - w);          // even
      mbar_wait(bar_full + 8 * s, ph);
      const uint32_t* st = reinterpret_cast<const uint32_t*>(smem_raw + (size_t)s * STAGE);
      // strips: side A planes 0..NP-1 (two genome blocks each), then side B
      const uint32_t* sa = st + a_off;
      const uint32_t* sb = st + NP * 2 * (kIbsStripBytes / 4) + b_off;
#pragma unroll 1
      for (uint32_t k = 0; k < nw; k += 2) {
        uint32_t A[2][NP][4], B[2][NP][TJ];
#pragma unroll
        for (int d = 0; d < 2; ++d)
#pragma unroll
          for (int p = 0; p < NP; ++p) {
            const uint4 a = *reinterpret_cast<const uint4*>(sa + p * 2 * (kIbsStripBytes / 4) + (k + d) * 32);
            A[d][p][0] = a.x; A[d][p][1] = a.y; A[d][p][2] = a.z; A[d][p][3] = a.w;
            if constexpr (TJ == 4) {
              const uint4 b = *reinterpret_cast<const uint4*>(sb + p * 2 * (kIbsStripBytes / 4) + (k + d) * 32);
              B[d][p][0] = b.x; B[d][p][1] = b.y; B[d][p][2] = b.z; B[d][p][3] = b.w;
            } else {
              const uint2 b = *reinterpret_cast<const uint2*>(sb + p * 2 * (kIbsStripBytes / 4) + (k + d) * 32);
              B[d][p][0] = b.x; B[d][p][1] = b.y;
            }
          }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < TJ; ++j) {
            uint32_t t[2][NQ];
#pragma unroll
            for (int d = 0; d < 2; ++d) {
              const uint32_t dl = A[d][0][i] ^ B[d][0][j];
              const uint32_t dh = A[d][1][i] ^ B[d][1][j];
              if (MISSING) {
                const uint32_t v = A[d][2][i] & B[d][2][j];
                t[d][1] = dl & v;
                // dh & ~t1 & v as ONE lop3 on (dh, t1, v): left to itself the compiler expands ~t1 & v into ~dl & v (4 inputs, 2 LOP3)
                asm("lop3.b32 %0, %1, %2, %3, 0x20;" : "=r"(t[d][0]) : "r"(dh), "r"(t[d][1]), "r"(v));
                t[d][NQ - 1] = v;
              } else {
                t[d][1] = dl;
                t[d][0] = dh & ~dl;
              }
            }
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
              uint32_t carry;
              csa(carry, ones[q][i][j], ones[q][i][j], t[0][q], t[1][q]);
              acc[q][i][j] += __popc(carry);
            }
          }
      }
      if (warp == 0 && !prod.done(n_units)) prod.issue(P, n_units, smem_raw, STAGE, bar_full, bar_empty, lane);
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_empty + 8 * s);
      if (++s == kIbsStages) { s = 0; ph ^= 1; }
    }

    uint32_t* out = P.acc + (size_t)tile * 3 * kIbsTileCells;
#pragma unroll
    for (int q = 0; q < NQ; ++q)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint32_t c[TJ];
#pragma unroll
        for (int j = 0; j < TJ; ++j) c[j] = 2u * acc[q][i][j] + __popc(ones[q][i][j]);
        uint32_t* o = out + (size_t)q * kIbsTileCells + (ty * 4 + i) * kIbsT + tx * TJ;
        if (P.n_chunks > 1) {
#pragma unroll
          for (int j = 0; j < TJ; ++j) if (c[j]) atomicAdd(o + j, c[j]);
        } else {
#pragma unroll
          for (int j = 0; j < TJ; ++j) o[j] = c[j];
        }
      }
  }
}

// ---- "dense minus sparse" for code-3 cells ------------------------------------------------------------------------------
// When the population's code-3 cells are indexed (sparse_events.cuh: genome-major, row-sorted keys), the dense kernel runs
// its two-plane form on PRE-MASKED planes (code 3 -> 0) and this pair of kernels repairs the result exactly:
//   a pair (a,b) was counted at a locus where a is coded 3 as if a were hom-ref: IBS1 if b is het, IBS0 if b is hom-alt.
//   C1[a][b] = #{l in dropped(a) : b het},  C0[a][b] = #{l in dropped(a) : b hom-alt},  J[a][b] = #{l in dropped(a) : b coded 3}
//   IBS1 = IBS1' - C1[a][b] - C1[b][a],  IBS0 = IBS0' - C0[a][b] - C0[b][a],  valid = L - |dropped(a)| - |dropped(b)| + J[a][b]
// The counts come from the loci-major matrix: a thread owns one genome of one side of a tile, walks that genome's dropped
// rows and adds the partner unit's three 64-genome bit vectors into bit-sliced counters (one 16-byte load per row).
__global__ void __launch_bounds__(256)
k_ibs_premask(const uint4* __restrict__ lo, const uint4* __restrict__ hi, uint64_t n_vec, uint4* __restrict__ lo_m, uint4* __restrict__ hi_m) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_vec) return;
  const uint4 a = lo[i], b = hi[i];
  lo_m[i] = make_uint4(a.x & ~b.x, a.y & ~b.y, a.z & ~b.z, a.w & ~b.w);
  hi_m[i] = make_uint4(b.x & ~a.x, b.y & ~a.y, b.z & ~a.z, b.w & ~a.w);
}

constexpr int kIbsFixLevels = 16;               // counter levels; 32,760 rows per genome between flushes
constexpr int kIbsFixLow = 4;                   // levels 0..3 take 8 rows at a time; then level 3 (weight 8) moves into levels 4..15
constexpr uint32_t kIbsFixRows = (1u << (kIbsFixLevels - 1)) - 8;    // rows a thread adds between two flushes of its counters

// Sparse repair of the code-3 cells (dense-minus-sparse, DESIGN 4b). A thread owns one genome of one side of a tile and one
// segment (blockIdx.y of gridDim.y) of that genome's dropped rows; it adds the partner unit's three 64-bit vectors (hom-alt,
// het, code 3) into bit-sliced counters. The counters are two-stage: a row costs a ripple through levels 0..3; after 8 rows
// (residue <= 7, so no carry leaves level 3) the bit of level 3 moves up, and levels 4..15 count units of 8 -- a third of the
// logic of a 16-level ripple per row. With gridDim.y > 1 plane 2 (J) must be zero on
// entry and is accumulated atomically.
__global__ void __launch_bounds__(128)
k_ibs_missing_fix(const uint4* __restrict__ packed, uint32_t units, const unsigned long long* __restrict__ keys,
                  const uint64_t* __restrict__ seg, uint64_t n_genomes, const uint2* __restrict__ tiles, uint32_t* __restrict__ acc) {
  const uint32_t tile = blockIdx.x;
  const uint2 tc = tiles[tile];
  const uint32_t side = threadIdx.x >> 6, al = threadIdx.x & 63;
  const uint64_t a = (uint64_t)(side ? tc.y : tc.x) * kIbsT + al;
  const uint32_t partner = side ? tc.x : tc.y;
  const bool split = gridDim.y > 1;
  uint32_t* out = acc + (size_t)tile * 3 * kIbsTileCells;
  uint64_t k = 0, k_end = 0;
  if (a < n_genomes) {
    const uint64_t k0 = seg[a], len = seg[a + 1] - k0;
    k = k0 + len * blockIdx.y / gridDim.y;
    k_end = k0 + len * (blockIdx.y + 1) / gridDim.y;
  }
  bool first = true;
  do {
    uint64_t cnt[3][kIbsFixLevels];
#pragma unroll
    for (int q = 0; q < 3; ++q)
#pragma unroll
      for (int lv = 0; lv < kIbsFixLevels; ++lv) cnt[q][lv] = 0;
    const uint64_t k_stop = min(k_end, k + (uint64_t)kIbsFixRows);
    while (k < k_stop) {
      // eight rows at a time: the eight keys, then the eight partner units, are requested together (the walk is bound by the
      // latency of these two dependent loads, not by the counters)
      const uint32_t n8 = (uint32_t)min((uint64_t)8, k_stop - k);
      uint4 v8[8];
      {
        uint32_t row8[8];
#pragma unroll
        for (uint32_t i = 0; i < 8; ++i) row8[i] = i < n8 ? (uint32_t)keys[k + i] : 0u;
#pragma unroll
        for (uint32_t i = 0; i < 8; ++i) v8[i] = i < n8 ? __ldg(packed + (size_t)row8[i] * units + partner) : make_uint4(0u, 0u, 0u, 0u);
      }
      k += n8;
#pragma unroll
      for (uint32_t i = 0; i < 8; ++i) {
        const uint4 v = v8[i];                               // rows past n8 are all-zero units: they add nothing
        const uint64_t lo = (uint64_t)v.x | ((uint64_t)v.y << 32), hi = (uint64_t)v.z | ((uint64_t)v.w << 32);
        uint64_t x[3] = {hi & ~lo, lo & ~hi, lo & hi};
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          uint64_t carry = x[q];
#pragma unroll
          for (int lv = 0; lv < kIbsFixLow; ++lv) {
            const uint64_t t = cnt[q][lv] & carry;
            cnt[q][lv] ^= carry;
            carry = t;
          }
        }
      }
      // the low counter held at most 7 before these <= 8 rows: its level 3 (weight 8) moves into level 4 (weight 8) and clears
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        uint64_t carry = cnt[q][kIbsFixLow - 1];
        cnt[q][kIbsFixLow - 1] = 0;
#pragma unroll
        for (int lv = kIbsFixLow; lv < kIbsFixLevels; ++lv) {
          const uint64_t t = cnt[q][lv] & carry;
          cnt[q][lv] ^= carry;
          carry = t;
        }
      }
    }
    for (int b = 0; b < kIbsT; ++b) {
      uint32_t c[3];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        uint32_t s = 0;
#pragma unroll
        for (int lv = 0; lv < kIbsFixLow - 1; ++lv) s += (uint32_t)((cnt[q][lv] >> b) & 1ull) << lv;
        // level kIbsFixLow - 1 was moved up: levels >= kIbsFixLow count units of 2^(kIbsFixLow - 1)
#pragma unroll
        for (int lv = kIbsFixLow; lv < kIbsFixLevels; ++lv) s += (uint32_t)((cnt[q][lv] >> b) & 1ull) << (lv - 1);
        c[q] = s;
      }
      const uint32_t cell = side ? (uint32_t)b * kIbsT + al : al * kIbsT + (uint32_t)b;
      if (c[0]) atomicSub(out + cell, c[0]);
      if (c[1]) atomicSub(out + kIbsTileCells + cell, c[1]);
      if (side == 0) {                            // J is symmetric: side 0 alone writes it
        if (split) { if (c[2]) atomicAdd(out + 2 * kIbsTileCells + cell, c[2]); }
        else if (first) out[2 * kIbsTileCells + cell] = c[2];
        else if (c[2]) out[2 * kIbsTileCells + cell] += c[2];
      }
    }
    first = false;
  } while (k < k_end);
}

// Third plane of the in-kernel form (populations whose code-3 cells are too many to index).
__global__ void __launch_bounds__(256)
k_valid_plane(const uint4* __restrict__ lo, const uint4* __restrict__ hi, uint64_t n_vec, uint4* __restrict__ valid) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_vec) return;
  const uint4 a = lo[i], b = hi[i];
  valid[i] = make_uint4(~(a.x & b.x), ~(a.y & b.y), ~(a.z & b.z), ~(a.w & b.w));
}

// acc -> {IBS0, IBS1, IBS2, valid} in the caller's layout.
//   mode 0: out[tile][64][64][4]                                       (compact tiles, the multi-GPU payload)
//   mode 1: out[(a - row_begin)][n_genomes][4] for a in [row_begin,row_end); with `mirror` also the transposed cell
__global__ void __launch_bounds__(256)
k_ibs_finalize(const uint32_t* __restrict__ acc, const uint2* __restrict__ tiles, uint32_t n_tiles,
               int valid_mode /* 0: n_loci for every pair; 1: acc[2] = valid count; 2: acc[2] = J, seg = dropped-cell segments */,
               const uint64_t* __restrict__ seg, uint32_t n_loci,
               int mode, uint64_t n_genomes, uint64_t row_begin, uint64_t row_end, int mirror, uint32_t* __restrict__ out) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (uint64_t)n_tiles * kIbsTileCells) return;
  const uint32_t tile = (uint32_t)(idx / kIbsTileCells), cell = (uint32_t)(idx % kIbsTileCells);
  const uint32_t* a3 = acc + (size_t)tile * 3 * kIbsTileCells + cell;
  const uint32_t c0 = a3[0], c1 = a3[kIbsTileCells];
  const uint2 tc = tiles[tile];
  const uint64_t a = (uint64_t)tc.x * kIbsT + cell / kIbsT, b = (uint64_t)tc.y * kIbsT + cell % kIbsT;
  const bool live = a < n_genomes && b < n_genomes;
  uint32_t cv = n_loci;
  if (valid_mode == 1) cv = a3[2 * kIbsTileCells];
  else if (valid_mode == 2 && live) cv = n_loci - (uint32_t)(seg[a + 1] - seg[a]) - (uint32_t)(seg[b + 1] - seg[b]) + a3[2 * kIbsTileCells];
  const uint4 r = live ? make_uint4(c0, c1, cv - c0 - c1, cv) : make_uint4(0, 0, 0, 0);    // cells of padding genomes read 0
  if (mode == 0) { reinterpret_cast<uint4*>(out)[idx] = r; return; }
  if (!live) return;
  if (a >= row_begin && a < row_end) reinterpret_cast<uint4*>(out)[(a - row_begin) * n_genomes + b] = r;
  if (mirror && tc.x != tc.y && b >= row_begin && b < row_end) reinterpret_cast<uint4*>(out)[(b - row_begin) * n_genomes + a] = r;
}

}  // namespace kgl
