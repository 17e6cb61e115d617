// gram_i8.cuh -- K5: the genotype Gram matrix S = G G^T on the 5th-generation tensor cores (tcgen05.mma kind::i8, sm_100a).
//
// G[g][l] in {0,1,2} is the alt-allele dosage of genome g at locus l (code 3 -> 0), so S[i][j] = sum_l g_il g_jl is an exact
// int32 for L < 2^29. The centred relationship matrix follows without floating point in the contraction (SURVEY 8d):
//     sum_l (g_il - 2 p_l)(g_jl - 2 p_l) = S[i][j] - 2 (Gp)_i - 2 (Gp)_j + 4 sum_l p_l^2
// and, without code-3 cells, S also ties the tensor-core path to the popcount path: sum_l (g_il - g_jl)^2 = IBS1 + 4 IBS0
// = S[i][i] + S[j][j] - 2 S[i][j]  (tests/test_gpu_parity.py).
//
// Operands never exist as int8 in HBM. Input is a genome-major 2-bit code matrix (16 loci per uint32, built once per
// upload by k_codes16 from the sample-major planes); expander warps turn every 32-bit word into 16 int8 with the byte
// permuter (expand16: 9 integer ops per 16 bytes) and write them straight into the 128-byte-swizzled K-major layout
// tcgen05 reads. HBM/L2 traffic is therefore 1/4 byte per genotype, and the expansion costs 0.56 integer ops per operand
// byte = 0.0044 per MAC at a 256 x 256 tile.
//
// CTA = 21 warps: 0-3 epilogue (TMEM lane quadrants 0-3), 4 MMA issuer (one elected thread) + TMEM allocator, 5-20 expanders
// (512 threads = one per operand row of a stage).
// Work unit = (256 x 256 output tile, chunk of K); per K-stage of 128 loci: A 256 x 128 B, B 256 x 128 B (64 KB), 3 stages. The
// tile is two M = 128 MMAs on one B operand: a third less shared-memory traffic per MAC than 128 x 256 (the round-1 shape, bound
// by exactly that traffic: 2.0 -> 3.0 PetaOP/s).
//   expanders : wait empty[s] -> LDG (prefetched a stage ahead) -> expand -> st.shared (swizzled) -> fence.proxy.async -> arrive full[s]
//   MMA       : wait full[s] -> 2 x 4 x tcgen05.mma (K = 32 each, descriptors advanced by 32 B inside the swizzle atom)
//               -> tcgen05.commit empty[s]; after the unit's last stage tcgen05.commit tmem_full[a]
//   epilogue  : wait tmem_full[a] -> tcgen05.ld 32x32b.x32 -> st / red.add to S (int32 adds commute: split-K is exact)
//               -> arrive tmem_empty. The two 256-column accumulators of a tile fill TMEM: unit u+1 starts after unit u's epilogue.
#pragma once
#include "stream_common.cuh"

namespace kgl {

constexpr int kGramM = 256, kGramN = 256, kGramK = 128;         // tile (two M = 128 MMAs share the B operand); K-stage = 128 loci = 128 B per operand row
constexpr int kGramMmaM = 128;                                   // rows per tcgen05.mma (cta_group::1)
constexpr int kGramStages = 3;
constexpr int kGramExpWarps = 16;                                // expander warps: one thread per operand row of a stage (256 + 256)
constexpr int kGramThreads = (5 + kGramExpWarps) * 32;
constexpr uint32_t kGramABytes = kGramM * kGramK, kGramBBytes = kGramN * kGramK;
constexpr uint32_t kGramStageBytes = kGramABytes + kGramBBytes;  // 64 KB
constexpr size_t kGramSmem = (size_t)kGramStages * kGramStageBytes + 1024 /* alignment slack */ + 256 /* barriers */;

// Code matrix layout ("row-block major"): uint32 [ld / 128][k_stages][128 rows][8 words]; a word holds 16 loci, 2 bits each,
// code 3 kept (also at loci >= n_loci: the sample-major planes code them 3), rows >= n_genomes zero. One K-stage of one 128-row block is 4 KB contiguous, so the
// expanders' loads are fully coalesced (16 B per lane, 512 B per warp).
__host__ __device__ inline uint64_t gram_code_index(uint64_t row, uint64_t word, uint64_t k_stages) {
  return (((row >> 7) * k_stages + (word >> 3)) * 128 + (row & 127)) * 8 + (word & 7);
}

struct GramParams {
  const uint32_t* codes;      // layout above
  // B operand (the rows tile column tj selects); nullptr = codes. Its own rows in the same layout and k_stages: the Gram runs of
  // pca.cuh contract a code matrix with a block of base-4 digit rows, a rectangular output written with ld as its row pitch
  const uint32_t* codes_b;
  uint32_t k_stages;          // ceil(n_loci / 128)
  const uint2* tiles;         // (ti, tj): rows 128 ti .., columns 256 tj ..
  uint32_t n_tiles;
  uint32_t stages_per_chunk, n_chunks;
  int32_t* out;               // [ld][ld] (rectangular products: rows of A x ld, ld >= 256 x the largest tile column + 256)
  uint64_t ld;
  // value of a 2-bit code as an operand byte: byte c of the table is the value of code c. 0x00020100 is the dosage {0,1,2} with
  // code 3 read as 0; 0x00000100 / 0x00010000 are the indicators "heterozygous" / "homozygous alternate" (pairwise IBS, ibs_gram.cuh)
  uint32_t table_a, table_b;
  // != 0: tile t of the list is written as its own 256 x 256 block at out + t * 65536 (row stride 256) instead of into the ld x ld
  // matrix -- populations whose N x N matrix would not fit (pairwise IBS, ibs_gram.cuh)
  uint32_t compact;
};

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// K-major operand tile, 128-byte swizzle: rows of 128 B, 8-row groups 1024 B apart (UMMA::SmemDescriptor: start >> 4 in
// [0,14), LBO [16,30) unused for swizzled K-major (1), SBO >> 4 in [32,46), version 1 at [46,48), SWIZZLE_128B = 2 at [61,64)).
__device__ __forceinline__ uint64_t tc_smem_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// UMMA::InstrDescriptor for kind::i8: c_format S32 (2) at [4,6), a/b format unsigned 8-bit (0), K-major both, N >> 3 at [17,23), M >> 4 at [24,29).
constexpr uint32_t kGramIdesc = (2u << 4) | ((uint32_t)(kGramN >> 3) << 17) | ((uint32_t)(kGramMmaM >> 4) << 24);

__device__ __forceinline__ void tc_mma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(kGramIdesc), "r"(accumulate), "r"(0u) : "memory");
}

// 16 two-bit codes -> 16 bytes with the byte permuter: a PRMT selector is four nibbles, so x & 0x3333 selects the bytes
// {c0, c2, c4, c6} of the table {0,1,2,3} and (x >> 2) & 0x3333 the bytes {c1, c3, c5, c7}. The loci of a word come out
// de-interleaved (even, odd, even, odd); A and B are expanded by the same function and a dot product does not care about
// the order of its terms. 2 LOP3 + 3 SHF + 4 PRMT per 16 bytes.
__device__ __forceinline__ uint4 expand16(uint32_t x, uint32_t table) {
  const uint32_t m0 = x & 0x33333333u, m1 = (x >> 2) & 0x33333333u;
  return make_uint4(__byte_perm(table, 0u, m0), __byte_perm(table, 0u, m1), __byte_perm(table, 0u, m0 >> 16), __byte_perm(table, 0u, m1 >> 16));
}

__global__ void __launch_bounds__(kGramThreads, 1)
k_gram_i8(const GramParams P) {
  extern __shared__ unsigned char gram_smem_raw[];
  // 1024-byte alignment for the 128-byte swizzle atoms
  const uint32_t raw = smem_u32(gram_smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  unsigned char* smem = gram_smem_raw + (base - raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kGramStages * kGramStageBytes);
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + kGramStages);
  const uint32_t bar_tfull = smem_u32(bars + 2 * kGramStages), bar_tempty = smem_u32(bars + 2 * kGramStages + 2);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kGramStages + 4);
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    for (int s = 0; s < kGramStages; ++s) { mbar_init(bar_full + 8 * s, kGramExpWarps * 32); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_tfull, 1); mbar_init(bar_tempty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t n_units = P.n_tiles * P.n_chunks;

  if (warp >= 5) {
    // ===================== expanders: thread t owns one operand row of every stage: A row t (t < 128) or B row t - 128 ====
    const uint32_t t = tid - 5 * 32;
    const uint32_t is_b = t >= (uint32_t)kGramM ? 1u : 0u;
    const uint32_t r = is_b ? t - kGramM : t;                    // row inside the A tile / the B tile
    const uint32_t sw = r & 7;                                   // swizzle phase of the row
    const uint32_t table = is_b ? P.table_b : P.table_a;
    const uint32_t* codes = is_b && P.codes_b ? P.codes_b : P.codes;
    const uint32_t row_off = (is_b ? kGramABytes : 0u) + (r >> 3) * 1024 + sw * 128;
    uint32_t s = 0, ph = 0, it = 0;
    constexpr int D = 3;                                          // register prefetch depth in stages (L2/HBM latency ~ one stage time)
    uint4 nx[D][2];                                              // the row's eight words (128 loci) of a stage
    struct Cursor { uint32_t u, ks, ns; };
    auto stages_of = [&](uint32_t uu) {
      const uint32_t chunk = uu / P.n_tiles;
      return min(P.stages_per_chunk, P.k_stages - chunk * P.stages_per_chunk);
    };
    auto advance = [&](Cursor& c) {
      if (++c.ks == c.ns) { c.u += gridDim.x; c.ks = 0; c.ns = c.u < n_units ? stages_of(c.u) : 0; }
    };
    auto fetch = [&](const Cursor& c, uint4 (&dst)[2]) {
      if (c.u >= n_units) return;
      const uint32_t chunk = c.u / P.n_tiles, tile = c.u - chunk * P.n_tiles;
      const uint2 tc = P.tiles[tile];
      const uint64_t ks = (uint64_t)chunk * P.stages_per_chunk + c.ks;
      const uint64_t block = (uint64_t)2 * (is_b ? tc.y : tc.x) + (r >> 7);
      const uint4* src = reinterpret_cast<const uint4*>(codes + (block * P.k_stages + ks) * 1024 + (uint64_t)(r & 127) * 8);
      dst[0] = __ldg(src); dst[1] = __ldg(src + 1);
    };
    Cursor cons{blockIdx.x, 0, 0}, pre;
    cons.ns = cons.u < n_units ? stages_of(cons.u) : 0;
    pre = cons;
#pragma unroll
    for (int j = 0; j < D; ++j) { fetch(pre, nx[j]); advance(pre); }
    while (cons.u < n_units) {
#pragma unroll
      for (int j = 0; j < D; ++j) {
        if (cons.u >= n_units) break;
        const uint32_t wds[8] = {nx[j][0].x, nx[j][0].y, nx[j][0].z, nx[j][0].w, nx[j][1].x, nx[j][1].y, nx[j][1].z, nx[j][1].w};
        fetch(pre, nx[j]); advance(pre);
        if (it >= (uint32_t)kGramStages) mbar_wait(bar_empty + 8 * s, ph ^ 1);
        unsigned char* row = smem + (size_t)s * kGramStageBytes + row_off;
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) *reinterpret_cast<uint4*>(row + ((c ^ sw) * 16)) = expand16(wds[c], table);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(bar_full + 8 * s);
        ++it;
        if (++s == kGramStages) { s = 0; ph ^= 1; }
        advance(cons);
      }
    }
  } else if (warp == 4) {
    // ===================== MMA issuer =====================
    uint32_t s = 0, ph = 0, ui = 0;
    for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x, ++ui) {
      const uint32_t chunk = u / P.n_tiles;
      const uint32_t ns = min(P.stages_per_chunk, P.k_stages - chunk * P.stages_per_chunk);
      // one accumulator set (2 x 256 columns = all of TMEM): the MMAs of a unit start when the epilogue of the unit before has
      // drained it -- a unit is thousands of stages long, the epilogue a few microseconds
      if (ui >= 1) mbar_wait(bar_tempty, (ui - 1) & 1);
      tc_fence_after();
      for (uint32_t k = 0; k < ns; ++k) {
        mbar_wait(bar_full + 8 * s, ph);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t sa = base + s * kGramStageBytes, sb = sa + kGramABytes;
#pragma unroll
          for (uint32_t kk = 0; kk < kGramK / 32; ++kk) {
            const uint64_t bdesc = tc_smem_desc(sb + kk * 32);
            tc_mma_i8(tmem_base, tc_smem_desc(sa + kk * 32), bdesc, (k | kk) ? 1u : 0u);                                        // rows 0..127
            tc_mma_i8(tmem_base + kGramN, tc_smem_desc(sa + kGramMmaM * kGramK + kk * 32), bdesc, (k | kk) ? 1u : 0u);          // rows 128..255
          }
          tc_commit(bar_empty + 8 * s);
          if (k + 1 == ns) tc_commit(bar_tfull);
        }
        __syncwarp();
        if (++s == kGramStages) { s = 0; ph ^= 1; }
      }
    }
  } else {
    // ===================== epilogue: warp q owns TMEM lanes 32 q .. 32 q + 31 =====================
    uint32_t ui = 0;
    for (uint32_t u = blockIdx.x; u < n_units; u += gridDim.x, ++ui) {
      const uint32_t chunk = u / P.n_tiles, tile = u - chunk * P.n_tiles;
      const uint2 tc = P.tiles[tile];
      mbar_wait(bar_tfull, ui & 1);
      tc_fence_after();
#pragma unroll 1
      for (uint32_t half = 0; half < 2; ++half) {
        const uint64_t row = (uint64_t)tc.x * kGramM + half * kGramMmaM + warp * 32 + lane;
        int32_t* orow = P.compact ? P.out + ((size_t)tile * kGramM + half * kGramMmaM + warp * 32 + lane) * kGramN
                                  : P.out + row * P.ld + (uint64_t)tc.y * kGramN;
        const uint32_t taddr = tmem_base + half * kGramN + ((warp * 32) << 16);
#pragma unroll 1
        for (uint32_t c0 = 0; c0 < (uint32_t)kGramN; c0 += 32) {
          uint32_t v[32];
          asm volatile(
              "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
              : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
              : "r"(taddr + c0));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (P.n_chunks > 1) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (v[j]) atomicAdd(orow + c0 + j, (int32_t)v[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<uint4*>(orow + c0 + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_tempty);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
}

// Genome-major 2-bit codes from the sample-major planes: codes[g][w16] holds loci 16 w16 .. 16 w16 + 15 of genome g, code 3
// kept. One thread per (genome, 32-locus word) -> two output words.
__global__ void __launch_bounds__(256)
k_codes16(const uint32_t* __restrict__ sm_lo, const uint32_t* __restrict__ sm_hi, uint64_t n_gblocks, uint64_t n_words,
          uint64_t k_stages, uint64_t n_rows, uint32_t* __restrict__ codes /* zeroed */) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;     // ((gb * n_words) + w) * 32 + lane
  if (idx >= n_gblocks * n_words * 32) return;
  const uint64_t lane = idx & 31, w = (idx >> 5) % n_words, gb = (idx >> 5) / n_words;
  const uint32_t lo = sm_lo[idx], hi = sm_hi[idx];
  uint32_t out[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    uint32_t a = (lo >> (16 * h)) & 0xFFFFu, b = (hi >> (16 * h)) & 0xFFFFu;
    // spread 16 bits to even positions
    a = (a | (a << 8)) & 0x00FF00FFu; a = (a | (a << 4)) & 0x0F0F0F0Fu; a = (a | (a << 2)) & 0x33333333u; a = (a | (a << 1)) & 0x55555555u;
    b = (b | (b << 8)) & 0x00FF00FFu; b = (b | (b << 4)) & 0x0F0F0F0Fu; b = (b | (b << 2)) & 0x33333333u; b = (b | (b << 1)) & 0x55555555u;
    out[h] = a | (b << 1);
  }
  const uint64_t row = gb * 32 + lane;
  if (row >= n_rows || w * 2 + 1 >= k_stages * 8) return;
  codes[gram_code_index(row, w * 2, k_stages)] = out[0];
  codes[gram_code_index(row, w * 2 + 1, k_stages)] = out[1];
}

// ---- rank-one terms of the centred matrix -----------------------------------------------------------------------------------
// a[g] = sum_l p_l g_gl over the non-reference cells of genome g (lane per genome on the sample-major planes, the chunk's
// frequencies in shared memory), in chunks of 2,048 loci that are then added in a fixed order.
constexpr int kDotWords = 64;
__global__ void __launch_bounds__(256)
k_dosage_dot(const uint32_t* __restrict__ sm_lo, const uint32_t* __restrict__ sm_hi, uint64_t n_gblocks, uint64_t n_words, uint64_t n_loci,
             const float* __restrict__ af_pop, double* __restrict__ chunk_out /* [n_chunks][n_gblocks * 32] */) {
  __shared__ double s_p[kDotWords * 32];
  const uint64_t w0 = (uint64_t)blockIdx.y * kDotWords;
  for (int i = threadIdx.x; i < kDotWords * 32; i += 256) {
    const uint64_t l = w0 * 32 + i;
    double p = 0.0;
    if (l < n_loci) { const float a = af_pop[l]; if (a == a) { p = (double)a; p = p < 0.0 ? 0.0 : (p > 1.0 ? 1.0 : p); } }
    s_p[i] = p;
  }
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t gb = (uint64_t)blockIdx.x * 8 + warp;
  if (gb >= n_gblocks) return;
  double het = 0.0, hom = 0.0;
  const uint64_t w1 = min(w0 + (uint64_t)kDotWords, n_words);
  for (uint64_t w = w0; w < w1; ++w) {
    const uint64_t o = (gb * n_words + w) * 32 + lane;
    const uint32_t lo = sm_lo[o], hi = sm_hi[o], both = lo & hi;
    uint32_t a = lo & ~both, b = hi & ~both;
    const double* pw = s_p + (w - w0) * 32;
    while (a) { const int i = __ffs(a) - 1; a &= a - 1; het += pw[i]; }
    while (b) { const int i = __ffs(b) - 1; b &= b - 1; hom += pw[i]; }
  }
  chunk_out[(uint64_t)blockIdx.y * n_gblocks * 32 + gb * 32 + lane] = het + 2.0 * hom;
}

// gp[g] = sum of the chunks in order; gp[n_rows] = sum_l p_l^2 (block n_blocks - 1, fixed-order tree).
__global__ void __launch_bounds__(256)
k_dosage_reduce(const double* __restrict__ chunk_out, uint64_t n_chunks, uint64_t n_rows, const float* __restrict__ af_pop, uint64_t n_loci,
                double* __restrict__ gp) {
  if (blockIdx.x == gridDim.x - 1) {
    __shared__ double s[256];
    double v = 0.0;
    for (uint64_t l = threadIdx.x; l < n_loci; l += 256) {
      const float a = af_pop[l];
      if (a == a) { double p = (double)a; p = p < 0.0 ? 0.0 : (p > 1.0 ? 1.0 : p); v += p * p; }
    }
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if ((int)threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) gp[n_rows] = s[0];
    return;
  }
  const uint64_t g = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (g >= n_rows) return;
  double v = 0.0;
  for (uint64_t c = 0; c < n_chunks; ++c) v += chunk_out[c * n_rows + g];
  gp[g] = v;
}

// Upper-triangle tiles -> the caller's symmetric [n][n] matrix: int32 Gram matrix, or the centred double matrix
// S - 2 (a_i + a_j) + 4 sum p^2.
__global__ void __launch_bounds__(256)
k_gram_finalize(const int32_t* __restrict__ gram, uint64_t ld, uint64_t n, const double* __restrict__ gp /* null: integer output */,
                uint64_t gp_rows, void* __restrict__ out) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * n) return;
  const uint64_t i = idx / n, j = idx % n;
  const int32_t s = i <= j ? gram[i * ld + j] : gram[j * ld + i];
  if (gp == nullptr) static_cast<int32_t*>(out)[idx] = s;
  else static_cast<double*>(out)[idx] = ((double)s - 2.0 * (gp[i] + gp[j])) + 4.0 * gp[gp_rows];
}

}  // namespace kgl
