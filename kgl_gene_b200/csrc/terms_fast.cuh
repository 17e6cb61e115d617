// terms_fast.cuh -- the estimator sweeps behind the streaming pass (RitlandLocus / HallME / log-likelihood root search)
// as table-driven kernels over an interleaved 2-bit copy of the sample-major planes. Bound: the FP64 pipe.
//
// Every term of processRitlandLocus (calc.cpp:390-423), processHallME (calc.cpp:260-283) and d/df logLikelihood
// (calc.cpp:94-129) depends on the cell's genotype code, on per-(population, locus) constants and -- for the iterative
// estimators -- on the genome's current f. A CTA (one per SM) walks a contiguous range of 256-locus tiles. Per tile it builds
// a table {population, locus, code} -> constant in shared memory (the IEEE divides live here, once per locus instead of
// once per cell), then its warps sweep all genome blocks over the tile: lane = genome, one 64-bit code word (32 loci) per
// step. A cell costs one shift + one LOP3 (table address = base | code * 8, the locus goes into the load's immediate), one
// LDS.64 and the arithmetic below; cells that do not count (locus not selected for the population, rare major allele,
// heterozygous or dropped code, ...) read a neutral entry (1e300 -> reciprocal 1e-300, absorbed by the sums), so the inner
// loop has no predicate at all.
//
//   HALL    f/(f + (1-f) a) = 1/(1 + a k), k = (1-f)/f per genome    3.5 FP64 instructions per cell
//   NEWTON  t = (1-a)/(a + f (1-a)) = 1/(f + r), r = a/(1-a)         5 per cell (sum t, sum t^2)
//           two cells share one reciprocal (MUFU.RCP64H + 2 DFMA): fast_cell2
//   LIMITS  (once per root search) per genome: the left end of its feasible region fmin = max over homozygous cells of
//           (1e-10 - a^2)/(a (1-a))  [prob = a^2 + f a (1-a) >= small_prob, calc.cpp:108-110] and the smallest 2 a a2 over its
//           heterozygous cells -- so the Newton sweep needs no per-cell clamp test: a genome left of fmin is "clamped"
//           (k_ll_step only moves right then); a genome whose heterozygous terms could clamp, or that sits within rounding
//           of fmin, is re-evaluated cell by cell by k_genome_terms<TERM_NEWTON> (sample_major.cuh; normally no genome).
//   RITLAND sum over cells of v[locus][code], v = (1/p - 1)[hom-alt, p > 0.001] - (1/q - 1)[non-reference, q > 0.01]: one
//           DADD per cell; the hom-alt cells of p <= 0.001 loci are counted with a mask and POPC per word.
// Late Newton sweeps gather only the genomes that are still searching (FastParams::list).
// Measured on 2,504 x 1.1 M (B200): HALL 1.06 ms, NEWTON 1.27 ms per sweep = 56 / 65 % of the measured FP64 issue rate (ncu:
// profiles/r01_terms_fast_{hall,newton}_ncu_*); the cell-by-cell kernels they replace took 6.6 / 8.3 ms.
#pragma once
#include "common.cuh"

namespace kgl {

// FAST_NEWTON_U: unphased populations (Q6). A hom-alt pair is a heterozygous term 2 (1-f) p p there, which -- unlike 2 p q --
// can exceed 1 and is then clamped (calc.cpp:124): the sweep also counts, per genome, the code-2 cells with 2 p p (1-f) > 1.
enum { FAST_RITLAND = 0, FAST_HALL = 1, FAST_NEWTON = 2, FAST_LIMITS = 3, FAST_NEWTON_U = 4 };
constexpr int kFastMaxWarps = 24;                    // CTA = 16, 20 or 24 warps (the count that wastes the fewest genome-block slots)
constexpr int kFastBodyWords = 4;                    // words of the unrolled inner body
constexpr int kFastTileWords = 8;                    // words per table tile (two bodies)
constexpr int kFastTile = kFastTileWords * 32;       // loci per table tile
constexpr double kHuge = 1e300;                      // LIMITS: +-infinity stand-in
constexpr double kNeutral = 1e150;                   // NEWTON: r of a cell that does not count (the product of two stays finite)
constexpr double kHallHuge = 1e60;                   // HALL: a of a cell that does not count, and the cap of |(1-f)/f|

// Table entry of one (population, locus, genotype code): E doubles. Rows are padded so that consecutive populations start
// 8 (E = 1) / 16 (E = 2) banks apart.
__host__ __device__ constexpr int fast_entry(int mode) { return (mode == FAST_LIMITS || mode == FAST_NEWTON_U) ? 2 : 1; }
__host__ __device__ constexpr int fast_n_acc(int mode) { return mode == FAST_HALL ? 1 : mode == FAST_NEWTON_U ? 3 : 2; }
__host__ __device__ constexpr int fast_stride(int mode) { return (kFastTile * 4 + 4) * fast_entry(mode); }   // doubles per population row
template <int MODE> struct FastAcc { static constexpr int N = fast_n_acc(MODE); };

struct FastParams {
  const uint2* codes;          // [n_gblocks][n_words][32] interleaved 2-bit codes (k_to_sample_codes)
  uint64_t n_gblocks, n_words, n_loci, n_genomes, n_genomes_padded;
  const uint32_t* selw;        // [n_pop][n_words] selected & valid
  const float* af;             // [n_pop][n_loci]
  const uint8_t* superpop;     // [n_genomes]
  int n_pop, unphased;
  uint64_t tile_begin, tile_end;   // tiles that can hold a selected locus (the window of the last select_loci); others are skipped
  uint32_t tiles_per_chunk;    // grid.x chunks of this many tiles
  uint32_t slots;              // genome blocks per warp; grid.y = ceil(n_gblocks / (warps per CTA * slots))
  const double* f;             // [n_genomes_padded] current iterate (HALL / NEWTON)
  double* out;                 // [n_chunks][n_genomes_padded][FastAcc::N]
  // Late Newton sweeps: only the genomes still searching, gathered through a list. Lane i of compact block b works on genome
  // list[32 b + i]; n_gblocks counts compact blocks and out is indexed by the compact position. Null: every genome.
  const uint32_t* list; uint64_t n_list;
  const uint32_t* n_list_dev;  // when set: the list's current length on the device (<= n_list, which sized the grid)
  // HALL / NEWTON sweeps after the first: the two per-locus constants {hom-ref entry, hom-alt entry} of every population,
  // computed once per estimator run by k_terms_table instead of once per tile and CTA ([n_pop][n_words * 32]). Null: the tile
  // build computes them (single-sweep modes).
  const double2* table;
};

// Interleaved code copy of the sample-major planes: word (gb, w, lane) -> {cells 0..15, cells 16..31}, cell i of a half at
// bits 2i (lo plane) and 2i+1 (hi plane), so that one shift and one mask turn a cell into a table offset.
__device__ __forceinline__ uint32_t spread16(uint32_t x) {
  x &= 0xFFFFu;
  x = (x | (x << 8)) & 0x00FF00FFu;
  x = (x | (x << 4)) & 0x0F0F0F0Fu;
  x = (x | (x << 2)) & 0x33333333u;
  x = (x | (x << 1)) & 0x55555555u;
  return x;
}
__global__ void __launch_bounds__(256)
k_to_sample_codes(const uint32_t* __restrict__ sm_lo, const uint32_t* __restrict__ sm_hi, uint64_t n, uint2* __restrict__ codes) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t lo = sm_lo[i], hi = sm_hi[i];
  codes[i] = make_uint2(spread16(lo) | (spread16(hi) << 1), spread16(lo >> 16) | (spread16(hi >> 16) << 1));
}

// 1/d without the IEEE divide: x0 = MUFU.RCP64H, one Newton step x = x0 (1 + e), e = 1 - d x0. Measured on the B200
// (tools/kbench, 2^26 arguments over [2^-40, 2^40]): max relative error of x0 9.9e-7 (2^-19.9), of x 9.9e-13; a second-order
// step x0 (1 + e + e^2) reaches 2.2e-16 for one more DFMA per cell. The estimators' contract is 1e-6
// relative on F; a 1e-12 relative error in every term moves the HallME fixed point and the likelihood root by < 1e-12.
__device__ __forceinline__ double fast_rcp(double d) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  const double e = fma(-d, x, 1.0);
  return fma(x, e, x);
}

// Shared-memory address of cell j (0..15) of a code half z: base | (code * 8 E), the locus offset goes into the load's
// immediate. One shift and one LOP3 per cell.
template <int E, int J>
__device__ __forceinline__ uint32_t cell_addr(uint32_t z, uint32_t base) {
  constexpr int kShift = (E == 1) ? 3 : 4;              // log2(entry bytes)
  constexpr uint32_t kMask = 3u << kShift;
  const uint32_t y = (2 * J >= kShift) ? (z >> (2 * J - kShift)) : (z << (kShift - 2 * J));
  uint32_t a;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(a) : "r"(y), "r"(kMask), "r"(base));
  return a;
}

template <int E, int OFF>
__device__ __forceinline__ void lds_entry(uint32_t addr, double& v0, double& v1) {
  if (E == 1) { asm("ld.shared.f64 %0, [%1+%2];" : "=d"(v0) : "r"(addr), "n"(OFF)); v1 = 0.0; }
  else asm("ld.shared.v2.f64 {%0, %1}, [%2+%3];" : "=d"(v0), "=d"(v1) : "r"(addr), "n"(OFF));
}

// Two cells (loci J, J+1 of a code half) per step. The iterative modes share ONE reciprocal between the two denominators:
//   1/d1 + 1/d2 = (d1 + d2) x,  1/d1^2 + 1/d2^2 = ((d1 + d2) x)^2 - 2 x,  x = 1/(d1 d2)
// which halves the MUFU traffic and, for HALL, takes the FP64 instructions per cell from 4 to 3.5. A neutral entry (1e150 /
// 1e60) paired with a real one contributes (d1 + 1e150)/(d1 1e150) = 1/d1 to within 1e-150; two neutral entries give 2e-150.
template <int MODE, int TW, int HALF, int J>
__device__ __forceinline__ void fast_cell2(uint32_t z, uint32_t base, double f, double upper, double (&acc)[FastAcc<MODE>::N]) {
  constexpr int E = fast_entry(MODE);
  constexpr int kOff = (TW * 32 + HALF * 16 + J) * 4 * E * 8;      // byte offset of locus J inside the body's part of the row
  const uint32_t a1 = cell_addr<E, J>(z, base), a2 = cell_addr<E, J + 1>(z, base);
  double v0, v1, w0, w1;
  lds_entry<E, kOff>(a1, v0, v1);
  lds_entry<E, kOff + 4 * E * 8>(a2, w0, w1);
  if (MODE == FAST_HALL) {
    const double d1 = fma(v0, f, 1.0), d2 = fma(w0, f, 1.0);        // f here is (1-f)/f: f/(f + (1-f) a) = 1/(1 + a (1-f)/f)
    const double x = fast_rcp(__dmul_rn(d1, d2));
    acc[0] = fma(__dadd_rn(d1, d2), x, acc[0]);
  } else if (MODE == FAST_NEWTON || MODE == FAST_NEWTON_U) {
    const double d1 = __dadd_rn(f, v0), d2 = __dadd_rn(f, w0);      // t = 1/(f + r)
    const double x = fast_rcp(__dmul_rn(d1, d2));
    const double u = __dmul_rn(__dadd_rn(d1, d2), x);               // t1 + t2
    acc[0] = __dadd_rn(acc[0], u);
    acc[1] = fma(-2.0, x, fma(u, u, acc[1]));                       // t1^2 + t2^2 = (t1 + t2)^2 - 2 t1 t2
    if (MODE == FAST_NEWTON_U) {
      if (v1 > upper) acc[2] = __dadd_rn(acc[2], 1.0);
      if (w1 > upper) acc[2] = __dadd_rn(acc[2], 1.0);
    }
  } else if (MODE == FAST_LIMITS) {
    acc[0] = fmax(acc[0], fmax(v0, w0)); acc[1] = fmin(acc[1], fmin(v1, w1));
  } else {  // FAST_RITLAND
    acc[0] = __dadd_rn(acc[0], __dadd_rn(v0, w0));
  }
}

template <int MODE, int TW, int HALF, int J>
struct FastHalf {
  static __device__ __forceinline__ void run(uint32_t z, uint32_t base, double f, double upper, double (&acc)[FastAcc<MODE>::N]) {
    fast_cell2<MODE, TW, HALF, J>(z, base, f, upper, acc);
    FastHalf<MODE, TW, HALF, J + 2>::run(z, base, f, upper, acc);
  }
};
template <int MODE, int TW, int HALF>
struct FastHalf<MODE, TW, HALF, 16> {
  static __device__ __forceinline__ void run(uint32_t, uint32_t, double, double, double (&)[FastAcc<MODE>::N]) {}
};
template <int MODE, int TW>
__device__ __forceinline__ void fast_word(uint2 z, uint32_t base, double f, double upper, double (&acc)[FastAcc<MODE>::N]) {
  FastHalf<MODE, TW, 0, 0>::run(z.x, base, f, upper, acc);
  FastHalf<MODE, TW, 1, 0>::run(z.y, base, f, upper, acc);
}

// The two table constants of one (population, locus) for the single-value modes: {entry of code 0, entry of code 2}.
template <int MODE>
__device__ __forceinline__ double2 fast_constants(bool sel, double p, double q, bool unphased) {
  const bool ref_in = sel && q > kMinMajorFreq;          // the hom-ref cell counts (freq.cpp:532)
  const bool alt_in = sel && !unphased;                  // the hom-alt cell is MINOR_HOMOZYGOUS (phased populations)
  if (MODE == FAST_HALL) {
    // a; a cell that does not count, or whose denominator would be zero at every f (a = 0, calc.cpp:268), gets 1e60: its
    // term vanishes in the sum
    return make_double2((ref_in && q > 0.0) ? q : kHallHuge, (alt_in && p > 0.0) ? p : kHallHuge);
  }
  const double uq = __dsub_rn(1.0, q), up = __dsub_rn(1.0, p);      // NEWTON: r = a / (1 - a)
  return make_double2((ref_in && uq > 0.0) ? __ddiv_rn(q, uq) : kNeutral, (alt_in && up > 0.0) ? __ddiv_rn(p, up) : kNeutral);
}

template <int MODE>
__global__ void __launch_bounds__(256)
k_terms_table(const uint32_t* __restrict__ selw, const float* __restrict__ af, uint64_t n_loci, uint64_t n_words, int n_pop,
              int unphased, double2* __restrict__ table) {
  const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int kk = blockIdx.y;
  if (l >= n_words * 32 || kk >= n_pop) return;
  const bool sel = l < n_loci && ((selw[(uint64_t)kk * n_words + (l >> 5)] >> (l & 31)) & 1u);
  double p = 0.0, q = 1.0;
  if (sel) { const LocusFreq lf = locus_freq(af[(uint64_t)kk * n_loci + l]); p = lf.p; q = lf.q; }
  table[(uint64_t)kk * n_words * 32 + l] = fast_constants<MODE>(sel, p, q, unphased != 0);
}

template <int MODE>
__global__ void __launch_bounds__(kFastMaxWarps * 32, 1)
k_terms_fast(const FastParams P) {
  constexpr int NACC = FastAcc<MODE>::N, E = fast_entry(MODE), STRIDE = fast_stride(MODE);
  static_assert(kFastBodyWords == 4 && kFastTileWords % kFastBodyWords == 0, "one fast_word per word of the body");
  extern __shared__ __align__(128) unsigned char fast_smem[];
  const int n_warps = blockDim.x >> 5, n_thr = blockDim.x;
  double* tab = reinterpret_cast<double*>(fast_smem);                   // [kMaxPop][STRIDE]: (locus, code, E)
  double* s_acc = tab + kMaxPop * STRIDE;                               // [slots][NACC][n_thr]
  uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_acc + (size_t)P.slots * NACC * n_thr);   // RITLAND: [kMaxPop][kFastTileWords][2]

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint64_t gb_first = (uint64_t)blockIdx.y * n_warps * P.slots + warp;      // this warp's genome blocks: gb_first + s * n_warps
  const uint32_t my_slots = gb_first >= P.n_gblocks ? 0u
      : (uint32_t)min((uint64_t)P.slots, (P.n_gblocks - gb_first + n_warps - 1) / n_warps);
  const uint64_t t_begin = P.tile_begin + (uint64_t)blockIdx.x * P.tiles_per_chunk;
  const uint64_t t_end = min(t_begin + (uint64_t)P.tiles_per_chunk, P.tile_end);
  const double init0 = (MODE == FAST_LIMITS) ? -kHuge : 0.0, init1 = (MODE == FAST_LIMITS) ? kHuge : 0.0;

  for (uint32_t s = 0; s < P.slots; ++s)
#pragma unroll
    for (int j = 0; j < NACC; ++j) s_acc[(s * NACC + j) * n_thr + threadIdx.x] = (j == 0) ? init0 : (j == 1) ? init1 : 0.0;

  // The codes of the next (tile, body, genome block) are requested before the current ones are worked on.
  constexpr uint64_t kNoGenome = ~0ull;
  const uint64_t n_list = (P.list && P.n_list_dev) ? min(P.n_list, (uint64_t)*P.n_list_dev) : P.n_list;
  if (P.list && n_list == 0) return;                                      // every genome has finished: nothing to sweep
  auto genome_of = [&](uint32_t s) -> uint64_t {                          // the lane's genome in slot s
    const uint64_t pos = (gb_first + (uint64_t)s * n_warps) * 32 + lane;
    if (!P.list) return pos;
    return pos < n_list ? (uint64_t)P.list[pos] : kNoGenome;
  };
  auto load_codes = [&](uint64_t t, int body, uint32_t s, uint2 (&z)[kFastBodyWords]) {
    const uint64_t g = genome_of(s);
#pragma unroll
    for (int tw = 0; tw < kFastBodyWords; ++tw) {
      const uint64_t w = t * kFastTileWords + body * kFastBodyWords + tw;
      z[tw] = (w < P.n_words && g != kNoGenome) ? __ldg(P.codes + ((g >> 5) * P.n_words + w) * 32 + (g & 31))
                                                : make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);
    }
  };
  uint2 zn[kFastBodyWords];
  if (my_slots && t_begin < t_end) load_codes(t_begin, 0, 0, zn);

  for (uint64_t t = t_begin; t < t_end; ++t) {
    __syncthreads();
    // ---- constants of the tile: one (population, locus) per thread step, four codes each ----
    for (int idx = threadIdx.x; idx < P.n_pop * kFastTile; idx += n_thr) {
      const int kk = idx / kFastTile, j = idx % kFastTile;
      const uint64_t w = t * kFastTileWords + (j >> 5);
      const uint64_t l = t * kFastTile + j;
      if ((MODE == FAST_HALL || MODE == FAST_NEWTON) && P.table) {            // constants from the per-run table
        const double neutral = (MODE == FAST_HALL) ? kHallHuge : kNeutral;
        const double2 v = w < P.n_words ? P.table[(uint64_t)kk * P.n_words * 32 + l] : make_double2(neutral, neutral);
        double* e = tab + kk * STRIDE + j * 4;
        e[0] = v.x; e[1] = neutral; e[2] = v.y; e[3] = neutral;
        continue;
      }
      const bool sel = w < P.n_words && l < P.n_loci && ((P.selw[(uint64_t)kk * P.n_words + w] >> (j & 31)) & 1u);
      double p = 0.0, q = 1.0;
      if (sel) { const LocusFreq lf = locus_freq(P.af[(uint64_t)kk * P.n_loci + l]); p = lf.p; q = lf.q; }
      const bool ref_in = sel && q > kMinMajorFreq;          // the hom-ref cell counts (freq.cpp:532)
      const bool alt_in = sel && !P.unphased;                 // the hom-alt cell is MINOR_HOMOZYGOUS (phased populations)
      double* e = tab + kk * STRIDE + j * 4 * E;             // e[code * E + k]
      if (MODE == FAST_NEWTON || MODE == FAST_NEWTON_U) {
        const double2 v = fast_constants<FAST_NEWTON>(sel, p, q, P.unphased != 0);
        e[0 * E] = v.x; e[1 * E] = kNeutral; e[2 * E] = v.y; e[3 * E] = kNeutral;
        if (MODE == FAST_NEWTON_U) { e[1] = 0.0; e[3] = 0.0; e[5] = sel ? __dmul_rn(__dmul_rn(2.0, p), p) : 0.0; e[7] = 0.0; }
      } else if (MODE == FAST_HALL) {
        const double2 v = fast_constants<FAST_HALL>(sel, p, q, P.unphased != 0);
        e[0] = v.x; e[1] = kHallHuge; e[2] = v.y; e[3] = kHallHuge;
      } else if (MODE == FAST_LIMITS) {
        // {left end of the feasible region of a homozygous cell, 2 a a2 of a heterozygous cell}
        const double uq = __dsub_rn(1.0, q), up = __dsub_rn(1.0, p);
        const double dq = __dmul_rn(q, uq), dp = __dmul_rn(p, up);
        e[0] = !ref_in ? -kHuge : (dq > 0.0 ? __ddiv_rn(__dsub_rn(kSmallProb, __dmul_rn(q, q)), dq) : (q == 0.0 ? kHuge : -kHuge));
        e[1] = kHuge;
        e[2] = -kHuge; e[3] = sel ? __dmul_rn(__dmul_rn(2.0, p), q) : kHuge;                       // code 1: 2 p q
        e[4] = !alt_in ? -kHuge : (dp > 0.0 ? __ddiv_rn(__dsub_rn(kSmallProb, __dmul_rn(p, p)), dp) : (p == 0.0 ? kHuge : -kHuge));
        e[5] = (sel && P.unphased) ? __dmul_rn(__dmul_rn(2.0, p), p) : kHuge;                      // unphased hom-alt pair: 2 p p (Q6)
        e[6] = -kHuge; e[7] = kHuge;
      } else {  // FAST_RITLAND: (1/p - 1)[hom-alt, p > 0.001] - (1/q - 1)[non-reference cell, q > 0.01]
        const double c0 = ref_in ? __dsub_rn(__ddiv_rn(1.0, q), 1.0) : 0.0;
        const double c2 = (alt_in && p > kRitlandMinFreq) ? __dsub_rn(__ddiv_rn(1.0, p), 1.0) : 0.0;
        e[0] = 0.0; e[1] = -c0; e[2] = __dsub_rn(c2, c0); e[3] = -c0;
        // loci whose hom-alt cells are skipped (p <= 0.001, calc.cpp:397): a mask in the layout of the code words
        const uint32_t skip = __ballot_sync(kFull, alt_in && !(p > kRitlandMinFreq));
        if (lane == 0) {
          s_mask[(kk * kFastTileWords + (j >> 5)) * 2 + 0] = spread16(skip);
          s_mask[(kk * kFastTileWords + (j >> 5)) * 2 + 1] = spread16(skip >> 16);
        }
      }
    }
    __syncthreads();

    for (int body = 0; body < kFastTileWords / kFastBodyWords; ++body) {
      for (uint32_t s = 0; s < my_slots; ++s) {
        const uint64_t g = genome_of(s);
        const int k = (g < P.n_genomes) ? P.superpop[g] : 0;
        double f = ((MODE == FAST_HALL || MODE == FAST_NEWTON || MODE == FAST_NEWTON_U) && g != kNoGenome) ? P.f[g] : 0.0;
        const double upper = (MODE == FAST_NEWTON_U) ? __ddiv_rn(1.0, __dsub_rn(1.0, f)) : 0.0;   // 2 p p (1-f) > 1  <=>  2 p p > 1/(1-f)
        if (MODE == FAST_HALL) {                 // k = (1-f)/f. f = 0: every term vanishes; f = 1: k = 0 would turn the neutral entries (a = 1e60)
          f = fmin(fmax(__ddiv_rn(__dsub_rn(1.0, f), f), -kHallHuge), kHallHuge);   // into terms, so k stays >= 1e-30 (a real term moves by < 1e-30)
          if (f >= 0.0 && f < 1e-30) f = 1e-30;
        }
        const uint32_t base = (uint32_t)__cvta_generic_to_shared(tab + k * STRIDE + body * kFastBodyWords * 32 * 4 * E);
        uint2 z[kFastBodyWords];
#pragma unroll
        for (int tw = 0; tw < kFastBodyWords; ++tw) z[tw] = zn[tw];
        {   // next item: next genome block of this body, else the next body / tile
          uint32_t ns = s + 1; int nb = body; uint64_t nt = t;
          if (ns == my_slots) { ns = 0; if (++nb == kFastTileWords / kFastBodyWords) { nb = 0; ++nt; } }
          if (nt < t_end) load_codes(nt, nb, ns, zn);
        }
        double acc[NACC];
#pragma unroll
        for (int j = 0; j < NACC; ++j) acc[j] = (j == 0) ? init0 : (j == 1) ? init1 : 0.0;
        fast_word<MODE, 0>(z[0], base, f, upper, acc);
        fast_word<MODE, 1>(z[1], base, f, upper, acc);
        fast_word<MODE, 2>(z[2], base, f, upper, acc);
        fast_word<MODE, 3>(z[3], base, f, upper, acc);
        if (MODE == FAST_RITLAND) {
          int cnt = 0;
#pragma unroll
          for (int tw = 0; tw < kFastBodyWords; ++tw) {
            const uint32_t* m = s_mask + (k * kFastTileWords + body * kFastBodyWords + tw) * 2;
            cnt += __popc((z[tw].x >> 1) & ~z[tw].x & m[0]) + __popc((z[tw].y >> 1) & ~z[tw].y & m[1]);   // code 2: hi set, lo clear
          }
          acc[1] = (double)cnt;
        }
#pragma unroll
        for (int j = 0; j < NACC; ++j) {
          double* sa = s_acc + (s * NACC + j) * n_thr + threadIdx.x;
          if (MODE == FAST_LIMITS && j == 0) *sa = fmax(*sa, acc[j]);
          else if (MODE == FAST_LIMITS && j == 1) *sa = fmin(*sa, acc[j]);
          else *sa = __dadd_rn(*sa, acc[j]);
        }
      }
    }
  }

  for (uint32_t s = 0; s < my_slots; ++s) {
    const uint64_t pos = (gb_first + (uint64_t)s * n_warps) * 32 + lane;
    double* out = P.out + ((uint64_t)blockIdx.x * P.n_genomes_padded + pos) * NACC;
#pragma unroll
    for (int j = 0; j < NACC; ++j) out[j] = s_acc[(s * NACC + j) * n_thr + threadIdx.x];
  }
}

// Sum of one genome's chunk outputs by the eight lanes that share it (lane8 = threadIdx.x & 7): lane8 adds the chunks
// c = lane8, lane8 + 8, ... and a three-step butterfly combines the eight partial sums -- a fixed order, 18 dependent loads
// instead of 144 at C2. Every lane of the warp must call it; all eight lanes return the total.
template <int NOUT>
__device__ __forceinline__ void chunk_sum8(const double* __restrict__ chunk_out, uint64_t n_chunks, uint64_t n_genomes_padded,
                                           uint64_t pos, bool live, double (&sum)[NOUT]) {
  const int lane8 = threadIdx.x & 7;
#pragma unroll
  for (int j = 0; j < NOUT; ++j) sum[j] = 0.0;
  if (live)
    for (uint64_t c = lane8; c < n_chunks; c += 8) {
      const double* o = chunk_out + (c * n_genomes_padded + pos) * NOUT;
#pragma unroll
      for (int j = 0; j < NOUT; ++j) sum[j] += o[j];
    }
#pragma unroll
  for (int j = 0; j < NOUT; ++j)
#pragma unroll
    for (int m = 1; m < 8; m <<= 1) sum[j] += __shfl_xor_sync(kFull, sum[j], m);
}

// ---- reductions over the locus chunks --------------------------------------------------------------------------------
// limits[g] = {fmin, cmin, n_het}; n_het (heterozygous cells of this locus shard) is stashed from the phase-0 partials
// before they are all-reduced (k_stash_nhet).
__global__ void __launch_bounds__(256)
k_limits_reduce(const double* __restrict__ chunk_out, uint64_t n_chunks, uint64_t n_genomes_padded, uint64_t n_genomes,
                double* __restrict__ limits) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  double fmin_ = -kHuge, cmin = kHuge;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    const double* o = chunk_out + (c * n_genomes_padded + g) * 2;
    fmin_ = fmax(fmin_, o[0]); cmin = fmin(cmin, o[1]);
  }
  limits[g * 3 + 0] = fmin_; limits[g * 3 + 1] = cmin;
}

__global__ void __launch_bounds__(256)
k_stash_nhet(const double* __restrict__ partials, int part_count, int i_majhet, int i_minhet, uint64_t n_genomes, double* __restrict__ limits) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  limits[g * 3 + 2] = partials[g * part_count + i_majhet] + partials[g * part_count + i_minhet];
}

// Newton sweep: iter[g] = {dLL/df, d2LL/df2, clamped homozygous terms, clamped heterozygous terms} of this locus shard, as
// k_genome_terms<TERM_NEWTON> defines them. state[g]: 0 summed here, 1 left of the feasible region, 2 needs the exact
// cell-by-cell evaluation (n_slow counts them).
constexpr double kLimitMargin = 1e-9;
__global__ void __launch_bounds__(256)
k_newton_reduce(const double* __restrict__ chunk_out, int n_out /* 2, or 3 with the upper-clamped count */, uint64_t n_chunks,
                uint64_t n_genomes_padded, uint64_t n_genomes, const uint32_t* __restrict__ list, uint64_t n_list,
                const uint32_t* __restrict__ n_list_dev, const double* __restrict__ f, const double* __restrict__ limits, const uint32_t* __restrict__ done,
                double valid_min /* sums from the moment tables hold for f >= valid_min (terms_moments.cuh); -kHuge otherwise */,
                double* __restrict__ iter, uint8_t* __restrict__ state, uint32_t* __restrict__ n_slow) {
  const uint64_t pos = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3;       // position in chunk_out, eight lanes each
  if (list && n_list_dev) n_list = min(n_list, (uint64_t)*n_list_dev);
  const bool live = pos < (list ? n_list : n_genomes);
  double sums[3];
  if (n_out > 2) chunk_sum8<3>(chunk_out, n_chunks, n_genomes_padded, pos, live, sums);
  else { double s2[2]; chunk_sum8<2>(chunk_out, n_chunks, n_genomes_padded, pos, live, s2); sums[0] = s2[0]; sums[1] = s2[1]; sums[2] = 0.0; }
  if (!live || (threadIdx.x & 7) != 0) return;
  const uint64_t g = list ? list[pos] : pos;
  double* I = iter + g * 4;
  const double x = f[g], fmin_ = limits[g * 3 + 0], cmin = limits[g * 3 + 1], nhet = limits[g * 3 + 2];
  const double band = kLimitMargin * fmax(1.0, fabs(fmin_));
  uint8_t st = 0;
  if (done && done[g]) st = 1;                                  // converged genomes: values are not read any more
  else if (x < fmin_ - band) st = 1;
  else if (x < fmin_ + band || x < valid_min) st = 2;
  else if (nhet > 0.0 && !((1.0 - x) * cmin > kSmallProb * (1.0 + kLimitMargin))) st = 2;
  state[g] = st;
  if (st == 1) { I[0] = 0.0; I[1] = 0.0; I[2] = 1.0; I[3] = 0.0; return; }
  if (st == 2) { I[0] = I[1] = I[2] = I[3] = 0.0; atomicAdd(n_slow, 1u); return; }
  const double s1 = sums[0], s2 = sums[1], clamped_het = sums[2];
  const double t = 1.0 / (1.0 - x), n_terms = nhet - clamped_het;
  I[0] = s1 - n_terms * t;
  I[1] = -s2 - n_terms * t * t;
  I[2] = 0.0; I[3] = clamped_het;
}

// Ordered list of the genomes whose root search has not finished (one block; N is at most a few hundred thousand).
__global__ void __launch_bounds__(1024)
k_compact_active(const uint32_t* __restrict__ done, uint64_t n_genomes, uint32_t* __restrict__ list, uint32_t* __restrict__ count) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (uint64_t g0 = 0; g0 < n_genomes; g0 += 1024) {
    const uint64_t g = g0 + threadIdx.x;
    const bool active = g < n_genomes && !done[g];
    const uint32_t bal = __ballot_sync(kFull, active);
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    uint32_t before = s_base;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (active) list[before + __popc(bal & ((1u << lane) - 1u))] = (uint32_t)g;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < 32; ++w) t += s_warp[w]; s_base += t; }
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = s_base;
}

// Adds the exact evaluation of the state-2 genomes (chunk outputs of k_genome_terms<TERM_NEWTON>, 4 per genome).
__global__ void __launch_bounds__(256)
k_newton_add_slow(const double* __restrict__ chunk_out, uint64_t n_chunks, uint64_t n_genomes_padded, uint64_t n_genomes,
                  const uint8_t* __restrict__ state, const uint32_t* __restrict__ n_slow, double* __restrict__ iter) {
  if (*n_slow == 0) return;
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes || state[g] != 2) return;
  for (int j = 0; j < 4; ++j) {
    double s = 0.0;
    for (uint64_t c = 0; c < n_chunks; ++c) s += chunk_out[(c * n_genomes_padded + g) * 4 + j];
    iter[g * 4 + j] = s;
  }
}

// HallME: iter[g][0] = sum over homozygous cells of f/(f + (1-f) a). Eight lanes per genome.
__global__ void __launch_bounds__(256)
k_hall_reduce(const double* __restrict__ chunk_out, uint64_t n_chunks, uint64_t n_genomes_padded, uint64_t n_genomes,
              double* __restrict__ iter) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t g = t >> 3;
  double s[1];
  chunk_sum8<1>(chunk_out, n_chunks, n_genomes_padded, g, g < n_genomes, s);
  if (g < n_genomes && (threadIdx.x & 7) == 0) iter[g * 4] = s[0];
}

}  // namespace kgl
