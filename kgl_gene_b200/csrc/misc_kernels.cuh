// misc_kernels.cuh -- estimator finalisation, iterative updates and the synthetic generator.
#pragma once
#include "common.cuh"
#include "locus_kernels.cuh"
#include "../../include/kgl_b200.h"

namespace kgl {

// Per-genome partial sums that are additive over locus shards (multi-GPU all-reduce payload), doubles.
enum { PART_NMAJHOM = 0, PART_NMAJHET, PART_NMINHOM, PART_NMINHET,
       PART_EMAJHOM, PART_EMAJHET, PART_EMINHOM, PART_EMINHET,
       PART_RSUM, PART_RCOUNT,            // Ritland numerator / denominator
       PART_COUNT = 16 };
// Per-iteration payload of the iterative estimators (second all-reduce buffer): HallME uses slot 0, the likelihood
// root search slots 0..3 = {dLL, d2LL, clamped hom terms, clamped het terms}.
constexpr int ITER_COUNT = 4;

// Adds the Ritland terms (reduced over locus chunks) to the partials.
__global__ void __launch_bounds__(256)
k_ritland_partials(const double* __restrict__ chunk_out, uint64_t n_chunks, uint64_t n_genomes_padded, int n_out,
                   const DenseTotals totals, const uint8_t* __restrict__ superpop, uint64_t n_genomes,
                   double* __restrict__ partials) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  // chunk outputs of k_terms_fast<FAST_RITLAND>: {sum of (1/p - 1) over hom-alt cells with p > 0.001 minus sum of (1/q - 1)
  // over the non-reference cells of q > 0.01 rows, number of hom-alt cells with p <= 0.001}
  double sdiff = 0.0, c2x = 0.0;
  for (uint64_t c = 0; c < n_chunks; ++c) {
    const double* o = chunk_out + (c * n_genomes_padded + g) * n_out;
    sdiff += o[0]; c2x += o[1];
  }
  const int k = superpop[g];
  double* P = partials + g * PART_COUNT;
  const double n_het = P[PART_NMAJHET] + P[PART_NMINHET];
  P[PART_RSUM] = (totals.get(k, TOT_W0) + sdiff) - n_het;
  P[PART_RCOUNT] = P[PART_NMAJHOM] + (P[PART_NMINHOM] - c2x) + n_het;
}

__device__ __forceinline__ void fill_results(const double* P, kgl_b200_locus_results& r) {
  r.major_homo_count = (uint64_t)llrint(P[PART_NMAJHOM]);   r.major_homo_freq = P[PART_EMAJHOM];
  r.major_hetero_count = (uint64_t)llrint(P[PART_NMAJHET]); r.major_hetero_freq = P[PART_EMAJHET];
  r.minor_homo_count = (uint64_t)llrint(P[PART_NMINHOM]);   r.minor_homo_freq = P[PART_EMINHOM];
  r.minor_hetero_count = (uint64_t)llrint(P[PART_NMINHET]); r.minor_hetero_freq = P[PART_EMINHET];
  r.total_allele_count = r.major_homo_count + r.major_hetero_count + r.minor_homo_count + r.minor_hetero_count;
}

// processSimple (calc.cpp:333-359) / processRitlandLocus (calc.cpp:423) closed forms from the (all-reduced) partials.
__device__ __forceinline__ kgl_b200_locus_results closed_form(const double* P, int algorithm) {
  kgl_b200_locus_results r;
  fill_results(P, r);
  double coeff = 0.0;
  if (algorithm == KGL_B200_ALGO_RITLAND) {
    coeff = (P[PART_RCOUNT] > 0.0) ? P[PART_RSUM] / P[PART_RCOUNT] : 0.0;
  } else {
    if (r.total_allele_count > 0) {
      const double observed_homozygous = (double)(r.minor_homo_count + r.major_homo_count);
      const double expected_homozygous = r.minor_homo_freq + r.major_homo_freq;
      coeff = (observed_homozygous - expected_homozygous) / ((double)r.total_allele_count - expected_homozygous);
    }
  }
  r.inbred_allele_sum = coeff;
  return r;
}

__global__ void __launch_bounds__(256)
k_finalize_closed_form(const double* __restrict__ partials, uint64_t n_genomes, int algorithm,
                       kgl_b200_locus_results* __restrict__ out, double* __restrict__ f_out) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  const kgl_b200_locus_results r = closed_form(partials + g * PART_COUNT, algorithm);
  if (out) out[g] = r;
  if (f_out) f_out[g] = r.inbred_allele_sum;
}

// Moments of this locus shard from the fused pass: counts (vertical counters), dense totals and sparse corrections.
// n_lo / n_hi: set lo / hi bits of the genome over its selected rows; n3: code-3 cells among them; nzr: non-reference cells in
// rare-major rows; d_majhom / d_minhom: class frequencies of the genome's dropped loci (code-3 cells + hom-ref cells of
// rare-major rows).
__device__ __forceinline__ void moment_partials_from(uint64_t g, double n_lo, double n_hi, double n3, double nzr, double d_majhom,
                                                     double d_minhom, const DenseTotals& totals, int k, int unphased,
                                                     double* __restrict__ partials, kgl_b200_locus_results* __restrict__ simple_out) {
  double T[TOT_COUNT];
#pragma unroll
  for (int j = 0; j < TOT_W0; ++j) T[j] = totals.get(k, j);
  const double n1 = n_lo - n3, n2 = n_hi - n3;
  // hom-ref cells in q > 0.01 rows: all such rows minus the non-reference cells that sit in them
  const double n_majhom = T[TOT_TQ] - ((n1 + n2 + n3) - nzr);
  double P[PART_COUNT];
  P[PART_NMAJHOM] = n_majhom;
  P[PART_NMAJHET] = n1;
  P[PART_NMINHOM] = unphased ? 0.0 : n2;
  P[PART_NMINHET] = unphased ? n2 : 0.0;
  // dropped cells: code 3 in selected rows (n3) and hom-ref cells of rare-q rows; their class frequencies leave the sums.
  const double n_dropped = (T[TOT_T] - T[TOT_TQ]) - nzr + n3;
  P[PART_EMAJHOM] = T[TOT_EMAJHOM] - d_majhom;
  P[PART_EMINHOM] = T[TOT_EMINHOM] - d_minhom;
  // the three normalised class frequencies of a locus sum to 1, so the dropped majHet mass is n_dropped - majHom - minHom
  P[PART_EMAJHET] = T[TOT_EMAJHET] - (n_dropped - d_majhom - d_minhom);
  P[PART_EMINHET] = 0.0;
#pragma unroll
  for (int j = PART_RSUM; j < PART_COUNT; ++j) P[j] = 0.0;
  double2* dst = reinterpret_cast<double2*>(partials + g * PART_COUNT);
#pragma unroll
  for (int j = 0; j < PART_COUNT / 2; ++j) dst[j] = make_double2(P[2 * j], P[2 * j + 1]);
  if (simple_out) simple_out[g] = closed_form(P, KGL_B200_ALGO_SIMPLE);
}

// Fallback path (populations whose code-3 cells are not indexed): assembles the partials from the arrays the separate kernels
// left (k_sum_cta_counts, k_dropped_scan, k_locus_prepare).
__global__ void __launch_bounds__(256)
k_moment_partials(const uint32_t* __restrict__ gcounts /* [g]{set lo bits, set hi bits} over the selected rows */,
                  const uint32_t* __restrict__ n3s, const DenseTotals totals,
                  const unsigned long long* __restrict__ ecorr_scan_fx, const uint32_t* __restrict__ nz_rare,
                  const unsigned long long* __restrict__ ecorr_rare_fx, double fx_inv, const uint8_t* __restrict__ superpop,
                  uint64_t n_genomes, int unphased, double* __restrict__ partials,
                  kgl_b200_locus_results* __restrict__ simple_out /* nullable: also apply processSimple (calc.cpp:333-359) */) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  const double da = (double)(long long)(ecorr_scan_fx[g * 2 + 0] + ecorr_rare_fx[g * 2 + 0]) * fx_inv;
  const double dm = (double)(long long)(ecorr_scan_fx[g * 2 + 1] + ecorr_rare_fx[g * 2 + 1]) * fx_inv;
  moment_partials_from(g, (double)gcounts[g * 2], (double)gcounts[g * 2 + 1], (double)n3s[g], (double)nz_rare[g], da, dm, totals,
                       superpop[g], unphased, partials, simple_out);
}

// ---- locus-sharded exchange over NVLink peer memory (kgl_b200_enqueue_count_and_inbreed_peer) ------------------------------
// Every rank owns an exchange region [2 parities][n_genomes_padded][PART_COUNT] doubles + 64 flags, mapped into every peer
// (CUDA IPC). A step: the moment kernel of rank r writes its partials into parity (epoch & 1) of its own region;
// k_peer_exchange then (1) publishes `epoch` into flag[r] of every peer's region, (2) waits until its own flags of all
// ranks have reached `epoch`, (3) reads the partials of every rank straight from peer memory, adds them in rank order (the same
// order on every rank: bit-identical results everywhere) and applies the Simple closed form. One launch replaces
// all-reduce + finalize; there is no NCCL call on the step's path. Two parities suffice: a rank can be at most one step ahead
// of a peer, because its next exchange waits for that peer's next flag.
constexpr int kPeerMaxRanks = 64;
constexpr unsigned long long kPeerTimeoutNsDefault = 10ull * 1000 * 1000 * 1000;   // 10 s
struct PeerParams {
  unsigned char* base[kPeerMaxRanks];   // exchange regions, index = rank (own region included)
  uint32_t rank, world;
  uint64_t parity_doubles;              // n_genomes_padded * PART_COUNT
  uint64_t epoch;
  uint64_t n_genomes;
  unsigned long long timeout_ns;
  double* partials_out;                 // reduced partials (local copy, for inbreed_fetch-style consumers)
  kgl_b200_locus_results* results;
  unsigned int* error_word;             // set to 1 when a peer did not arrive in time; checked by the fetch entry points
};

__device__ __forceinline__ unsigned long long* peer_flags(unsigned char* base, uint64_t parity_doubles) {
  return reinterpret_cast<unsigned long long*>(base + 2 * parity_doubles * 8);
}

// Publishes this rank's epoch into every peer's region. A launch of its own, ahead of k_peer_exchange on the stream: the
// waiting blocks of k_peer_exchange then never depend on one of their own grid being scheduled first.
__global__ void __launch_bounds__(kPeerMaxRanks)
k_peer_publish(const PeerParams P) {
  if (threadIdx.x < P.world) {
    __threadfence_system();             // the moment kernel that preceded this launch has completed: its stores are in L2
    unsigned long long* f = peer_flags(P.base[threadIdx.x], P.parity_doubles) + P.rank;
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(f), "l"((unsigned long long)P.epoch) : "memory");
  }
}

// Grid: at most one resident wave (the host caps it); genomes are walked with a grid stride.
__global__ void __launch_bounds__(256)
k_peer_exchange(const PeerParams P) {
  __shared__ int s_timed_out;
  // (2) wait for every rank's flag in the local region. A peer that never arrives (its process died) must not hang the GPU:
  // after the timeout the step gives up, every result row of this rank becomes NaN / zero and the error word is set --
  // kgl_b200_inbreed_fetch / kgl_b200_fetch_locus_counts then fail with KGL_B200_ERR_PEER until the regions are exported and
  // attached again.
  if (threadIdx.x == 0) s_timed_out = 0;
  __syncthreads();
  if (threadIdx.x < P.world) {
    const unsigned long long* f = peer_flags(P.base[P.rank], P.parity_doubles) + threadIdx.x;
    unsigned long long v, t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    do {
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
      if (v < P.epoch) {
        __nanosleep(100);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > P.timeout_ns) { s_timed_out = 1; break; }
      }
    } while (v < P.epoch);
  }
  __syncthreads();
  const bool timed_out = s_timed_out != 0;
  if (timed_out && threadIdx.x == 0) atomicExch(P.error_word, 1u);
  // (3) gather + fixed-order sum + closed form. Eight lanes per genome, one pair of doubles each; the loads of up to eight
  // ranks are in flight together (an NVLink round trip is ~1.5 us: serialised they would cost more than the all-reduce).
  const uint64_t n_items = (P.n_genomes * 8 + 31) / 32 * 32;          // whole warps: every lane reaches the __syncwarp
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n_items; t += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t g = t >> 3;
    const int jp = (int)(t & 7);
    const bool live = g < P.n_genomes;
    double s0 = 0.0, s1 = 0.0;
    if (live) {
      if (!timed_out) {
        const uint64_t off = (P.epoch & 1ull) * P.parity_doubles + g * PART_COUNT + jp * 2;
        for (uint32_t r0 = 0; r0 < P.world; r0 += 8) {
          double a[8], b[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            a[i] = 0.0; b[i] = 0.0;
            if (r0 + i < P.world) {
              const double* src = reinterpret_cast<const double*>(P.base[r0 + i]) + off;
              asm volatile("ld.relaxed.sys.global.v2.f64 {%0, %1}, [%2];" : "=d"(a[i]), "=d"(b[i]) : "l"(src) : "memory");
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) if (r0 + i < P.world) { s0 += a[i]; s1 += b[i]; }    // rank order
        }
      }
      P.partials_out[g * PART_COUNT + jp * 2] = s0;
      P.partials_out[g * PART_COUNT + jp * 2 + 1] = s1;
    }
    __syncwarp();
    if (live && jp == 0) {
      double sum[PART_COUNT];
#pragma unroll
      for (int j = 0; j < PART_COUNT; ++j) sum[j] = __ldcg(P.partials_out + g * PART_COUNT + j);
      kgl_b200_locus_results r = closed_form(sum, KGL_B200_ALGO_SIMPLE);
      if (timed_out) {                   // the whole row: no count or sum of a step that did not complete is reported
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        r.major_hetero_freq = r.minor_hetero_freq = r.minor_homo_freq = r.major_homo_freq = r.inbred_allele_sum = nan;
      }
      P.results[g] = r;
    }
  }
}

// processHallME: f <- (1/n) * sum_hom f/(f+(1-f)a)   (calc.cpp:285). flag[0] = max |delta| bits (atomicMax on the ordered int).
__global__ void __launch_bounds__(256)
k_hall_update(const double* __restrict__ partials, const double* __restrict__ iter, uint64_t n_genomes, double* __restrict__ f,
              unsigned long long* __restrict__ flag) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  const double* P = partials + g * PART_COUNT;
  const double n = P[PART_NMAJHOM] + P[PART_NMAJHET] + P[PART_NMINHOM] + P[PART_NMINHET];
  // f == 0 is a fixed point (every term is 0/(0 + a), calc.cpp:268-272) and an unstable one: the sweeps must not leave it through
  // the 1e-60 the table kernel's neutral entries leave behind
  // A genome without any term is 0/0 in the reference (calc.cpp:285), not the 1e-60 / 0 the neutral entries would make of it.
  const double nf = n > 0.0 ? (f[g] == 0.0 ? 0.0 : __ddiv_rn(iter[g * ITER_COUNT], n)) : __ddiv_rn(0.0, n);
  const double delta = fabs(nf - f[g]);
  f[g] = nf;
  if (delta == delta) atomicMax(flag, (unsigned long long)__double_as_longlong(delta));   // non-negative doubles order like ints
}

// ---- log-likelihood maximiser (processLogLikelihood, calc.cpp:154-216) --------------------------------------------
// The reference maximises the clamped objective over [-1,1] with Nelder-Mead from random starts. The clamp at 1e-10 is a
// numerical guard: left of the largest pole of a homozygous term the objective has convex kinks and extra local maxima,
// and which one Nelder-Mead returns depends on its random start. The product returns the maximiser over the FEASIBLE
// region (no homozygous probability clamped), where the objective is smooth and concave -- this is what the reference
// returns for every genome of the golden fixtures (tests/test_oracle_vs_reference.py). Bracketed Newton on dLL/df:
// a clamped homozygous term means "left of the feasible region" (move right); otherwise the sign of dLL/df updates the
// bracket and the Newton step is taken when it stays inside it (else bisection). state: bracket a,b ; done flag.
__global__ void __launch_bounds__(256)
k_ll_init(const double* __restrict__ partials, uint64_t n_genomes, double* __restrict__ f, double* __restrict__ bracket,
          uint32_t* __restrict__ done) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  const double* P = partials + g * PART_COUNT;
  const double n = P[PART_NMAJHOM] + P[PART_NMAJHET] + P[PART_NMINHOM] + P[PART_NMINHET];
  double x = 0.0;                                        // start: the Simple estimate (calc.cpp:344)
  if (n > 0.0) {
    const double oh = P[PART_NMINHOM] + P[PART_NMAJHOM], eh = P[PART_EMINHOM] + P[PART_EMAJHOM];
    x = (oh - eh) / (n - eh);
  }
  if (!(x > -1.0 && x < 1.0)) x = 0.0;
  bracket[g * 2 + 0] = -1.0; bracket[g * 2 + 1] = 1.0;
  done[g] = (n <= 0.0) ? 1u : 0u;
  f[g] = (n <= 0.0) ? 0.0 : x;
}

__global__ void __launch_bounds__(256)
k_ll_step(const double* __restrict__ iter, uint64_t n_genomes, double tol, double* __restrict__ f,
          double* __restrict__ bracket, uint32_t* __restrict__ done, unsigned long long* __restrict__ flag) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  if (done[g]) return;
  const double* I = iter + g * ITER_COUNT;
  const double g1 = I[0], g2 = I[1];
  const bool hom_clamped = I[2] > 0.0;
  double a = bracket[g * 2 + 0], b = bracket[g * 2 + 1];
  const double x = f[g];
  if (hom_clamped || g1 > 0.0) a = x; else b = x;
  double nx = 0.5 * (a + b);
  bool newton_converged = false;
  if (!hom_clamped && g2 < 0.0) {
    const double cand = x - g1 / g2;
    // a Newton step below the tolerance ends the search even when rounding puts it on the bracket's edge (x itself is an
    // end of the bracket by now); without this test such a genome falls back to ~40 bisection passes over the matrix
    if (fabs(cand - x) < tol) { nx = (cand > a && cand < b) ? cand : x; newton_converged = true; }
    else if (cand > a && cand < b) nx = cand;
  }
  bracket[g * 2 + 0] = a; bracket[g * 2 + 1] = b;
  f[g] = nx;
  if (newton_converged || fabs(nx - x) < tol || (b - a) < tol) done[g] = 1;
  else atomicAdd(flag, 1ull);
}

__global__ void __launch_bounds__(256)
k_store_coeff(const double* __restrict__ partials, const double* __restrict__ f, uint64_t n_genomes,
              kgl_b200_locus_results* __restrict__ out) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  kgl_b200_locus_results r;
  fill_results(partials + g * PART_COUNT, r);
  r.inbred_allele_sum = f[g];
  out[g] = r;
}

__global__ void k_fill_double(double* p, uint64_t n, double v) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

__global__ void k_genome_counts_raw(const uint32_t* __restrict__ gcounts, const uint32_t* __restrict__ n3s, uint64_t n_genomes,
                                    uint64_t n_loci, uint64_t* __restrict__ out) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= n_genomes) return;
  const uint64_t n3 = n3s[g], n1 = gcounts[g * 2] - n3, n2 = gcounts[g * 2 + 1] - n3;
  out[g * 4 + 0] = n_loci - n1 - n2 - n3; out[g * 4 + 1] = n1; out[g * 4 + 2] = n2; out[g * 4 + 3] = n3;
}

// ---- AF-bin passes (CalcFWS, kga_PfEMP/kga_analysis_PfEMP_FWS.cpp:15-101) ------------------------------------------------
// Row mask of one bin: the P7FrequencyFilter pair AF >= lower and not AF >= upper (kgl_variant_filter_Pf7.cpp:20-66; a
// variant without the AF field passes both filters and is therefore in no bin); with locus_counts also "some genome
// carries the variant" (a filtered PopulationDB only holds variants that occur). One thread per row, one warp-pair per
// 64-row summary.
__global__ void __launch_bounds__(256)
k_bin_flags(const float* __restrict__ af_pop, const uint32_t* __restrict__ locus_counts /* nullable [L][4] */, uint64_t n_loci,
            uint64_t padded_rows, double lower, double upper, const uint8_t* __restrict__ keep /* nullable: kgl_b200_set_locus_filter */,
            uint16_t* __restrict__ flags16, uint16_t* __restrict__ sum64, uint32_t* __restrict__ n_rows) {
  __shared__ uint32_t s_bal[8];
  const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool in = false;
  if (l < n_loci) {
    const float a = af_pop[l];
    if (a == a) {
      const double v = (double)a;
      in = v >= lower && !(v >= upper);
      if (in && locus_counts) in = (locus_counts[l * 4 + 1] + locus_counts[l * 4 + 2]) != 0;
      if (in && keep) in = keep[l] != 0;
    }
  }
  if (l < padded_rows) flags16[l] = in ? 1u : 0u;
  const uint32_t bal = __ballot_sync(kFull, in);
  if ((threadIdx.x & 31) == 0) { s_bal[threadIdx.x >> 5] = bal; if (bal) atomicAdd(n_rows, (uint32_t)__popc(bal)); }
  __syncthreads();
  if (threadIdx.x < 4) {
    const uint64_t grp = (uint64_t)blockIdx.x * 4 + threadIdx.x;
    if (grp * 64 < padded_rows) {
      const uint32_t b0 = s_bal[threadIdx.x * 2], b1 = s_bal[threadIdx.x * 2 + 1];
      const uint32_t all = (b0 == 0xFFFFFFFFu && b1 == 0xFFFFFFFFu) ? 1u : 0u, any = (b0 | b1) ? 1u : 0u;
      sum64[grp] = (uint16_t)(all | (any << 8));
    }
  }
}

// AlleleSummmary of every genome over the masked rows: {referenceHomozygous_, minorHeterozygous_, minorHomozygous_, code 3}.
__global__ void k_genome_counts_masked(const uint32_t* __restrict__ gcounts, const uint32_t* __restrict__ n3s, uint64_t n_genomes,
                                       const uint32_t* __restrict__ n_rows, uint64_t* __restrict__ out, uint64_t* __restrict__ rows_out) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g == 0) *rows_out = *n_rows;
  if (g >= n_genomes) return;
  const uint64_t n3 = n3s[g], n1 = gcounts[g * 2] - n3, n2 = gcounts[g * 2 + 1] - n3;
  out[g * 4 + 0] = (uint64_t)(*n_rows) - n1 - n2 - n3; out[g * 4 + 1] = n1; out[g * 4 + 2] = n2; out[g * 4 + 3] = n3;
}

// ---------------------------------------------------------------------------------------------------------------------
// Synthetic genotypes, bit-identical to kgl_gene_b200/synth.py (numpy) -- the tests compare the two cell by cell.
// One thread = one 128-bit unit (64 genomes) of one locus row.
__global__ void __launch_bounds__(256)
k_synth(uint64_t seed, uint64_t n_genomes, uint64_t n_loci, uint64_t locus_base, uint64_t units,
        const float* __restrict__ af, const uint8_t* __restrict__ superpop, const double* __restrict__ inbreeding,
        uint64_t miss_threshold, uint4* __restrict__ packed) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_loci * units) return;
  const uint64_t l = idx / units, unit = idx % units;
  uint64_t lo = 0, hi = 0;
  for (int b = 0; b < 64; ++b) {
    const uint64_t g = unit * 64 + b;
    if (g >= n_genomes) break;
    const float a = af[(uint64_t)superpop[g] * n_loci + l];
    double p = (double)a;
    p = (a != a) ? 0.0 : (p < 0.0 ? 0.0 : (p > 1.0 ? 1.0 : p));
    const double q = __dsub_rn(1.0, p), F = inbreeding[g];
    const double pq = __dmul_rn(p, q);
    const double t0 = __dadd_rn(__dmul_rn(q, q), __dmul_rn(F, pq));
    const double t1 = __dadd_rn(t0, __dmul_rn(__dmul_rn(2.0, pq), __dsub_rn(1.0, F)));
    const uint64_t h1 = mix64(seed ^ ((locus_base + l) << 32) ^ g);
    const uint64_t h2 = mix64(h1 ^ 0xD6E8FEB86659FD93ULL);
    const double u = __dmul_rn((double)(h1 >> 11), 1.0 / 9007199254740992.0);
    unsigned code = (unsigned)(u >= t0) + (unsigned)(u >= t1);
    if ((h2 >> 40) < miss_threshold) code = 3;
    lo |= (uint64_t)(code & 1u) << b;
    hi |= (uint64_t)(code >> 1) << b;
  }
  packed[idx] = make_uint4((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
}

}  // namespace kgl
