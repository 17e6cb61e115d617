/* kgl_oracle.h -- TEST INFRASTRUCTURE. CPU restatement of KGL_Gene's population-genotype hot path.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load this
 * library, and only as the checker. The product (kgl_gene_b200/) never links or calls it.
 *
 * Parity status: PINNED for allele counting, locus selection, generateFrequencies, Simple, RitlandLocus,
 * logLikelihood(f) and the 50-sweep HallME map -- each is checked against outputs of the reference's own
 * code (oracle/_ref/kgl_ref_harness, built from /root/reference) in tests/test_oracle_vs_reference.py via
 * the committed fixtures under tests/golden/. UNPINNED: the Nelder-Mead optimiser itself (nlopt is an
 * un-vendored, un-versioned dependency) and pairwise IBS (no reference implementation exists; SURVEY 8c).
 *
 * All functions work on the flattened population (include/kgl_b200.h layout):
 *   packed  loci-major, row_bytes = 16*ceil(N/64); unit u = {u64 lo, u64 hi}; code = lo + 2*hi
 *   af      float[n_pop][L], NaN = no frequency for that super-population
 */
#ifndef KGL_ORACLE_H
#define KGL_ORACLE_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Field order of kga::LocusResults (kga_analysis_inbreed_output.h:21-35), genome id dropped. */
typedef struct {
  uint64_t major_hetero_count; double major_hetero_freq;
  uint64_t minor_hetero_count; double minor_hetero_freq;
  uint64_t minor_homo_count;   double minor_homo_freq;
  uint64_t major_homo_count;   double major_homo_freq;
  uint64_t total_allele_count; double inbred_allele_sum;
} kgl_oracle_locus_results;

enum { KGL_ORACLE_SIMPLE = 0, KGL_ORACLE_RITLAND = 1, KGL_ORACLE_HALLME = 2, KGL_ORACLE_LOGLIKELIHOOD = 3 };

/* RetrieveLociiVector::getAllelesFromTo / getAllelesCount (kga_analysis_inbreed_locus.cpp:21,105).
 * mode 0 = FromTo (stop when offset > upper), 1 = Count (stop when `count` loci selected; `upper` ignored).
 * Writes selected[l] = 1 for the chosen loci, returns how many; *last_index = index of the last chosen locus. */
size_t kgl_oracle_select_loci(const uint32_t* offsets, const float* af, size_t n_loci,
                              uint64_t lower, uint64_t upper, uint64_t spacing, uint64_t count,
                              double min_af, double max_af, int mode, uint8_t* selected, size_t* last_index);

/* Multi-allelic loci (oracle/flat_io.h, trailing section of KGLFLAT1): rows of the locus table with up to three alternate
 * alleles -- af f32[n_pop][n_multi][3] per allele slot (NaN = none), cells u8[n_multi][n_genomes] (0 hom-ref; low nibble the
 * first variant's slot + 1, 4 = not in the list; high nibble the second variant's, 0 = none; 0xFF = more than two variants).
 * Copied; used by every later kgl_oracle_select_loci_pop / kgl_oracle_inbreed* / kgl_oracle_loglik_grid call until reset with
 * n_multi = 0. The general forms of AlleleFreqVector, alleleClassFrequencies and the classification
 * (kga_analysis_inbreed_freq.cpp:18-57,127-217,452-543) apply at those rows. */
void kgl_oracle_set_multi(size_t n_multi, const uint32_t* rows, const float* af, const uint8_t* cells, size_t n_pop,
                          size_t n_genomes, size_t n_loci);
size_t kgl_oracle_select_loci_pop(const uint32_t* offsets, const float* af, size_t n_loci, size_t pop,
                                  uint64_t lower, uint64_t upper, uint64_t spacing, uint64_t count,
                                  double min_af, double max_af, int mode, uint8_t* selected, size_t* last_index);

/* InbreedingCalculation::generateFrequencies + process{Simple,RitlandLocus,HallME,LogLikelihood}
 * (kga_analysis_inbreed_freq.cpp:425-583, kga_analysis_inbreed_calc.cpp:319,375,226,154), biallelic loci.
 * selected: u8[n_pop][n_loci] from kgl_oracle_select_loci; superpop: u8[n_genomes]; unphased: SURVEY Q6.
 * HallME: start[g] is the EM start value, `sweeps` EM sweeps are run (reference: exactly 50, Q1); sweeps < 0 iterates
 *         to the fixed point. LogLikelihood: the converged argmax over [-1,1] of the reference objective. */
void kgl_oracle_inbreed(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                        const float* af, size_t n_pop, const uint8_t* selected, const uint8_t* superpop,
                        int unphased, int algorithm, const double* start, int sweeps,
                        kgl_oracle_locus_results* out);

/* The same for the listed genomes only (out[i] belongs to genomes[i]; NULL = the first n_some): checks at full BASELINE
 * width where the 50-sweep / root-search estimators over every genome would take minutes of CPU. */
void kgl_oracle_inbreed_some(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                             const float* af, size_t n_pop, const uint8_t* selected, const uint8_t* superpop,
                             int unphased, int algorithm, const double* start, int sweeps,
                             const uint32_t* genomes, size_t n_some, kgl_oracle_locus_results* out);

/* != 0: the per-genome sums of the calls above (expected class frequencies, Ritland's locus sum) are added with Neumaier's
 * compensation instead of in the reference's order and precision. Set it around a call, not across threads. */
void kgl_oracle_set_compensated_sums(int on);

/* InbreedingCalculation::logLikelihood (kga_analysis_inbreed_calc.cpp:94-129) on a grid of f values. out[g][i]. */
void kgl_oracle_loglik_grid(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                            const float* af, size_t n_pop, const uint8_t* selected, const uint8_t* superpop,
                            int unphased, const double* grid, size_t n_grid, double* out);

/* VariantDBVariant::summaryByVariant / summaryByGenome / populationSummary (kgl_variant_db_variant.cpp:126,180,234).
 * locus_counts u32[L][4] and genome_counts u64[N][4] hold the number of cells with code 0,1,2,3
 * (the reference's AlleleSummmary is columns 0,1,2; code 3 has no reference counterpart). */
void kgl_oracle_allele_count(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                             uint32_t* locus_counts, uint64_t* genome_counts);

/* Pairwise IBS (no reference code; standard definitions, SURVEY 8c). out u32[N][N][4] = ibs0, ibs1, ibs2, valid. */
void kgl_oracle_ibs(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci, uint32_t* out);

/* The same counts for the genomes [row_begin, row_end) against all genomes by AND/XOR + popcount over 64-locus words of
 * genome-major bit-planes ("popcount CPU restatement for scale", SURVEY 8c). out u32[row_end - row_begin][N][4]. */
void kgl_oracle_ibs_band_popcount(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                                  size_t row_begin, size_t row_end, uint32_t* out);

/* Dosage Gram matrix gram i32[N][N] = sum_l g_a g_b (code 3 -> 0) and, when af_pop and grm are given, the centred matrix
 * grm f64[N][N] = sum_l (g_a - 2p)(g_b - 2p), p = clamp(af_pop[l], 0, 1), absent AF -> 0. No reference code (SURVEY 8d, K5). */
void kgl_oracle_gram(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci, const float* af_pop,
                     int32_t* gram, double* grm);

/* Synthetic genotype law shared with the product's device generator (kgl_b200_synth_genotypes): counter-based
 * splitmix64 per cell, genotype drawn from {q^2+Fpq, 2pq(1-F), p^2+Fpq} (the law of
 * AlleleFreqVector::unadjustedAlleleClassFrequencies, kga_analysis_inbreed_freq.cpp:127-205). */
void kgl_oracle_synth_genotypes(uint64_t seed, size_t n_genomes, size_t n_loci, size_t locus_base,
                                const float* af, size_t n_pop, const uint8_t* superpop,
                                const double* inbreeding, double missing_rate, uint8_t* packed, size_t row_bytes);

int kgl_oracle_threads(void);

#ifdef __cplusplus
}
#endif
#endif
