/* kgl_b200.h -- C ABI of the B200-native population-genotype hot path for KGL_Gene.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types, no exceptions. A KGL_Gene maintainer binds
 * it from a VirtualAnalysis subclass (kgl_app/kgl_package_analysis_virtual.h:20-55) -- see INTEGRATION.md and
 * kgl_gene_b200/host/ for the C++ host layer (flattener, locus selection, window loop, CSV writer) that sits on top.
 * Every entry point names the reference routine it replaces (paths relative to the KGL_Gene tree).
 *
 * Threading: a context is used from one host thread at a time (the reference calls its analysis stages sequentially
 * from the main thread, kgl_app/kgl_package.cpp:17-77). Several contexts (one per GPU / per rank) may coexist.
 * There is NO CPU fallback: every compute entry point fails with KGL_B200_ERR_NO_DEVICE / _CUDA when no sm_100 device
 * is usable.
 *
 * ---- data layout (what the host flattener emits) ------------------------------------------------------------------
 *  genotype matrix  loci-major, 2 bits per genome, rows aligned to 128 bits:
 *                   row_bytes = 16 * ceil(n_genomes / 64); row l = units u = 0..row_bytes/16-1;
 *                   unit u = { uint64 lo, uint64 hi } (little endian) for genomes 64u .. 64u+63,
 *                   code(g) = bit(lo, g%64) + 2*bit(hi, g%64):
 *                     0 = no variant at the offset (hom-ref)           kga_analysis_inbreed_freq.cpp:521-541
 *                     1 = one copy of the locus' alt allele (het)       :464-472
 *                     2 = two copies (hom-alt)                          :476-479
 *                     3 = dropped / unclassifiable / missing           (first variant not in the AF list, >2 variants, ...)
 *                   padding genomes (>= n_genomes) must be 0.
 *  allele frequency float[n_pop][n_loci], the INFO float exactly as the reference stores it
 *                   (kgl_variant_factory_vcf_parse_info.cpp:232); NaN = no value for that super-population.
 *                   Populations are indexed AFR, AMR, EAS, EUR, SAS, ALL (kgl_variant_db_freq.h:55-71).
 *  super-population uint8[n_genomes], index of each genome's PED super-population (kgl_hsgenealogy_parser.h:68).
 *  locus selection  uint8[n_loci], bit k set = locus is in super-population k's locus list for the current window
 *                   (InbreedSampling::getLocusList, kga_analysis_inbreed_locus.cpp:263).
 */
#ifndef KGL_B200_H
#define KGL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KGL_B200_OK             0
#define KGL_B200_ERR_INVALID    1   /* bad argument */
#define KGL_B200_ERR_STATE      2   /* call order: something required has not been uploaded yet */
#define KGL_B200_ERR_CUDA       3   /* a CUDA call failed; see kgl_b200_last_error */
#define KGL_B200_ERR_NO_DEVICE  4   /* no usable sm_100 GPU */
#define KGL_B200_ERR_NOMEM      5
#define KGL_B200_ERR_PEER       6   /* a peer rank did not reach the exchange in time; export / attach the regions again */

#define KGL_B200_MAX_POP 6

/* InbreedingCalculation::inbreeding_algo_map_ (kga_analysis_inbreed_calc.h:103-118). */
#define KGL_B200_ALGO_SIMPLE        0   /* "Simple"        processSimple         calc.cpp:319 */
#define KGL_B200_ALGO_RITLAND       1   /* "RitlandLocus"  processRitlandLocus   calc.cpp:375 */
#define KGL_B200_ALGO_HALLME        2   /* "HallME"        processHallME         calc.cpp:226 */
#define KGL_B200_ALGO_LOGLIKELIHOOD 3   /* "Loglikelihood" processLogLikelihood  calc.cpp:154 */

typedef struct kgl_b200_ctx kgl_b200_ctx;

/* Same fields, same order as kga::LocusResults (kga_analysis_inbreed_output.h:21-35) without the genome id string. */
typedef struct kgl_b200_locus_results {
  uint64_t major_hetero_count; double major_hetero_freq;
  uint64_t minor_hetero_count; double minor_hetero_freq;
  uint64_t minor_homo_count;   double minor_homo_freq;
  uint64_t major_homo_count;   double major_homo_freq;
  uint64_t total_allele_count; double inbred_allele_sum;
} kgl_b200_locus_results;

/* Options of the iterative estimators. Zero-initialise for the defaults. */
typedef struct kgl_b200_inbreed_options {
  /* HallME: EM start value per genome (NULL = 0.25 for all) and number of sweeps. The reference runs exactly 50 sweeps
   * from a random start in (0,0.5] (SURVEY Q1-Q3); sweeps == 0 means 50; sweeps < 0 iterates to the EM fixed point. */
  const double* hall_start;
  int32_t hall_sweeps;
  /* Loglikelihood: bracketed Newton on d/df of the reference objective over the feasible region (no homozygous
   * probability clamped), from the Simple estimate; stops when |step| < ll_tolerance (0 = 1e-12) or after
   * ll_max_iterations (0 = 200). */
  double ll_tolerance;
  int32_t ll_max_iterations;
  /* != 0: the moments pass of kgl_b200_inbreed_accumulate also produces the per-locus allele counts of this rank's
   * locus shard (the fused pass of kgl_b200_run_count_and_inbreed, split around the all-reduce). */
  int32_t count_loci;
  /* HallME / Loglikelihood sweeps: 0 = from the per-genome moment tables built once per selection (terms_moments.cuh; a sweep
   * then reads no genotype), != 0 = every sweep evaluates every cell (the exact kernels, which the tables fall back to for
   * genomes outside their domain). Both follow calc.cpp:94-129,257-285; they agree to < 1e-10. */
  int32_t exact_sweeps;
  /* != 0: the sparse half of the moment tables is built by the CUDA-core kernel (k_mom_build) instead of the tensor-core one
   * (k_mom_mma). Same integers either way; the tensor-core builder is several times faster. */
  int32_t moments_on_cuda_cores;
  /* kgl_b200_run_inbreed only: != 0 = go through kgl_b200_inbreed_accumulate / kgl_b200_inbreed_update sweep by sweep (what a
   * locus-sharded caller does around its all-reduce) instead of running all sweeps of all genomes in one launch over the tables. */
  int32_t sweep_by_sweep;
} kgl_b200_inbreed_options;

/* ---- lifetime ------------------------------------------------------------------------------------------------- */
const char* kgl_b200_version(void);
int  kgl_b200_device_count(void);
int  kgl_b200_create(int device, kgl_b200_ctx** ctx);
void kgl_b200_destroy(kgl_b200_ctx* ctx);
/* Message of the last failure on this context (ctx == NULL: of the last failed kgl_b200_create on this thread). */
const char* kgl_b200_last_error(const kgl_b200_ctx* ctx);
/* All kernels of this context are enqueued on `cuda_stream` (a cudaStream_t; NULL = the context's own stream). */
int  kgl_b200_set_stream(kgl_b200_ctx* ctx, void* cuda_stream);
int  kgl_b200_synchronize(kgl_b200_ctx* ctx);

/* ---- population upload (host buffers; replaces walking PopulationDB per genome, kga_analysis_inbreed_freq.cpp:436-452) */
int kgl_b200_upload_genotypes(kgl_b200_ctx* ctx, uint64_t n_genomes, uint64_t n_loci, uint64_t row_bytes, const void* packed);
int kgl_b200_upload_loci(kgl_b200_ctx* ctx, uint64_t n_loci, uint32_t n_pop, const float* af, const uint32_t* offsets);
int kgl_b200_set_genome_superpop(kgl_b200_ctx* ctx, uint64_t n_genomes, const uint8_t* superpop);
/* Pf7-style population: all variants UNPHASED, so a hom-alt pair is classified MINOR_HETEROZYGOUS (SURVEY Q6). */
int kgl_b200_set_unphased(kgl_b200_ctx* ctx, int unphased);

/* Loci with several alternate alleles (the "3 + side list" rows of the flattener contract; call after the three uploads above).
 * rows[n_multi]: ascending rows of the locus table -- there the frequency table is ignored (treated as "no value") and the matrix
 * holds only 0 (hom-ref) and 3 (see cells). af float[n_pop][n_multi][3]: frequency of allele slot 0..2 (the order of the locus'
 * variant array) per super-population, NaN = the allele has no value for it. cells uint8[n_multi][n_genomes]: 0 = hom-ref; low
 * nibble = allele slot + 1 of the FIRST variant at the offset (4 = an allele that is not in the list), high nibble = the second
 * variant's (0 = none); 0xFF = more than two variants. The general form of the reference's classification applies there:
 * AlleleFreqVector over several alleles, major frequency = complement of their sum, MINOR_HETEROZYGOUS for two different
 * alleles, the class frequencies of alleleClassFrequencies (kga_analysis_inbreed_freq.cpp:18-57,127-217,452-543). For the pairwise
 * kernels such a cell is "missing". kgl_b200_run_multi_allele_count: per-allele summaries (one VariantDBVariant column per
 * allele, kgl_variant_db_variant.cpp:14-30): counts uint32[n_multi][3][3] = genomes with 0, 1, 2 copies of allele slot a. */
int kgl_b200_upload_multi_allelic(kgl_b200_ctx* ctx, uint64_t n_multi, const uint32_t* rows, const float* af, const uint8_t* cells);
int kgl_b200_run_multi_allele_count(kgl_b200_ctx* ctx, uint32_t* counts);

/* Locus selection for the current window. kgl_b200_select_loci applies RetrieveLociiVector::getLociiFromTo
 * (kga_analysis_inbreed_locus.cpp:21-72,76) to every super-population: loci with lower <= offset <= upper, at least
 * `spacing` apart, valid AF with 0 < AF and min_af <= AF <= max_af. n_selected (nullable) receives n_pop counts.
 * kgl_b200_set_locus_selection uploads a mask computed elsewhere. Default after kgl_b200_upload_loci: nothing selected. */
int kgl_b200_select_loci(kgl_b200_ctx* ctx, uint64_t lower, uint64_t upper, uint64_t spacing,
                         double min_af, double max_af, uint64_t* n_selected);
int kgl_b200_set_locus_selection(kgl_b200_ctx* ctx, uint64_t n_loci, const uint8_t* selected);
/* RetrieveLociiVector::getLociiCount (kga_analysis_inbreed_locus.cpp:159-183): how InbreedingAnalysis::populationInbreeding
 * defines its windows (kga_analysis_inbreed_diploid.cpp:48-51,69-73). The first `count` loci of super-population `pop` that
 * the accept rule of kgl_b200_select_loci takes from `lower` on: *n_found of them (<= count), *last_offset = offset of the last
 * one (the window's upper bound). Replaces the selection. */
int kgl_b200_count_loci(kgl_b200_ctx* ctx, uint32_t pop, uint64_t lower, uint64_t spacing, uint64_t count, double min_af, double max_af,
                        uint64_t* n_found, uint64_t* last_offset);
/* Per-locus verdict of the variant-level population filters, applied by kgl_b200_select_loci / kgl_b200_count_loci and the AF-bin
 * passes: keep uint8[n_loci], 0 = the locus is never selected (its genotypes still count in kgl_b200_run_allele_count). What the
 * reference does by copying the population through viewFilter: AndFilter(SNPFilter(), PassFilter()) on the frequency source
 * (kga_analysis_inbreed.cpp:79), P7VariantFilter / P7FrequencyFilter / SNPFilter of FilterPf7::qualityFilter
 * (kga_analysis_library/kga_analysis_lib_PfFilter.cpp:62-92). NULL clears it; kgl_b200_upload_loci clears it. */
int kgl_b200_set_locus_filter(kgl_b200_ctx* ctx, uint64_t n_loci, const uint8_t* keep);
int kgl_b200_get_locus_selection(kgl_b200_ctx* ctx, uint64_t n_loci, uint8_t* selected);

/* Synthetic population generated on the device (configs too large to stage through a PopulationDB; the law is
 * InbreedSynthetic's, kga_analysis_inbreed_syngen.cpp:20-196). Needs upload_loci + set_genome_superpop first.
 * Cells are a pure function of (seed, locus_base + locus, genome), so shards of one population can be generated
 * independently on different GPUs. */
int kgl_b200_synth_genotypes(kgl_b200_ctx* ctx, uint64_t seed, uint64_t n_genomes, uint64_t n_loci, uint64_t locus_base,
                             const double* inbreeding, double missing_rate);
int kgl_b200_download_genotypes(kgl_b200_ctx* ctx, uint64_t n_bytes, void* packed);

/* ---- hot path, host-buffer results (synchronous) ------------------------------------------------------------------ */
/* VariantDBVariant::summaryByVariant / summaryByGenome / populationSummary (kgl_variant_db_variant.cpp:126,180,234):
 * locus_counts uint32[n_loci][4] and genome_counts uint64[n_genomes][4] = number of cells with code 0,1,2,3
 * (AlleleSummmary = {referenceHomozygous_, minorHeterozygous_, minorHomozygous_} = columns 0,1,2). Either may be NULL. */
int kgl_b200_run_allele_count(kgl_b200_ctx* ctx, uint32_t* locus_counts, uint64_t* genome_counts);

/* InbreedingCalculation::process{Simple,RitlandLocus,HallME,LogLikelihood} for every genome over the selected loci
 * (kga_analysis_inbreed_calc.cpp:319,375,226,154 on top of generateFrequencies, kga_analysis_inbreed_freq.cpp:425-583).
 * out[n_genomes]. options may be NULL. */
int kgl_b200_run_inbreed(kgl_b200_ctx* ctx, int algorithm, const kgl_b200_inbreed_options* options,
                         kgl_b200_locus_results* out);

/* The sweeps of the last HallME / Loglikelihood run on this context: 0 the exact kernels, 1 moment tables built on the CUDA cores,
 * 2 moment tables built on the tensor cores. */
int kgl_b200_inbreed_used_moment_tables(const kgl_b200_ctx* ctx);

/* The fused streaming pass the benchmark times: one read of the genotype matrix yields the per-locus allele counts
 * AND the per-genome Simple moments (class counts, expected class-frequency sums, F). Either output may be NULL. */
int kgl_b200_run_count_and_inbreed(kgl_b200_ctx* ctx, uint32_t* locus_counts, kgl_b200_locus_results* out);

/* InbreedingCalculation::logLikelihood (kga_analysis_inbreed_calc.cpp:94-129) on a grid of f values: out[n_genomes][n_grid]. */
int kgl_b200_run_loglik_grid(kgl_b200_ctx* ctx, const double* grid, uint64_t n_grid, double* out);

/* Pairwise identity-by-state between genomes [row_begin,row_end) and all genomes, over all loci:
 * out uint32[row_end-row_begin][n_genomes][4] = {IBS0, IBS1, IBS2, loci valid in both}. (No reference routine exists;
 * the matrix is the one VariantDBVariant::genomeData() describes, kgl_variant_db_variant.h:49-51; SURVEY 8c.) */
int kgl_b200_run_ibs(kgl_b200_ctx* ctx, uint64_t row_begin, uint64_t row_end, uint32_t* out);

/* The same matrix as 64 x 64 sample-pair tiles, the unit that is dealt to GPUs (SURVEY 8e: "upper-triangular sample-pair
 * tiles dealt block-cyclically"). The tile grid has tiles_per_side = ceil(n_genomes / 64) rows; only the upper triangle
 * (ti <= tj) exists, numbered row-major: t = 0 is (0,0), t = 1 is (0,1), ... n_upper_tiles = side (side + 1) / 2.
 * kgl_b200_run_ibs_tiles computes tiles first, first + stride, ... (count of them; rank r of R ranks passes first = r,
 * stride = R) into out uint32[count][64][64][4] = {IBS0, IBS1, IBS2, valid}; cell [i][j] of tile (ti,tj) is the pair
 * (64 ti + i, 64 tj + j); cells of padding genomes are 0. */
int kgl_b200_ibs_tile_grid(kgl_b200_ctx* ctx, uint64_t* tiles_per_side, uint64_t* n_upper_tiles);
/* The dense part of every IBS entry point runs on the tensor cores when it can (default): IBS0 / IBS1 follow exactly from three
 * int8 Gram matrices -- heterozygous indicator, hom-alt indicator, dosage (ibs_gram.cuh) -- at ~3 PetaOP/s instead of 5 LOP3 + 1
 * POPC per pair-word. The matrices exist only as the 256 x 256 blocks under the tiles of a call, so any width works; it needs
 * n_loci < 2^29 and code-3 cells that are indexed or absent; otherwise, or with enable = 0, the popcount tile kernel runs. Same
 * integers either way. */
int kgl_b200_set_ibs_tensor_cores(kgl_b200_ctx* ctx, int enable);
int kgl_b200_ibs_used_tensor_cores(const kgl_b200_ctx* ctx);     /* the last IBS call: 1 tensor cores, 0 popcount kernel */
int kgl_b200_run_ibs_tiles(kgl_b200_ctx* ctx, uint64_t first, uint64_t stride, uint64_t count, uint32_t* out);

/* KING-robust kinship (Manichaikul et al., Bioinformatics 2010; the between-family estimator of PLINK 2's --make-king), for
 * structured populations: it needs no allele frequencies. For genomes a, b over the loci where neither is coded 3 (multi-allelic
 * rows count as missing for their non-reference cells, as in kgl_b200_run_ibs):
 *     kinship = 0.5 - (4 IBS0 + IBS1) / (4 min(het_a, het_b))        NaN when min(het_a, het_b) == 0
 * het_a / het_b = heterozygous loci of a / of b among the loci valid in both; het_het = loci where both are heterozygous
 * (het_a + het_b = IBS1 + 2 het_het). Counts are exact integers and the kinship is one IEEE division and one subtraction in
 * double. IBS0 / IBS1 come from the IBS path (tensor cores or popcount kernel, kgl_b200_set_ibs_tensor_cores), het_het and the
 * per-pair het counts from int8 Gram runs on the tensor cores (king.cuh). n_loci < 2^29. Both entry points need a genotype upload
 * (KGL_B200_ERR_STATE before it). */
typedef struct kgl_b200_king_pair {          /* 40 bytes */
  uint32_t a, b;                             /* genome indices, a < b */
  uint32_t n_valid, ibs0, ibs1, het_het, het_a, het_b;
  double kinship;
} kgl_b200_king_pair;
/* kinship double[row_end-row_begin][n_genomes]: genomes [row_begin,row_end) against all genomes (the band / whole-matrix logic of
 * kgl_b200_run_ibs). The diagonal is 0.5 for a genome with a heterozygous locus. */
int kgl_b200_run_king(kgl_b200_ctx* ctx, uint64_t row_begin, uint64_t row_end, double* kinship);
/* Every pair a < b with kinship >= min_kinship (NaN never qualifies) inside the given 64 x 64 tiles (coords uint32[n_coords][2] =
 * (tile row, tile column) with tile row <= tile column, e.g. a rank's shards.block_tile_coords; NULL or n_coords == 0 = the whole
 * upper triangle), in ascending (a, b) order. *n_pairs = the true total; if it exceeds capacity nothing is copied and the call
 * returns KGL_B200_ERR_NOMEM: retry with capacity = *n_pairs (the retry computes every tile again). A tile outside the grid or below the diagonal: KGL_B200_ERR_INVALID.
 * 0.0442 (~2^-4.5) keeps third-degree relatives and closer. */
int kgl_b200_run_king_pairs(kgl_b200_ctx* ctx, uint64_t n_coords, const uint32_t* coords, double min_kinship, uint64_t capacity,
                            kgl_b200_king_pair* pairs, uint64_t* n_pairs);

/* Genotype PCA (the ancestry axes of PLINK 2's --pca approx; Galinsky et al. 2016): the top principal components of the
 * variance-standardised genotype matrix, matrix-free. For locus l with raw counts n0..n3 (kgl_b200_run_allele_count),
 * v = n0 + n1 + n2 and p = (n1 + 2 n2) / (2 v). The used loci U are those with keep[l] != 0 (keep NULL = every locus) and
 * 0 < p < 1; M = |U| (multi-allelic rows hold only 0 and 3: p = 0, never used). For l in U and a cell not coded 3,
 *     z_lg = (g_lg - 2 p_l) / sqrt(2 p_l (1 - p_l)),   every other z_lg = 0    (code-3 cells mean-imputed, as PLINK does)
 * and Psi = Z^T Z / M is PLINK's variance-standardised relationship matrix. It is never formed: Z^T Z times a block of <= 48
 * columns runs as exact int8 Gram runs on the tensor cores against the block written as base-4 digits of a 30-bit fixed-point
 * form (2^-29 of each column's largest entry; pca.cuh); the double arithmetic after the integer contractions is a fixed
 * sequence of IEEE operations, so results are reproducible bit for bit. kgl_b200_run_pca is randomized subspace iteration
 * (Halko, Martinsson & Tropp 2011, Alg. 4.4) on a block of b = 16 ceil((k + 6) / 16) columns from a Gaussian start block
 * that is a pure function of (seed, genome, column): `iterations` products each followed by a Householder QR, then
 * Rayleigh-Ritz with a cyclic Jacobi eigensolve of the b x b projection -- the QR and the eigensolve run on the host in
 * double. Outputs: eigenvalues[k] of Psi in descending order; scores double[n_genomes][k], the unit eigenvectors, each signed
 * so that its entry of largest magnitude is positive (the lowest index wins a tie); loadings (nullable) double[n_loci][k],
 * u_i = Z v_i / sqrt(M lambda_i), 0 at unused loci; *n_loci_used = M (nullable). Needs a genotype upload
 * (KGL_B200_ERR_STATE before it); KGL_B200_ERR_INVALID for k outside 1..40, k >= n_genomes, k > M, no used locus or
 * n_loci >= 2^28. LD pruning (kgl_b200_run_ld_prune below) gives a keep mask for it. There is no popcount form: kgl_b200_set_ibs_tensor_cores does not apply. The device keeps a loci-major
 * copy of the codes (n_genomes * n_loci / 4 bytes) from the first call after an upload. */
typedef struct kgl_b200_pca_options {        /* zero-initialise for the defaults */
  const uint8_t* keep;                       /* uint8[n_loci], 0 = leave the locus out; NULL = every locus */
  uint32_t n_components;                     /* k, 1..40; 0 = 10 */
  uint32_t iterations;                       /* q; 0 = 10 */
  uint64_t seed;                             /* start block */
} kgl_b200_pca_options;
int kgl_b200_run_pca(kgl_b200_ctx* ctx, const kgl_b200_pca_options* options, double* eigenvalues /* [k] */,
                     double* scores /* [n_genomes][k] */, double* loadings /* nullable, [n_loci][k] */, uint64_t* n_loci_used);
/* y = Z^T Z x (not divided by M) for a block of 1 <= n_cols <= 48 columns: the operator itself, on the loci of `keep` (as
 * above). A locus-sharded caller sums it over ranks. Same errors as kgl_b200_run_pca (n_cols outside 1..48: INVALID). */
int kgl_b200_run_grm_product(kgl_b200_ctx* ctx, const uint8_t* keep, uint32_t n_cols, const double* x /* [n_genomes][n_cols] */,
                             double* y /* [n_genomes][n_cols] */, uint64_t* n_loci_used);

/* Linkage disequilibrium between loci: the genotypic r^2 of locus pairs inside a window, and LD pruning -- what PCA and KING are
 * normally run on. No phasing is involved.
 * Eligible loci: exactly PCA's used set U above (keep[l] != 0, keep NULL = every locus, and 0 < p < 1 from the raw counts;
 * multi-allelic rows have p = 0 and are never eligible). rank(l) = index of l among the eligible loci.
 * Window: eligible i < j (locus rows) form an in-window pair iff
 *     (window_loci == 0 || rank(j) - rank(i) < window_loci)   -- the eligible loci are counted, as PLINK counts variants after filtering
 * and (window_bp == 0 || offset[j] - offset[i] <= window_bp)  -- the offsets of kgl_b200_upload_loci (sorted; KGL_B200_ERR_STATE
 *                                                                without them, KGL_B200_ERR_INVALID when they decrease)
 * Both limits 0: KGL_B200_ERR_INVALID.
 * r^2 is the squared Pearson correlation of the allele counts g in {0,1,2} over the genomes where neither cell is coded 3. With
 * q = g^2, c = the code-3 indicator, per-locus totals s = n1 + 2 n2, q = n1 + 4 n2, c = n3 and, over genomes, GG = sum g_i g_j,
 * CC = sum c_i c_j, GC_ij = sum g_i c_j, QC_ij = sum q_i c_j:
 *     n = N - c_i - c_j + CC,  S_i = s_i - GC_ij,  S_j = s_j - GC_ji,  Q_i = q_i - QC_ij,  Q_j = q_j - QC_ji
 *     cov = n GG - S_i S_j,  var_i = n Q_i - S_i^2,  var_j = n Q_j - S_j^2          (exact integers)
 *     r^2 = (cov * cov) / (var_i * var_j)                                           (each int64 exactly a double; three IEEE ops)
 * NaN when var_i or var_j is 0; a NaN never qualifies for the pair list and never prunes. The sums are exact int8 Gram runs on
 * the tensor cores over 256 x 256 tiles of loci along the diagonal (ld.cuh), so results are bit-reproducible.
 * Limits: n_genomes < 2^25 (every term < 4 N^2 < 2^53; else KGL_B200_ERR_INVALID), n_loci < 2^32. The device keeps PCA's
 * loci-major copy of the codes (n_genomes * n_loci / 4 bytes) from the first call after an upload.
 * Both entry points need a genotype upload (KGL_B200_ERR_STATE before it) and return KGL_B200_ERR_INVALID for a NaN threshold,
 * both windows 0 or a null output pointer. */
typedef struct kgl_b200_ld_options {         /* zero-initialise; 16 bytes */
  const uint8_t* keep;                       /* uint8[n_loci], 0 = leave the locus out; NULL = every locus (PCA's meaning) */
  uint32_t window_loci;                      /* 0 = no limit on the eligible-locus distance */
  uint32_t window_bp;                        /* 0 = no limit on the offset distance */
} kgl_b200_ld_options;
typedef struct kgl_b200_ld_pair {            /* 24 bytes */
  uint32_t a, b;                             /* locus rows, a < b */
  uint32_t n_valid, reserved;                /* n above (genomes valid at both loci); reserved = 0 */
  double r2;
} kgl_b200_ld_pair;
/* Every in-window pair with r^2 >= min_r2, in ascending (a, b) order. *n_pairs = the true total; if it exceeds capacity nothing is
 * copied and the call returns KGL_B200_ERR_NOMEM: retry with capacity = *n_pairs (the retry computes everything again). */
int kgl_b200_run_ld_pairs(kgl_b200_ctx* ctx, const kgl_b200_ld_options* options, double min_r2, uint64_t capacity,
                          kgl_b200_ld_pair* pairs, uint64_t* n_pairs);
/* Greedy LD pruning in locus order: eligible l is kept unless an EARLIER KEPT eligible locus i has (i, l) in the window and
 * r^2(i, l) > max_r2. keep_out uint8[n_loci] = 0/1 (0 for every ineligible locus), *n_kept = its sum. It is meant to be
 * passed straight to kgl_b200_pca_options.keep (run_pca then reports n_loci_used == n_kept), or used to drop loci before KING.
 * This is not PLINK's --indep-pairwise window/step procedure: it is the rule defined by the locus order alone, with one answer
 * whatever a step size would be. */
int kgl_b200_run_ld_prune(kgl_b200_ctx* ctx, const kgl_b200_ld_options* options, double max_r2, uint8_t* keep_out /* [n_loci] */,
                          uint64_t* n_kept);

/* Population differentiation between groups of genomes (the super-populations, Pf7 locations, or any labelling).
 * kgl_b200_run_group_counts: counts uint32[n_loci][n_groups][4], counts[l][k][c] = genomes of group k whose cell at locus l has
 * code c, counted as kgl_b200_run_allele_count counts them (multi-allelic rows: their matrix codes 0 and 3), so the sum over the
 * groups plus the genomes in no group is its locus_counts. group uint8[n_genomes]: 0 .. n_groups-1, or 0xFF = in no group;
 * group == NULL: the labels of kgl_b200_set_genome_superpop with n_groups = KGL_B200_MAX_POP (the argument is ignored). One read of
 * the resident matrix (fst.cuh). Errors: KGL_B200_ERR_STATE before a genotype upload, or for group == NULL without super-population
 * labels; KGL_B200_ERR_INVALID for n_groups outside 1..64 or a label >= n_groups other than 0xFF. */
int kgl_b200_run_group_counts(kgl_b200_ctx* ctx, uint32_t n_groups, const uint8_t* group /* [n_genomes] or NULL */,
                              uint32_t* counts /* [n_loci][n_groups][4] */);
/* F_ST between pairs of groups. Per group k at locus l, from its counts n0..n3 (code-3 cells are missing):
 *     v_k = n0 + n1 + n2,   p_k = (n1 + 2 n2) / (2 v_k),   h_k = n1 / v_k
 * Hudson (Hudson, Slatkin & Maddison 1992, as Bhatia et al. 2013 eq. 10; scikit-allel's hudson_fst), groups a, b:
 *     num = (p_a - p_b)^2 - p_a (1 - p_a) / (2 v_a - 1) - p_b (1 - p_b) / (2 v_b - 1)
 *     den = p_a (1 - p_b) + p_b (1 - p_a)
 * Weir & Cockerham 1984 (r = 2 groups; the alt allele's a, b, c -- for two alleles each allele has the same ones):
 *     n_bar = (v_a + v_b) / 2,   n_c = 2 v_a v_b / (v_a + v_b)            (= (r n_bar - sum v^2 / (r n_bar)) / (r - 1))
 *     p_bar = (s_a + s_b) / (2 (v_a + v_b)) with s = n1 + 2 n2,   s2 = (v_a (p_a - p_bar)^2 + v_b (p_b - p_bar)^2) / n_bar
 *     h_bar = (n1_a + n1_b) / (v_a + v_b),   pq = p_bar (1 - p_bar)
 *     a = (n_bar / n_c) (s2 - (pq - s2 / 2 - h_bar / 4) / (n_bar - 1))
 *     b = (n_bar / (n_bar - 1)) (pq - s2 / 2 - ((2 n_bar - 1) / (4 n_bar)) h_bar)
 *     c = h_bar / 2,   num = a,   den = (a + b) + c
 * Each formula is evaluated exactly as written, left to right, one IEEE round-to-nearest double operation at a time (no FMA), from
 * the exact integer counts (v, s, 2 v - 1, v_a v_b, v_a + v_b, n1_a + n1_b are integers converted once), so results are
 * reproducible bit for bit. A locus is used for a pair when keep[l] != 0 (keep NULL = every locus), v_a >= 1 and v_b >= 1
 * (Hudson: then 2 v - 1 >= 1; Weir-Cockerham: n_c > 0) and, for Weir-Cockerham, n_bar > 1 (v_a + v_b >= 3), and den != 0 (a locus
 * monomorphic across both groups contributes nothing). Genome-wide F_ST = sum num / sum den over the used loci, NaN when none is
 * used. Summation order, independent of the GPU and of any launch plan: the loci in blocks of 256 (rows 256 x .. 256 x + 255; a
 * locus that is not used, or past the last row, adds 0.0), each block summed as a halving tree (element i += element i + s for
 * s = 128, 64, .., 1), then the block sums added in block order from 0.0.
 * Windows (window_bp != 0; step_bp == 0 means step = window_bp): window w = 0 .. floor(max offset / step) covers the loci with
 * offsets in [w step, w step + window_bp), the offsets of kgl_b200_upload_loci (sorted; KGL_B200_ERR_STATE without them,
 * KGL_B200_ERR_INVALID when they decrease). Its sums add the used loci in row order from 0.0.
 * Outputs: fst double[n_pairs]; per_locus (nullable) double[n_pairs][n_loci][2] = (num, den), (0, 0) where not used; windows
 * (nullable) double[n_pairs][n_windows][3] = (sum num, sum den, loci used); *n_windows (nullable) = the number of windows (0 without), set only when the call succeeds.
 * The pairs are `pairs` [n_pairs][2] with a < b < n_groups, or, for n_pairs == 0 or pairs == NULL, every pair a < b in order
 * (0,1), (0,2), .., (1,2), ... The group counts stay on the device. Errors: those of kgl_b200_run_group_counts, and
 * KGL_B200_ERR_INVALID for a method other than 0 / 1, a bad pair, no pair (one group) or a null fst. */
#define KGL_B200_FST_HUDSON 0
#define KGL_B200_FST_WEIR_COCKERHAM 1
typedef struct kgl_b200_fst_options {       /* zero-initialise; 56 bytes */
  const uint8_t* group;   uint32_t n_groups;  /* as kgl_b200_run_group_counts */
  const uint8_t* keep;                        /* uint8[n_loci], NULL = every locus */
  uint32_t method;                            /* KGL_B200_FST_HUDSON or KGL_B200_FST_WEIR_COCKERHAM */
  uint32_t n_pairs;   const uint32_t* pairs;  /* [n_pairs][2] (a < b); 0 / NULL = every pair a < b */
  uint64_t window_bp, step_bp;                /* 0 = no windows */
} kgl_b200_fst_options;
int kgl_b200_run_fst(kgl_b200_ctx* ctx, const kgl_b200_fst_options* options, double* fst /* [n_pairs] */,
                     double* per_locus /* nullable, [n_pairs][n_loci][2] */, double* windows /* nullable, [n_pairs][n_windows][3] */,
                     uint64_t* n_windows);

/* Hardy-Weinberg equilibrium per locus and group, and variant QC (PLINK's --hardy and --hwe / --geno / --maf). The test assumes
 * diploid calls (for Pf7 a heterozygous call is a mixed infection, not a diploid genotype). Run it per super-population: pooling
 * differentiated populations fails HWE at nearly every common site (the Wahlund effect).
 * For group k at locus l with the counts n0..n3 of kgl_b200_run_group_counts (code 3 is missing):
 *     v = n0 + n1 + n2,  n_r = min(n1 + 2 n2, n1 + 2 n0) rare-allele copies,  n_c = 2 v - n_r
 * The support is h = n_r mod 2, .., n_r - 2, n_r heterozygotes; at h there are r = (n_r - h) / 2 rare and c = (n_c - h) / 2 common
 * homozygotes. Exact test (Wigginton, Cutler & Abecasis 2005) as this fixed sequence of IEEE double operations, round to nearest,
 * no FMA (every integer is computed exactly and converted once; all are exact in double because v < 2^25):
 *     mode m = floor(n_r n_c / (2 v)) in integers, plus 1 when its parity differs from n_r's;  P(m) = 1.0
 *     downward  P(h - 2) = (P(h) * (double)(h (h - 1))) / (double)(4 (r + 1) (c + 1))
 *     upward    P(h + 2) = (P(h) * (double)(4 r c)) / (double)((h + 2) (h + 1))
 *     S = 1.0, then + P(m - 2), + P(m - 4), .. (the terms below the mode in the order computed), then + P(m + 2), + P(m + 4), ..
 *     N = the same order from 0.0, adding only the terms with P(h) <= P(obs) * (1 + 2^-40) (the product rounded once), obs = n1
 *     p = N / S;  mid-p (midp = 1, Graffelman & Moreno 2013): p = (N - 0.5 * P(obs)) / S
 * The margin makes rounding-level near-ties count as ties. N adds a subset of S's terms in S's order and rounding is monotone, so
 * p <= 1 without a clamp, and p == 1.0 exactly when every term qualifies. p = 1 when n_r = 0 (also with midp); NaN when v = 0.
 * Floor: p = 0 when P(obs) underflows to 0.0 relative to the mode (PLINK reports smaller values there). A walk may stop a side
 * early, bit for bit the same (hwe.cuh): only terms under half an ulp of both sums are skipped.
 * Per-locus F (nullable f): F = 1 - (double)(2 v n1) / (double)(s (2 v - s)) with s = n1 + 2 n2 (one IEEE division and one
 * subtraction); NaN when v = 0 or s is 0 or 2 v. Multi-allelic rows (kgl_b200_upload_multi_allelic) hold only codes 0 and 3 and are
 * not biallelic genotypes: p and F are NaN there in every group.
 * Every result is per locus, so a locus-sharded multi-GPU caller runs each shard on its own GPU and needs no exchange.
 * Errors: those of kgl_b200_run_group_counts (KGL_B200_ERR_STATE before a genotype upload or for group == NULL without
 * super-population labels; KGL_B200_ERR_INVALID for n_groups outside 1..64 or a bad label), and KGL_B200_ERR_INVALID for midp other
 * than 0 / 1, a null output, or a group of 2^25 genomes or more. */
typedef struct kgl_b200_hardy_options {      /* zero-initialise; 16 bytes */
  const uint8_t* group;  uint32_t n_groups;  /* as kgl_b200_run_group_counts (NULL = super-population labels); pooled: all 0, 1 group */
  uint32_t midp;                             /* 0 = p, 1 = mid-p */
} kgl_b200_hardy_options;
int kgl_b200_run_hardy(kgl_b200_ctx* ctx, const kgl_b200_hardy_options* options, double* p_hwe /* [n_loci][n_groups] */,
                       double* f /* nullable, [n_loci][n_groups] */);
/* Variant QC: keep_out uint8[n_loci] = 1 for the loci that pass every filter whose threshold is not 0, *n_kept = their number.
 * Over ALL genomes, with the raw counts n0..n3 of kgl_b200_run_allele_count, v = n0 + n1 + n2, s = n1 + 2 n2:
 *     call rate (N - n3) / N >= min_call_rate       (PLINK --geno x is min_call_rate = 1 - x)
 *     MAF min(s, 2 v - s) / (2 v) >= min_maf        (v = 0 fails)
 * each one exact IEEE division of integers; and p >= min_hwe_p (kgl_b200_run_hardy with group / n_groups / midp) in every group with
 * v >= 1 (a group without calls does not vote). A threshold of 0 applies no filter (a zero-initialised struct filters nothing), and
 * min_hwe_p = 0 runs no test and needs no labels. keep_out is 0 for multi-allelic rows and where the input keep is 0. It is the mask
 * kgl_b200_pca_options.keep, kgl_b200_ld_options.keep and kgl_b200_fst_options.keep take, and kgl_b200_set_locus_filter takes it
 * too. Only the mask crosses PCIe (n_loci bytes). Errors: those of kgl_b200_run_hardy when min_hwe_p != 0 (STATE before a genotype
 * upload in any case), and KGL_B200_ERR_INVALID for a NaN threshold or one outside its range (min_call_rate and min_hwe_p in [0, 1],
 * min_maf in [0, 0.5]), midp other than 0 / 1, or a null output. */
typedef struct kgl_b200_qc_options {         /* zero-initialise; 48 bytes */
  const uint8_t* keep;                       /* uint8[n_loci] input mask, NULL = every locus */
  double min_call_rate;
  double min_maf;
  double min_hwe_p;
  const uint8_t* group;  uint32_t n_groups;  /* the groups of the test, as kgl_b200_hardy_options */
  uint32_t midp;
} kgl_b200_qc_options;
int kgl_b200_run_variant_qc(kgl_b200_ctx* ctx, const kgl_b200_qc_options* options, uint8_t* keep_out /* [n_loci] */, uint64_t* n_kept);
/* Terms of the exact test walked by the last kgl_b200_run_hardy / kgl_b200_run_variant_qc on this context, over all cells. */
uint64_t kgl_b200_last_hardy_terms(const kgl_b200_ctx* ctx);

/* CalcFWS::updateGenomeFWSMap (kga_PfEMP/kga_analysis_PfEMP_FWS.cpp:15-101): for each of n_bins allele-frequency bins
 * [lower[b], upper[b]) of AF column `pop` (the P7FrequencyFilter pair AF >= lower and not AF >= upper,
 * kgl_variant_filter_Pf7.cpp:20-66; a locus without AF is in no bin) the AlleleSummmary of every genome over the bin's loci:
 * genome_counts uint64[n_bins][n_genomes][4] = {referenceHomozygous_, minorHeterozygous_, minorHomozygous_, code 3},
 * bin_rows (nullable) uint64[n_bins] = loci in the bin. present_only != 0 restricts a bin to loci carried by at least one
 * genome -- the variants a filtered PopulationDB / VariantDBVariant holds (kgl_variant_db_variant.cpp:11-123).
 * Multi-allelic loci (kgl_b200_upload_multi_allelic): every listed allele is a variant of its own with its own AF (its element
 * of the record's Number=A list, kgl_variant_filter_Pf7.cpp:22-48) and is added to the bin it falls in; a genome has 0, 1 or 2
 * copies of it. Side cells with more than two variants (0xFF) do not record which alleles: no copy.
 * The per-variant half of CalcFWS (updateVariantFWSMap, :41-70) is kgl_b200_run_allele_count's locus_counts and, for those
 * loci, kgl_b200_run_multi_allele_count. */
int kgl_b200_run_binned_genome_counts(kgl_b200_ctx* ctx, uint32_t pop, uint32_t n_bins, const double* lower, const double* upper,
                                      int present_only, uint64_t* genome_counts, uint64_t* bin_rows);

/* HeteroHomoZygous::updateVariantAnalysisType for every genome (kga_PfEMP/kga_analysis_PfEMP_heterozygous.cpp:61-105), one raw
 * counting pass + the multi-allelic side cells: out uint64[n_genomes][7] = {total_variants_, snp_count_, indel_count_,
 * homozygous_minor_alleles_, heterozygous_minor_alleles_, heterozygous_reference_minor_alleles_, homozygous_reference_alleles_}
 * (the matrix path holds SNPs only: indel_count_ = 0; a code-3 cell of an ordinary row stands for other_allele_entries entries
 * of some other allele). kgl_b200_location_fis: HeteroHomoZygous::UpdateSampleLocation (:362-412) on those records -- host
 * arithmetic, no context: locations 0..n_locations-1 with their sample lists (location_begin[n_locations + 1] into
 * location_members; what Pf7SampleLocation::sampleRadius returns for the location), every genome's city and country location
 * (>= n_locations: none), its QC verdict (NULL: all pass); a city with fewer than min_location_samples QC-pass samples (the
 * reference's MINIMUM_LOCATION_SAMPLES_ = 20) falls back to the country; fis[g] = (H_exp - H_obs) / H_exp, 0 where undefined. */
int kgl_b200_run_hetero_homo(kgl_b200_ctx* ctx, int other_allele_entries, uint64_t* out);
int kgl_b200_location_fis(uint64_t n_genomes, const uint64_t* hetero_homo, uint32_t n_locations, const uint64_t* location_begin,
                          const uint32_t* location_members, const uint32_t* city_of_genome, const uint32_t* country_of_genome,
                          const uint8_t* qc_pass, uint32_t min_location_samples, double* fis);

/* Tensor-core variant of the pairwise path (BASELINE config 5, SURVEY 8d K5): the dosage Gram matrix
 * gram int32[n_genomes][n_genomes], gram[a][b] = sum over loci of g_a g_b with g in {0,1,2} (code 3 counts as 0: in the
 * variant DB "no entry at the offset" is the reference genotype, SURVEY Q5), contracted exactly in int8 x int8 -> int32 on
 * tcgen05; and the centred relationship matrix grm double[n][n] = sum_l (g_a - 2 p_l)(g_b - 2 p_l) with p the AF column
 * `pop` (absent AF -> 0), = gram - 2 (Gp)_a - 2 (Gp)_b + 4 sum p^2. Without code-3 cells gram[a][a] + gram[b][b] -
 * 2 gram[a][b] = IBS1 + 4 IBS0 of kgl_b200_run_ibs. n_loci < 2^29. */
int kgl_b200_run_gram(kgl_b200_ctx* ctx, int32_t* gram);
int kgl_b200_run_grm(kgl_b200_ctx* ctx, uint32_t pop, double* grm);

/* ---- resident / asynchronous building blocks (bench.py, multi-GPU drivers) ------------------------------------------ */
/* Enqueue the fused pass and return immediately; results stay in device buffers. The pass is spread over three streams -- the
 * streaming kernel on the context stream, the preparation of a pass and the tail of the pass before it on two internal
 * streams, where they run next to the streaming kernel -- so consecutive calls overlap. Every other entry point orders the
 * context stream after the pending tail before it does anything; kgl_b200_flush does only that (no host synchronisation), e.g.
 * before an event is recorded on the context stream to time a sequence of passes. The results of the last pass:
 * kgl_b200_inbreed_fetch (its per-genome Simple results; the pass ends an estimator begun with kgl_b200_inbreed_begin) and
 * kgl_b200_fetch_locus_counts. */
int kgl_b200_enqueue_count_and_inbreed(kgl_b200_ctx* ctx);
int kgl_b200_flush(kgl_b200_ctx* ctx);
/* Number of kernels this context has launched so far. */
uint64_t kgl_b200_launch_count(const kgl_b200_ctx* ctx);
/* Milliseconds the dominant streaming kernel (k_count_moments) took in the most recent enqueue/run, measured with
 * CUDA events around that launch on the context stream. Returns < 0 if none has run. Synchronises. */
float kgl_b200_last_stream_kernel_ms(kgl_b200_ctx* ctx);
/* The same measurement for every launch of that kernel since the last reset (up to 256), read after the fact so that
 * no host synchronisation lands inside a timed region. */
int kgl_b200_kernel_timer_reset(kgl_b200_ctx* ctx);
int kgl_b200_kernel_timer_read(kgl_b200_ctx* ctx, float* ms, uint32_t capacity, uint32_t* n);
/* Resident form of kgl_b200_run_ibs_tiles (count <= 8192 per call): the tiles stay in a device buffer that
 * kgl_b200_ibs_tiles_buffer exposes (uint32[count][64][64][4]) for a device-side gather. The ibs timer is the kernel timer
 * of the pairwise tile kernel (k_ibs_tiles). */
int kgl_b200_enqueue_ibs_tiles(kgl_b200_ctx* ctx, uint64_t first, uint64_t stride, uint64_t count);
/* The same for an explicit list of tiles, coords uint32[count][2] = (tile row, tile column) of 64-genome tiles (any cell of the
 * grid, count <= 8192): what a caller uses to deal the tiles of whole 256 x 256 blocks to a rank, the unit the tensor-core form
 * computes (kgl_gene_b200/shards.py: block_tile_coords). */
int kgl_b200_enqueue_ibs_tile_list(kgl_b200_ctx* ctx, uint64_t count, const uint32_t* coords);
int kgl_b200_run_ibs_tile_list(kgl_b200_ctx* ctx, uint64_t count, const uint32_t* coords, uint32_t* out);   /* any count; host result */
int kgl_b200_ibs_tiles_buffer(kgl_b200_ctx* ctx, void** device_ptr, uint64_t* n_u32);
/* Resident Gram contraction (the matrix stays on the device) and the milliseconds its tcgen05 kernel took. */
int kgl_b200_enqueue_gram(kgl_b200_ctx* ctx);
float kgl_b200_last_gram_kernel_ms(kgl_b200_ctx* ctx);
/* Multi-GPU form: rank r of R computes the 256 x 256 tiles r, r + R, ... of the upper triangle (first = r, stride = R) and
 * leaves the rest of its device matrix zero; a SUM all-reduce of kgl_b200_gram_buffer (int32[ld][ld], ld = n_genomes rounded
 * up to 256; 26 MB at 2,504 genomes -- SURVEY 8e) over the ranks assembles the matrix, kgl_b200_fetch_gram copies the
 * symmetric [n_genomes][n_genomes] result to the host. */
int kgl_b200_enqueue_gram_tiles(kgl_b200_ctx* ctx, uint64_t first, uint64_t stride);
int kgl_b200_gram_buffer(kgl_b200_ctx* ctx, void** device_ptr, uint64_t* n_int32, uint64_t* ld);
int kgl_b200_fetch_gram(kgl_b200_ctx* ctx, int32_t* gram);
int kgl_b200_ibs_timer_reset(kgl_b200_ctx* ctx);
int kgl_b200_ibs_timer_read(kgl_b200_ctx* ctx, float* ms, uint32_t capacity, uint32_t* n);
/* Copy the per-locus allele counts of the last fused pass to the host: uint32[n_loci][4]. */
int kgl_b200_fetch_locus_counts(kgl_b200_ctx* ctx, uint32_t* locus_counts);

/* Locus-sharded multi-GPU inbreeding: each rank holds a shard of the loci. begin() prepares `algorithm`;
 * accumulate() fills the context's per-genome partial-sum buffer (device, doubles) for the current iterate;
 * the caller all-reduces (SUM) that buffer across ranks (partials_buffer() exposes it); update() consumes the reduced
 * partials and reports whether the iteration has finished; fetch() copies the LocusResults to the host.
 * On one GPU run_inbreed() is exactly begin + (accumulate + update)* + fetch. After kgl_b200_enqueue_count_and_inbreed[_peer]
 * fetch() returns that pass's per-genome Simple results instead. */
int kgl_b200_inbreed_begin(kgl_b200_ctx* ctx, int algorithm, const kgl_b200_inbreed_options* options);
int kgl_b200_inbreed_accumulate(kgl_b200_ctx* ctx);
int kgl_b200_inbreed_partials_buffer(kgl_b200_ctx* ctx, void** device_ptr, uint64_t* n_doubles);
int kgl_b200_inbreed_update(kgl_b200_ctx* ctx, int* finished);
int kgl_b200_inbreed_fetch(kgl_b200_ctx* ctx, kgl_b200_locus_results* out);

/* The same locus-sharded step (allele counts + Simple, one rank per GPU of one node) with the exchange done by the step's
 * own kernel over NVLink peer memory instead of an all-reduce by the caller: every rank exports its exchange region once
 * (a CUDA IPC handle of KGL_B200_PEER_HANDLE_BYTES bytes, after its matrix is on the device), the caller gathers the
 * handles of all ranks (any transport) and attaches them; each kgl_b200_enqueue_count_and_inbreed_peer() then runs the fused
 * pass on the rank's shard and one kernel that signals the peers, waits for their partial sums, adds them in rank order and
 * applies the closed form. All ranks must call it the same number of times. Results: kgl_b200_inbreed_fetch,
 * kgl_b200_fetch_locus_counts. Replaces InbreedingAnalysis::processResults' per-genome fan-out over one population
 * (kga_analysis_inbreed_diploid.cpp:98-160) when that population is sharded by locus over GPUs.
 * Handles of regions exported by contexts of the SAME process (several GPUs driven by one process, or two contexts on one GPU)
 * are recognised by kgl_b200_peer_attach and mapped directly (CUDA IPC handles cannot be opened by their own process).
 * A peer that does not reach an exchange within the timeout (default 10 s; kgl_b200_peer_set_timeout_ms) makes that step
 * fail: its result rows read NaN / zero sums and kgl_b200_inbreed_fetch / kgl_b200_fetch_locus_counts return
 * KGL_B200_ERR_PEER until the regions have been exported and attached again. */
#define KGL_B200_PEER_HANDLE_BYTES 64
int kgl_b200_peer_export(kgl_b200_ctx* ctx, void* handle /* KGL_B200_PEER_HANDLE_BYTES */);
int kgl_b200_peer_attach(kgl_b200_ctx* ctx, uint32_t rank, uint32_t world, const void* handles /* world x KGL_B200_PEER_HANDLE_BYTES */);
int kgl_b200_peer_set_timeout_ms(kgl_b200_ctx* ctx, uint64_t milliseconds);
int kgl_b200_enqueue_count_and_inbreed_peer(kgl_b200_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* KGL_B200_H */
