/* kgl_oracle.c -- TEST INFRASTRUCTURE (see kgl_oracle.h). Plain-C restatement of the reference algorithms on the
 * flattened population. Compiled with -ffp-contract=off so every double operation rounds exactly like the
 * reference's (g++ -O3 on x86-64 does not contract either). OpenMP over genomes mirrors the reference's only
 * parallelism: one task per genome (kga_analysis_inbreed_diploid.cpp:117-150).
 *
 * Every function cites the reference file:line it follows; all paths are relative to /root/reference. */
#include "kgl_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

int kgl_oracle_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

static inline unsigned cell_code(const uint8_t* packed, size_t row_bytes, size_t locus, size_t genome) {
  const uint8_t* unit = packed + locus * row_bytes + (genome / 64) * 16;
  uint64_t lo, hi;
  memcpy(&lo, unit, 8);
  memcpy(&hi, unit + 8, 8);
  const unsigned bit = (unsigned)(genome % 64);
  return (unsigned)((lo >> bit) & 1u) | ((unsigned)((hi >> bit) & 1u) << 1);
}

static inline double clamp01(double x) { return x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x); }

/* AlleleFreqVector ctor + checkValidAlleleVector for ONE alternate allele
 * (kga_analysis_inbreed_freq.cpp:18-57,61-75): the frequency is the INFO float widened to double and clamped to
 * [0,1] (:47); the vector is valid iff it is non-empty (AF present) and sum - 1 <= 1e-5 (always true after clamp). */
static inline int allele_valid(float af, double* p) {
  if (isnan(af)) return 0;
  *p = clamp01((double)af);
  return 1;
}

/* majorAlleleFrequency(): clamp(1 - clamp(sum,0,1), 0, 1)  (kga_analysis_inbreed_freq.cpp:113-123). */
static inline double major_freq(double p) { return clamp01(1.0 - clamp01(p)); }

/* ---- multi-allelic loci (oracle/flat_io.h trailing section; set with kgl_oracle_set_multi, test infrastructure: not thread safe) */
static struct {
  size_t n_multi, n_genomes, n_loci, n_pop;
  uint32_t* rows; float* af; uint8_t* cells; int32_t* multi_of;
} g_multi;

void kgl_oracle_set_multi(size_t n_multi, const uint32_t* rows, const float* af, const uint8_t* cells, size_t n_pop,
                          size_t n_genomes, size_t n_loci) {
  free(g_multi.rows); free(g_multi.af); free(g_multi.cells); free(g_multi.multi_of);
  memset(&g_multi, 0, sizeof g_multi);
  if (n_multi == 0) return;
  g_multi.n_multi = n_multi; g_multi.n_genomes = n_genomes; g_multi.n_loci = n_loci; g_multi.n_pop = n_pop;
  g_multi.rows = (uint32_t*)malloc(n_multi * 4); memcpy(g_multi.rows, rows, n_multi * 4);
  g_multi.af = (float*)malloc(n_pop * n_multi * 3 * 4); memcpy(g_multi.af, af, n_pop * n_multi * 3 * 4);
  g_multi.cells = (uint8_t*)malloc(n_multi * n_genomes); memcpy(g_multi.cells, cells, n_multi * n_genomes);
  g_multi.multi_of = (int32_t*)malloc(n_loci * 4);
  for (size_t l = 0; l < n_loci; ++l) g_multi.multi_of[l] = -1;
  for (size_t m = 0; m < n_multi; ++m) g_multi.multi_of[rows[m]] = (int32_t)m;
}

static inline int multi_index(size_t locus) {
  return (g_multi.n_multi && locus < g_multi.n_loci) ? g_multi.multi_of[locus] : -1;
}

/* AlleleFreqVector of a multi-allelic locus for one super-population (kga_analysis_inbreed_freq.cpp:18-57): the alleles that have
 * a frequency for the population, in the order of the locus' variant array, each clamped to [0,1] (:47). slot[i] = allele slot. */
typedef struct { int n; int slot[3]; double p[3]; } allele_vector;
static allele_vector multi_vector(int m, size_t pop) {
  allele_vector v; v.n = 0;
  for (int a = 0; a < 3; ++a) {
    const float f = g_multi.af[(pop * g_multi.n_multi + (size_t)m) * 3 + (size_t)a];
    if (isnan(f)) continue;
    v.slot[v.n] = a; v.p[v.n] = clamp01((double)f); ++v.n;
  }
  return v;
}
static double vector_sum(const allele_vector* v) { double s = 0.0; for (int i = 0; i < v->n; ++i) s += v->p[i]; return s; }   /* sumAlleleFrequencies() :97 */
static int vector_valid(const allele_vector* v) {                                 /* checkValidAlleleVector() :61-75 */
  if (vector_sum(v) - 1.0 > 1.0e-05) return 0;                                    /* epsilon_class_ (freq.h) */
  return v->n > 0;
}
static int vector_find(const allele_vector* v, int slot) { for (int i = 0; i < v->n; ++i) if (v->slot[i] == slot) return i; return -1; }

/* alleleClassFrequencies(0.0) (:127-217 + normalize(), freq.h:54-63) of an allele vector: {majHom, majHet, minHom, minHet}. */
static void vector_class_freqs(const allele_vector* v, double out[4]) {
  const double inbreeding = 0.0;
  double sum_minor_freq = 0.0;
  for (int i = 0; i < v->n; ++i) sum_minor_freq += v->p[i];
  const double major_frequency = fmax(0.0, 1.0 - sum_minor_freq);                 /* :140 */
  double f[3];
  for (int i = 0; i < v->n; ++i) f[i] = (sum_minor_freq > 1.0) ? v->p[i] / sum_minor_freq : v->p[i];   /* :143-151 */
  double minor_homozygous = 0.0;
  for (int i = 0; i < v->n; ++i) minor_homozygous += (inbreeding * f[i]) + ((1.0 - inbreeding) * f[i] * f[i]);   /* :158 */
  double minor_heterozygous = 0.0;
  for (int i = 0; i < v->n; ++i)
    for (int j = i + 1; j < v->n; ++j) minor_heterozygous += (1.0 - inbreeding) * 2.0 * f[i] * f[j];              /* :170 */
  double major_homozygous = (inbreeding * major_frequency) + ((1.0 - inbreeding) * major_frequency * major_frequency);   /* :176 */
  double major_heterozygous = 0.0;
  for (int i = 0; i < v->n; ++i) major_heterozygous += (1.0 - inbreeding) * 2.0 * major_frequency * f[i];        /* :181 */
  major_homozygous = fmax(0.0, major_homozygous); major_heterozygous = fmax(0.0, major_heterozygous);
  minor_homozygous = fmax(0.0, minor_homozygous); minor_heterozygous = fmax(0.0, minor_heterozygous);
  const double sum_freqs = major_homozygous + major_heterozygous + minor_homozygous + minor_heterozygous;
  out[0] = major_homozygous / sum_freqs; out[1] = major_heterozygous / sum_freqs;
  out[2] = minor_homozygous / sum_freqs; out[3] = minor_heterozygous / sum_freqs;
}

size_t kgl_oracle_select_loci_pop(const uint32_t* offsets, const float* af, size_t n_loci, size_t pop,
                                  uint64_t lower, uint64_t upper, uint64_t spacing, uint64_t count,
                                  double min_af, double max_af, int mode, uint8_t* selected, size_t* last_index) {
  /* kgl_oracle_select_loci with the multi-allelic loci of kgl_oracle_set_multi: sum_frequencies = clamp(sum of the allele
   * frequencies, 0, 1) (minorAlleleFrequencies(), freq.cpp:107-111); af = the population's row of the main table. */
  size_t n_selected = 0;
  uint64_t previous_offset = 0;
  memset(selected, 0, n_loci);
  size_t l = 0;
  while (l < n_loci && offsets[l] < lower) ++l;
  for (; l < n_loci; ++l) {
    const uint64_t offset = offsets[l];
    if (mode == 0) { if (offset > upper) break; }
    else { if (n_selected >= count) break; }
    if (offset >= previous_offset + spacing || previous_offset == 0) {
      double sum_frequencies;
      const int m = multi_index(l);
      if (m >= 0) {
        const allele_vector v = multi_vector(m, pop);
        if (!vector_valid(&v)) continue;
        sum_frequencies = clamp01(vector_sum(&v));
      } else {
        double p;
        if (!allele_valid(af[l], &p)) continue;
        sum_frequencies = clamp01(p);
      }
      if (sum_frequencies == 0.0 || sum_frequencies < min_af || sum_frequencies > max_af) continue;
      previous_offset = offset;
      selected[l] = 1;
      if (last_index) *last_index = l;
      ++n_selected;
    }
  }
  return n_selected;
}

size_t kgl_oracle_select_loci(const uint32_t* offsets, const float* af, size_t n_loci,
                              uint64_t lower, uint64_t upper, uint64_t spacing, uint64_t count,
                              double min_af, double max_af, int mode, uint8_t* selected, size_t* last_index) {
  /* kga_analysis_inbreed_locus.cpp:21-72 (FromTo) and :105-156 (Count). */
  size_t n_selected = 0;
  uint64_t previous_offset = 0;
  memset(selected, 0, n_loci);
  size_t l = 0;
  while (l < n_loci && offsets[l] < lower) ++l;             /* getMap().lower_bound(lowerOffset)  (:26,:110) */
  for (; l < n_loci; ++l) {
    const uint64_t offset = offsets[l];
    if (mode == 0) { if (offset > upper) break; }             /* :33 */
    else { if (n_selected >= count) break; }                  /* :117 */
    if (offset >= previous_offset + spacing || previous_offset == 0) {   /* :38,:122 */
      double p;
      if (!allele_valid(af[l], &p)) continue;                /* :44,:128 */
      const double sum_frequencies = clamp01(p);             /* minorAlleleFrequencies()  :51 */
      if (sum_frequencies == 0.0 || sum_frequencies < min_af || sum_frequencies > max_af) continue;   /* :53-54 */
      previous_offset = offset;                              /* :61 */
      selected[l] = 1;
      if (last_index) *last_index = l;
      ++n_selected;
    }
  }
  return n_selected;
}

/* Per-genome sums over the loci (expected class frequencies, Ritland's locus sum). By default they are added locus by locus
 * in double, the reference's order and precision, which the golden cases match bit for bit. Over millions of loci that
 * sum drifts from the exact one by up to one rounding per locus, and terms that repeat (frequencies clipped to one value)
 * make the roundings add up; kgl_oracle_set_compensated_sums(1) adds them with Neumaier's compensation instead, for
 * comparisons with implementations whose sums are exact at that size (the device's fixed-point totals). */
static int g_compensated = 0;
void kgl_oracle_set_compensated_sums(int on) { g_compensated = on; }

typedef struct { double s, c; } oracle_sum;
static inline void sum_add(oracle_sum* a, double x) {
  if (!g_compensated) { a->s += x; return; }
  const double t = a->s + x;
  a->c += fabs(a->s) >= fabs(x) ? (a->s - t) + x : (x - t) + a->s;
  a->s = t;
}
static inline double sum_value(const oracle_sum* a) { return a->s + a->c; }

/* One classified locus of one genome: the information AlleleFreqInfo carries for the estimators. */
typedef struct { uint8_t cls; double first, second; } locus_term;
enum { CLS_MAJOR_HOM = 0, CLS_MAJOR_HET = 1, CLS_MINOR_HET = 2, CLS_MINOR_HOM = 3 };

/* generateFrequencies (kga_analysis_inbreed_freq.cpp:425-583) for one genome; returns the number of classified loci. */
static size_t generate_frequencies(const uint8_t* packed, size_t row_bytes, size_t n_loci, size_t genome,
                                   const float* af_pop, const uint8_t* sel_pop, int unphased, size_t pop,
                                   locus_term* terms, kgl_oracle_locus_results* r) {
  size_t n = 0;
  memset(r, 0, sizeof *r);
  oracle_sum f_major_homo = {0, 0}, f_major_hetero = {0, 0}, f_minor_homo = {0, 0}, f_minor_hetero = {0, 0};
  for (size_t l = 0; l < n_loci; ++l) {
    if (!sel_pop[l]) continue;                               /* locus_list holds only the selected loci (:439) */
    const int m = multi_index(l);
    if (m >= 0) {
      /* a locus with several alternate alleles: the general form of the classification (:452-543) */
      const allele_vector v = multi_vector(m, pop);
      if (!vector_valid(&v)) continue;                       /* :445-449 */
      const double q = clamp01(1.0 - clamp01(vector_sum(&v)));   /* majorAlleleFrequency() :113-123 */
      const uint8_t cell = g_multi.cells[(size_t)m * g_multi.n_genomes + genome];
      locus_term t;
      if (cell == 0) {                                       /* no variant at the offset (:521-541) */
        if (!(q > 0.01)) continue;
        t.cls = CLS_MAJOR_HOM; t.first = q; t.second = q;
      } else if (cell == 0xFF) {
        continue;                                            /* more than two variants: neither size() == 1 nor == 2 */
      } else {
        const int first = (cell & 15) - 1, second = (cell >> 4) - 1;
        const int i = first < 3 ? vector_find(&v, first) : -1;
        if (i < 0) continue;                                 /* the front variant is not in the AF list (:462) */
        if (second < 0) {                                    /* one variant: MAJOR_HETEROZYGOUS (:464-472) */
          t.cls = CLS_MAJOR_HET; t.first = v.p[i]; t.second = q;
        } else if (second == first && !unphased) {           /* front->homozygous(back): same allele, different phase (:476) */
          t.cls = CLS_MINOR_HOM; t.first = v.p[i]; t.second = v.p[i];
        } else {                                             /* different alleles, or the same allele unphased (Q6): :482-511 */
          const int j = second < 3 ? vector_find(&v, second) : -1;
          if (j < 0) continue;                               /* second minor not found (:500) */
          t.cls = CLS_MINOR_HET; t.first = v.p[i]; t.second = v.p[j];
        }
      }
      terms[n++] = t;
      double cf[4];
      vector_class_freqs(&v, cf);
      sum_add(&f_major_homo, cf[0]); sum_add(&f_major_hetero, cf[1]); sum_add(&f_minor_homo, cf[2]); sum_add(&f_minor_hetero, cf[3]);
      switch (t.cls) {
        case CLS_MINOR_HOM: ++r->minor_homo_count; break;
        case CLS_MAJOR_HET: ++r->major_hetero_count; break;
        case CLS_MINOR_HET: ++r->minor_hetero_count; break;
        default: ++r->major_homo_count; break;
      }
      continue;
    }
    double p;
    if (!allele_valid(af_pop[l], &p)) continue;              /* :445-449 */
    const double q = major_freq(p);
    const unsigned code = cell_code(packed, row_bytes, l, genome);
    locus_term t;
    if (code == 0) {                                         /* no variant at the offset (:521-541) */
      if (!(q > 0.01)) continue;                             /* minimum_major_frequency (:532-533) */
      t.cls = CLS_MAJOR_HOM; t.first = q; t.second = q;
    } else if (code == 1) {                                  /* one copy: MAJOR_HETEROZYGOUS (:464-472) */
      t.cls = CLS_MAJOR_HET; t.first = p; t.second = q;
    } else if (code == 2) {
      if (unphased) { t.cls = CLS_MINOR_HET; t.first = p; t.second = p; }   /* Q6: homozygous() needs differing phase (:476,:482-511) */
      else { t.cls = CLS_MINOR_HOM; t.first = p; t.second = p; }            /* :476-479 */
    } else {
      continue;                                              /* allele not in the AF list etc.: dropped (:462 never matches) */
    }
    terms[n++] = t;

    /* Statistics block (:549-579): alleleClassFrequencies(0.0) = unadjusted (:127-205) then normalize() (freq.h:54-63). */
    const double inbreeding = 0.0;
    const double sum_minor_freq = p;
    const double major_frequency = fmax(0.0, 1.0 - sum_minor_freq);        /* :140 */
    const double minor_frequency = (sum_minor_freq > 1.0) ? p / sum_minor_freq : p;   /* :143-151 */
    double minor_homozygous = 0.0;
    minor_homozygous += (inbreeding * minor_frequency) + ((1.0 - inbreeding) * minor_frequency * minor_frequency);   /* :158 */
    double minor_heterozygous = 0.0;                          /* one allele: no pairs (:166-174) */
    double major_homozygous = (inbreeding * major_frequency) + ((1.0 - inbreeding) * major_frequency * major_frequency); /* :176 */
    double major_heterozygous = 0.0;
    major_heterozygous += (1.0 - inbreeding) * 2.0 * major_frequency * minor_frequency;   /* :181 */
    major_homozygous = fmax(0.0, major_homozygous);           /* nonNegative() */
    major_heterozygous = fmax(0.0, major_heterozygous);
    minor_homozygous = fmax(0.0, minor_homozygous);
    minor_heterozygous = fmax(0.0, minor_heterozygous);
    const double sum_freqs = major_homozygous + major_heterozygous + minor_homozygous + minor_heterozygous;
    sum_add(&f_major_homo, major_homozygous / sum_freqs);     /* :553-556 */
    sum_add(&f_minor_homo, minor_homozygous / sum_freqs);
    sum_add(&f_major_hetero, major_heterozygous / sum_freqs);
    sum_add(&f_minor_hetero, minor_heterozygous / sum_freqs);
    switch (t.cls) {                                          /* :559-577 */
      case CLS_MINOR_HOM: ++r->minor_homo_count; break;
      case CLS_MAJOR_HET: ++r->major_hetero_count; break;
      case CLS_MINOR_HET: ++r->minor_hetero_count; break;
      default: ++r->major_homo_count; break;
    }
  }
  r->major_homo_freq = sum_value(&f_major_homo); r->major_hetero_freq = sum_value(&f_major_hetero);
  r->minor_homo_freq = sum_value(&f_minor_homo); r->minor_hetero_freq = sum_value(&f_minor_hetero);
  r->total_allele_count = n;                                  /* :548 */
  return n;
}

/* InbreedingCalculation::logLikelihood (kga_analysis_inbreed_calc.cpp:94-129). */
static double log_likelihood(double f, const locus_term* terms, size_t n) {
  double log_prob_sum = 0.0;
  const double small_prob = 1e-10;
  for (size_t i = 0; i < n; ++i) {
    double prob;
    if (terms[i].cls == CLS_MAJOR_HOM || terms[i].cls == CLS_MINOR_HOM) {
      const double freq_sqd = terms[i].first * terms[i].first;
      prob = (f * terms[i].first) + ((1.0 - f) * freq_sqd);
    } else {
      prob = 2 * (1.0 - f) * terms[i].first * terms[i].second;
    }
    prob = prob < small_prob ? small_prob : (prob > 1.0 ? 1.0 : prob);
    log_prob_sum += log(prob);
  }
  return log_prob_sum;
}

/* d/df and d2/df2 of logLikelihood over the terms that are not clamped, plus the clamp signature (numbers of clamped
 * homozygous / heterozygous terms). A clamped term is constant in f (calc.cpp:108,117), so it has no derivative. */
static void log_likelihood_deriv(double f, const locus_term* terms, size_t n, double* g1, double* g2, double* sig) {
  double d1 = 0.0, d2 = 0.0, chom = 0.0, chet = 0.0;
  const double small_prob = 1e-10;
  for (size_t i = 0; i < n; ++i) {
    const double a = terms[i].first;
    if (terms[i].cls == CLS_MAJOR_HOM || terms[i].cls == CLS_MINOR_HOM) {
      const double prob = (f * a) + ((1.0 - f) * (a * a));
      if (prob >= small_prob) {
        if (prob <= 1.0) { const double t = (1.0 - a) / (a + f * (1.0 - a)); d1 += t; d2 -= t * t; }
      } else chom += 1.0;
    } else {
      const double prob = 2 * (1.0 - f) * a * terms[i].second;
      if (prob >= small_prob && prob <= 1.0) { const double t = 1.0 / (1.0 - f); d1 -= t; d2 -= t * t; }
      else chet += 1.0;
    }
  }
  *g1 = d1; *g2 = d2; *sig = chom * 4294967296.0 + chet;
}

/* The maximum-likelihood inbreeding coefficient the reference's optimiser is after (kga_analysis_inbreed_calc.cpp:131-216).
 * The reference maximises the CLAMPED objective over [-1,1] with nlopt Nelder-Mead to xtol 1e-6 from random starts
 * (Q1,Q2). The clamp at 1e-10 (calc.cpp:98,108) is a numerical guard: left of the largest pole of a homozygous term that
 * term is constant, the objective gets a convex kink and can have extra local maxima there, and which one Nelder-Mead
 * returns depends on its random start. Parity is therefore defined against the maximiser over the FEASIBLE region -- the
 * f for which no homozygous probability is clamped -- where the objective is smooth and concave and the maximiser is
 * unique. It is located deterministically with a bracketed Newton iteration on dLL/df: a clamped homozygous term means
 * "left of the feasible region" (move right), otherwise the sign of dLL/df updates the bracket and a Newton step is
 * taken when it stays inside it (else bisection). Function-value searches (golden section, Nelder-Mead) cannot resolve
 * the maximiser below ~1e-8; the derivative can. The product (k_ll_step) runs the identical iteration. */
static double log_likelihood_argmax(const locus_term* terms, size_t n, double start) {
  if (n == 0) return 0.0;
  double a = -1.0, b = 1.0, x = start;
  if (!(x > a && x < b)) x = 0.0;
  const double tol = 1e-12;
  for (int it = 0; it < 200; ++it) {
    double g1, g2, sig;
    log_likelihood_deriv(x, terms, n, &g1, &g2, &sig);
    const int hom_clamped = sig >= 4294967296.0;
    if (hom_clamped || g1 > 0.0) a = x; else b = x;
    double nx = 0.5 * (a + b);
    int newton_converged = 0;
    if (!hom_clamped && g2 < 0.0) {
      const double cand = x - g1 / g2;
      /* a Newton step below the tolerance ends the search even when rounding puts it on the bracket's edge */
      if (fabs(cand - x) < tol) { nx = (cand > a && cand < b) ? cand : x; newton_converged = 1; }
      else if (cand > a && cand < b) nx = cand;
    }
    const int stop = newton_converged || fabs(nx - x) < tol || (b - a) < tol;
    x = nx;
    if (stop) break;
  }
  return x;
}

/* One EM sweep of processHallME (kga_analysis_inbreed_calc.cpp:257-285). */
static double hall_sweep(double inbreed_coefficient, const locus_term* terms, size_t n) {
  double expectation_sum = 0.0;
  for (size_t i = 0; i < n; ++i) {
    if (terms[i].cls == CLS_MAJOR_HOM || terms[i].cls == CLS_MINOR_HOM) {
      const double denominator = (inbreed_coefficient + ((1.0 - inbreed_coefficient) * terms[i].first));
      if (denominator != 0) expectation_sum += inbreed_coefficient / denominator;
    }
  }
  return expectation_sum / (double)n;
}

void kgl_oracle_inbreed(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                        const float* af, size_t n_pop, const uint8_t* selected, const uint8_t* superpop,
                        int unphased, int algorithm, const double* start, int sweeps,
                        kgl_oracle_locus_results* out) {
  kgl_oracle_inbreed_some(packed, row_bytes, n_genomes, n_loci, af, n_pop, selected, superpop, unphased, algorithm, start, sweeps,
                          NULL, n_genomes, out);
}

/* The same for a list of genomes (genomes == NULL: 0 .. n_some-1); out[i] belongs to genomes[i]. Every genome is an
 * independent task in the reference (kga_analysis_inbreed_diploid.cpp:117-150), so a subset is exact for its members. */
void kgl_oracle_inbreed_some(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                             const float* af, size_t n_pop, const uint8_t* selected, const uint8_t* superpop,
                             int unphased, int algorithm, const double* start, int sweeps,
                             const uint32_t* genomes, size_t n_some, kgl_oracle_locus_results* out) {
  (void)n_pop; (void)n_genomes;
#pragma omp parallel
  {
    locus_term* terms = (locus_term*)malloc(sizeof(locus_term) * (n_loci ? n_loci : 1));
#pragma omp for schedule(dynamic, 1)
    for (long gi = 0; gi < (long)n_some; ++gi) {
      const size_t g = genomes ? (size_t)genomes[gi] : (size_t)gi;
      const size_t k = superpop[g];
      kgl_oracle_locus_results r;
      const size_t n = generate_frequencies(packed, row_bytes, n_loci, g, af + k * n_loci, selected + k * n_loci,
                                            unphased, k, terms, &r);
      switch (algorithm) {
        case KGL_ORACLE_SIMPLE: {                              /* processSimple (calc.cpp:319-365) */
          double homozygous_inbreeding = 0.0;
          if (r.total_allele_count > 0) {
            const double observed_homozygous = (double)(r.minor_homo_count + r.major_homo_count);
            const double expected_homozygous = r.minor_homo_freq + r.major_homo_freq;
            homozygous_inbreeding = (observed_homozygous - expected_homozygous) / ((double)r.total_allele_count - expected_homozygous);
          }
          r.inbred_allele_sum = homozygous_inbreeding;
        } break;
        case KGL_ORACLE_RITLAND: {                             /* processRitlandLocus (calc.cpp:375-431) */
          const double minimum_frequency = 0.001;
          size_t sum_allele = 0;
          oracle_sum locus_allele_sum = {0, 0};
          for (size_t i = 0; i < n; ++i) {
            if (terms[i].cls == CLS_MAJOR_HOM || terms[i].cls == CLS_MINOR_HOM) {
              if (terms[i].first > minimum_frequency) {
                const double ratio = (1.0 / terms[i].first);
                sum_add(&locus_allele_sum, ratio);
                sum_add(&locus_allele_sum, -1.0);
                ++sum_allele;
              }
            } else {
              sum_add(&locus_allele_sum, -1.0);
              ++sum_allele;
            }
          }
          r.inbred_allele_sum = (sum_allele > 0 ? sum_value(&locus_allele_sum) / (double)sum_allele : 0.0);
        } break;
        case KGL_ORACLE_HALLME: {                              /* processHallME (calc.cpp:226-307); Q1: 50 sweeps */
          double f = start ? start[g] : 0.25;
          if (n == 0) { r.inbred_allele_sum = 0.0 / 0.0; break; }   /* 0/0 in :285, as the reference */
          if (sweeps >= 0) {
            for (int s = 0; s < sweeps; ++s) f = hall_sweep(f, terms, n);
          } else {
            for (int s = 0; s < 100000; ++s) { const double nf = hall_sweep(f, terms, n); const int done = fabs(nf - f) < 1e-15; f = nf; if (done) break; }
          }
          r.inbred_allele_sum = f;
        } break;
        default: {                                             /* processLogLikelihood (calc.cpp:154-216) */
          double simple = 0.0;                                 /* start: the Simple estimate (calc.cpp:344) */
          if (r.total_allele_count > 0) {
            const double oh = (double)(r.minor_homo_count + r.major_homo_count), eh = r.minor_homo_freq + r.major_homo_freq;
            simple = (oh - eh) / ((double)r.total_allele_count - eh);
          }
          r.inbred_allele_sum = log_likelihood_argmax(terms, n, simple);
        } break;
      }
      out[gi] = r;
    }
    free(terms);
  }
}

void kgl_oracle_loglik_grid(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                            const float* af, size_t n_pop, const uint8_t* selected, const uint8_t* superpop,
                            int unphased, const double* grid, size_t n_grid, double* out) {
  (void)n_pop;
#pragma omp parallel
  {
    locus_term* terms = (locus_term*)malloc(sizeof(locus_term) * (n_loci ? n_loci : 1));
#pragma omp for schedule(dynamic, 1)
    for (long gi = 0; gi < (long)n_genomes; ++gi) {
      const size_t g = (size_t)gi, k = superpop[g];
      kgl_oracle_locus_results r;
      const size_t n = generate_frequencies(packed, row_bytes, n_loci, g, af + k * n_loci, selected + k * n_loci, unphased, k, terms, &r);
      for (size_t i = 0; i < n_grid; ++i) out[g * n_grid + i] = log_likelihood(grid[i], terms, n);
    }
    free(terms);
  }
}

void kgl_oracle_allele_count(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                             uint32_t* locus_counts, uint64_t* genome_counts) {
  /* The byte-at-a-time switch of kgl_variant_db_variant.cpp:142-163 / :196-217, on 2-bit cells. Loci are dealt to the
   * threads; every thread keeps its own per-genome counters (integer sums: the order does not matter). */
  memset(locus_counts, 0, n_loci * 4 * sizeof(uint32_t));
  memset(genome_counts, 0, n_genomes * 4 * sizeof(uint64_t));
#pragma omp parallel
  {
    uint64_t* mine = (uint64_t*)calloc(n_genomes * 4 + 1, sizeof(uint64_t));
#pragma omp for schedule(static)
    for (long li = 0; li < (long)n_loci; ++li) {
      const size_t l = (size_t)li;
      for (size_t g = 0; g < n_genomes; ++g) {
        const unsigned c = cell_code(packed, row_bytes, l, g);
        ++locus_counts[l * 4 + c];
        ++mine[g * 4 + c];
      }
    }
#pragma omp critical
    for (size_t i = 0; i < n_genomes * 4; ++i) genome_counts[i] += mine[i];
    free(mine);
  }
}

void kgl_oracle_ibs(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci, uint32_t* out) {
  uint8_t* codes = (uint8_t*)malloc(n_genomes * n_loci + 1);
  for (size_t l = 0; l < n_loci; ++l)
    for (size_t g = 0; g < n_genomes; ++g) codes[g * n_loci + l] = (uint8_t)cell_code(packed, row_bytes, l, g);
#pragma omp parallel for schedule(dynamic, 1)
  for (long ai = 0; ai < (long)n_genomes; ++ai) {
    const size_t a = (size_t)ai;
    for (size_t b = 0; b < n_genomes; ++b) {
      uint32_t c[4] = {0, 0, 0, 0};
      const uint8_t* ga = codes + a * n_loci;
      const uint8_t* gb = codes + b * n_loci;
      for (size_t l = 0; l < n_loci; ++l) {
        if (ga[l] == 3 || gb[l] == 3) continue;
        const int d = abs((int)ga[l] - (int)gb[l]);
        ++c[2 - d];                                           /* |d|=0 -> IBS2, 1 -> IBS1, 2 -> IBS0 */
        ++c[3];
      }
      memcpy(out + (a * n_genomes + b) * 4, c, sizeof c);
    }
  }
  free(codes);
}

/* 64 x 64 bit-matrix transpose (recursive block swap): on return bit j of a[i] is bit i of the old a[j]. */
static void transpose64(uint64_t a[64]) {
  uint64_t m = 0x00000000FFFFFFFFULL;
  for (int j = 32; j != 0; j >>= 1, m ^= (m << j)) {
    for (int k = 0; k < 64; k = (k + j + 1) & ~j) {
      const uint64_t t = ((a[k] >> j) ^ a[k + j]) & m;
      a[k] ^= t << j;
      a[k + j] ^= t;
    }
  }
}

/* Popcount restatement of pairwise IBS "for scale" (SURVEY 8c/8d): genome-major thermometer bit-planes over 64-locus words,
 * X = (g >= 1), Y = (g == 2), V = (g != 3); for a pair dX = Xa ^ Xb, dY = Ya ^ Yb, v = Va & Vb:
 *   IBS0 = popc(dX & dY & v), IBS2 = popc(~(dX | dY) & v), IBS1 = popc(v) - IBS0 - IBS2.
 * Independent of the naive loop above (which it is checked against in tests/) and of the device kernel's two-plane / carry-save
 * form. out u32[row_end - row_begin][N][4]. */
void kgl_oracle_ibs_band_popcount(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci,
                                  size_t row_begin, size_t row_end, uint32_t* out) {
  const size_t n_words = (n_loci + 63) / 64, units = row_bytes / 16;
  uint64_t* X = (uint64_t*)calloc(n_genomes * n_words + 1, 8);
  uint64_t* Y = (uint64_t*)calloc(n_genomes * n_words + 1, 8);
  uint64_t* V = (uint64_t*)calloc(n_genomes * n_words + 1, 8);
#pragma omp parallel for schedule(dynamic, 1)
  for (long ui = 0; ui < (long)units; ++ui) {
    const size_t u = (size_t)ui;
    uint64_t lo[64], hi[64];
    for (size_t w = 0; w < n_words; ++w) {
      for (size_t i = 0; i < 64; ++i) {
        const size_t l = w * 64 + i;
        if (l < n_loci) { memcpy(&lo[i], packed + l * row_bytes + u * 16, 8); memcpy(&hi[i], packed + l * row_bytes + u * 16 + 8, 8); }
        else { lo[i] = ~0ULL; hi[i] = ~0ULL; }                       /* beyond the last locus: code 3, never valid */
      }
      transpose64(lo); transpose64(hi);                               /* now word b = the 64 loci of genome 64u + b */
      for (size_t b = 0; b < 64 && u * 64 + b < n_genomes; ++b) {
        const uint64_t l0 = lo[b], h0 = hi[b], valid = ~(l0 & h0);
        X[(u * 64 + b) * n_words + w] = (l0 | h0) & valid;
        Y[(u * 64 + b) * n_words + w] = h0 & valid;
        V[(u * 64 + b) * n_words + w] = valid;
      }
    }
  }
#pragma omp parallel for schedule(dynamic, 1)
  for (long ai = (long)row_begin; ai < (long)row_end; ++ai) {
    const size_t a = (size_t)ai;
    const uint64_t *xa = X + a * n_words, *ya = Y + a * n_words, *va = V + a * n_words;
    for (size_t b = 0; b < n_genomes; ++b) {
      const uint64_t *xb = X + b * n_words, *yb = Y + b * n_words, *vb = V + b * n_words;
      uint64_t c0 = 0, c2 = 0, cv = 0;
      for (size_t w = 0; w < n_words; ++w) {
        const uint64_t dx = xa[w] ^ xb[w], dy = ya[w] ^ yb[w], v = va[w] & vb[w];
        c0 += (uint64_t)__builtin_popcountll(dx & dy & v);
        c2 += (uint64_t)__builtin_popcountll(~(dx | dy) & v);
        cv += (uint64_t)__builtin_popcountll(v);
      }
      uint32_t* o = out + ((a - row_begin) * n_genomes + b) * 4;
      o[0] = (uint32_t)c0; o[1] = (uint32_t)(cv - c0 - c2); o[2] = (uint32_t)c2; o[3] = (uint32_t)cv;
    }
  }
  free(X); free(Y); free(V);
}

/* K5 checker: dosage Gram matrix S[a][b] = sum_l g_al g_bl with g in {0,1,2}, code 3 -> 0 (the DB's own convention: no entry at
 * an offset = reference, SURVEY Q5), and the centred form C[a][b] = sum_l (g_al - 2 p_l)(g_bl - 2 p_l) with p = clamp(AF,0,1)
 * of one population column (absent AF -> 0). No reference routine exists (SURVEY 8c/8d: the GRM variant is ours). */
void kgl_oracle_gram(const uint8_t* packed, size_t row_bytes, size_t n_genomes, size_t n_loci, const float* af_pop /* nullable */,
                     int32_t* gram, double* grm /* nullable */) {
  uint8_t* d = (uint8_t*)malloc(n_genomes * n_loci + 1);
  double* p = (double*)malloc((n_loci + 1) * sizeof(double));
  for (size_t l = 0; l < n_loci; ++l) {
    p[l] = (af_pop && !isnan(af_pop[l])) ? clamp01((double)af_pop[l]) : 0.0;
    for (size_t g = 0; g < n_genomes; ++g) {
      const unsigned c = cell_code(packed, row_bytes, l, g);
      d[g * n_loci + l] = (uint8_t)(c == 3 ? 0 : c);
    }
  }
#pragma omp parallel for schedule(dynamic, 1)
  for (long ai = 0; ai < (long)n_genomes; ++ai) {
    const size_t a = (size_t)ai;
    for (size_t b = 0; b < n_genomes; ++b) {
      const uint8_t* ga = d + a * n_loci;
      const uint8_t* gb = d + b * n_loci;
      long long s = 0;
      double c = 0.0;
      for (size_t l = 0; l < n_loci; ++l) {
        s += (long long)ga[l] * gb[l];
        if (grm) c += ((double)ga[l] - 2.0 * p[l]) * ((double)gb[l] - 2.0 * p[l]);
      }
      gram[a * n_genomes + b] = (int32_t)s;
      if (grm) grm[a * n_genomes + b] = c;
    }
  }
  free(d); free(p);
}

static inline uint64_t mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}

void kgl_oracle_synth_genotypes(uint64_t seed, size_t n_genomes, size_t n_loci, size_t locus_base,
                                const float* af, size_t n_pop, const uint8_t* superpop,
                                const double* inbreeding, double missing_rate, uint8_t* packed, size_t row_bytes) {
  (void)n_pop;
  const uint64_t miss_threshold = (uint64_t)(missing_rate * 16777216.0);
  memset(packed, 0, n_loci * row_bytes);
#pragma omp parallel for schedule(static)
  for (long li = 0; li < (long)n_loci; ++li) {
    const size_t l = (size_t)li;
    uint8_t* row = packed + l * row_bytes;
    for (size_t g = 0; g < n_genomes; ++g) {
      const float a = af[(size_t)superpop[g] * n_loci + l];
      const double p = isnan(a) ? 0.0 : clamp01((double)a);
      const double q = 1.0 - p, F = inbreeding[g];
      const double pq = p * q;
      const double t0 = q * q + F * pq;
      const double t1 = t0 + (2.0 * pq) * (1.0 - F);
      const uint64_t h1 = mix64(seed ^ ((uint64_t)(locus_base + l) << 32) ^ (uint64_t)g);
      const uint64_t h2 = mix64(h1 ^ 0xD6E8FEB86659FD93ULL);
      const double u = (double)(h1 >> 11) * (1.0 / 9007199254740992.0);
      unsigned code = (unsigned)(u >= t0) + (unsigned)(u >= t1);
      if ((h2 >> 40) < miss_threshold) code = 3;
      uint8_t* unit = row + (g / 64) * 16;
      const unsigned bit = (unsigned)(g % 64);
      if (code & 1u) unit[bit / 8] |= (uint8_t)(1u << (bit % 8));
      if (code & 2u) unit[8 + bit / 8] |= (uint8_t)(1u << (bit % 8));
    }
  }
}
