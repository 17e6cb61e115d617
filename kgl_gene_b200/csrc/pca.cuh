// pca.cuh -- the variance-standardised relationship operator Z^T Z as exact integer Gram runs (kgl_b200_run_grm_product,
// kgl_b200_run_pca).
//
// z_lg = (g_lg - 2 p_l) d_l over the used loci U (keep[l] != 0, 0 < p_l < 1) and the cells that are not coded 3, 0 elsewhere;
// d_l = 1 / sqrt(2 p_l (1 - p_l)), p_l = (n1 + 2 n2) / (2 (n0 + n1 + n2)) from the raw per-locus counts.
// A product with a thin block F (b <= 48 columns over a K index) runs on k_gram_i8 with F written as base-4 digits:
//   per column j, s_j = the largest integer with max |F 2^s_j| < 2^29, F_q = min(rint(F 2^s_j), 2^29 - 1) + 2^29 in [0, 2^30)
//   at the K positions that count (0 at the others) = 15 digits of 2 bits. One 256-row B block holds 16 columns x 15 digit rows
//   (row 15 jj + d of column jj), the indicator row 240 (code 1 at the positions that count) and 15 zero rows. The digit table
//   0x03020100 reads a digit as its value, so sum_d 4^d acc[15 jj + d] - 2^29 acc[240] = sum_k A_k (F_q,k - 2^29) exactly in
//   int64: every int32 accumulator is <= 2 * 3 * K < 2^31 for K < 2^28.
//   pass 1 (K = genomes): GX = G X, CX = C X on the loci-major codes (G dosage, C the code-3 indicator), S = sum_g X_q; then
//     Y_l = d_l 2^-s (GX - 2 p_l (S - CX)),  W_l = d_l Y_l,  V_l = 2 p_l W_l   (0 outside U)
//   pass 2 (K = loci, the positions that count are U): GW and CV on the genome-major codes, T = sum_l V_q;
//     X'_g = 2^-t GW - 2^-t' (T - CV)
// Every contraction is an exact integer; the double arithmetic after it is a fixed sequence of IEEE operations written with
// explicit _rn intrinsics (no contraction into fused multiply-adds), so the result does not depend on the schedule and a host
// restatement reproduces it bit for bit (tests/pca_oracle.py).
#pragma once
#include "gram_i8.cuh"

#include <cmath>
#include <vector>

namespace kgl {

constexpr int kPcaDigits = 15, kPcaColsPerBlock = 16, kPcaIndicatorRow = 240;
constexpr int kPcaMaxCols = 48;
constexpr uint32_t kPcaTableDigit = 0x03020100u;     // a B digit (code 0..3) is its own value
constexpr double kPcaQMax = 536870911.0;             // 2^29 - 1
constexpr long long kPcaOffset = 1ll << 29;

// s_j from the bits of max |F| over the column (a non-negative double orders like its bit pattern).
__device__ __forceinline__ int pca_shift(unsigned long long max_bits) {
  const double m = __longlong_as_double((long long)max_bits);
  if (m == 0.0) return 0;
  int e = 0;
  frexp(m, &e);                                      // m = f 2^e, f in [0.5, 1): m 2^(29 - e) in [2^28, 2^29)
  return 29 - e;
}

__device__ __forceinline__ long long pca_quant(double x, int s) { return (long long)fmin(rint(ldexp(x, s)), kPcaQMax); }

// sum_k A_k (F_q,k - 2^29) of column jj of B block cb, from one output row of a digit Gram run
__device__ __forceinline__ long long pca_digit_sum(const int32_t* row, uint32_t cb, uint32_t jj) {
  const int32_t* a = row + (size_t)cb * kGramN;
  long long v = 0;
#pragma unroll
  for (int d = kPcaDigits - 1; d >= 0; --d) v = (v << 2) + a[jj * kPcaDigits + d];
  return v - ((long long)a[kPcaIndicatorRow] << 29);
}

// Loci-major 2-bit codes in the row-block-major layout of gram_i8.cuh (row = locus, K = genomes, code 3 kept), from the
// uploaded planes: word w of row l = genomes 16 w .. 16 w + 15. Every word of the layout is written (zeros past the genomes).
__global__ void __launch_bounds__(256)
k_codes16_loci(const uint32_t* __restrict__ packed, uint64_t units, uint64_t rows, uint64_t k_stages, uint32_t* __restrict__ codes) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * k_stages * 8) return;
  const uint64_t wl = idx & 7, r = (idx >> 3) & 127, rest = idx >> 10;
  const uint64_t ks = rest % k_stages, rb = rest / k_stages;
  const uint64_t row = rb * 128 + r, w = ks * 8 + wl;
  uint32_t out = 0;
  if (w < units * 4) {
    const uint32_t* u = packed + row * units * 4 + (w >> 2) * 4;
    const uint32_t sh = (uint32_t)(w & 1) * 16;
    uint32_t a = (u[(w >> 1) & 1] >> sh) & 0xFFFFu, b = (u[2 + ((w >> 1) & 1)] >> sh) & 0xFFFFu;
    a = (a | (a << 8)) & 0x00FF00FFu; a = (a | (a << 4)) & 0x0F0F0F0Fu; a = (a | (a << 2)) & 0x33333333u; a = (a | (a << 1)) & 0x55555555u;
    b = (b | (b << 8)) & 0x00FF00FFu; b = (b | (b << 4)) & 0x0F0F0F0Fu; b = (b | (b << 2)) & 0x33333333u; b = (b | (b << 1)) & 0x55555555u;
    out = a | (b << 1);
  }
  codes[idx] = out;                                  // idx == gram_code_index(row, w, k_stages)
}

// p_l, d_l and the used-locus flag from the raw per-locus counts; n_used += |U|.
__global__ void __launch_bounds__(256)
k_pca_loci(const uint32_t* __restrict__ counts, const uint8_t* __restrict__ keep, uint64_t n_loci, double* __restrict__ p_out,
           double* __restrict__ d_out, uint8_t* __restrict__ used, unsigned long long* __restrict__ n_used) {
  const uint64_t l = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool u = false;
  if (l < n_loci) {
    const uint32_t n0 = counts[4 * l], n1 = counts[4 * l + 1], n2 = counts[4 * l + 2];
    const uint64_t v = (uint64_t)n0 + n1 + n2;
    double p = 0.0, d = 0.0;
    if ((keep == nullptr || keep[l] != 0) && v > 0) {
      p = __ddiv_rn((double)((uint64_t)n1 + 2ull * n2), (double)(2 * v));
      if (p > 0.0 && p < 1.0) {
        u = true;
        d = __ddiv_rn(1.0, __dsqrt_rn(__dmul_rn(__dmul_rn(2.0, p), __dsub_rn(1.0, p))));
      } else {
        p = 0.0;
      }
    }
    p_out[l] = p; d_out[l] = d; used[l] = u ? 1 : 0;
  }
  const uint32_t mask = __ballot_sync(0xFFFFFFFFu, u);
  if ((threadIdx.x & 31) == 0 && mask) atomicAdd(n_used, (unsigned long long)__popc(mask));
}

// max_bits[j] = bits of max_k |F[k][j]|, F row-major [rows][cols]; grid.y = column.
__global__ void __launch_bounds__(256)
k_pca_colmax(const double* __restrict__ F, uint64_t rows, uint32_t cols, unsigned long long* __restrict__ max_bits) {
  const uint32_t j = blockIdx.y;
  unsigned long long m = 0;
  for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < rows; k += (uint64_t)gridDim.x * blockDim.x)
    m = max(m, (unsigned long long)__double_as_longlong(fabs(F[k * cols + j])));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(max_bits + j, m);
}

// Digit rows of F [k_count][cols] (cols a multiple of 16) as the B operand: block cb = columns 16 cb .. 16 cb + 15, K = k_stages x
// 128 positions. A position counts when it is < k_count and, with `used`, used[k] != 0. sums[j] += sum_k F_q,k - 2^29 over the
// positions that count (two's complement in the uint64). Thread = (column j, a stride of 16-position words).
__global__ void __launch_bounds__(256)
k_pca_digits(const double* __restrict__ F, uint64_t k_count, uint32_t cols, const unsigned long long* __restrict__ max_bits,
             const uint8_t* __restrict__ used, uint64_t k_stages, uint32_t* __restrict__ digits, unsigned long long* __restrict__ sums) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, n_threads = (uint64_t)gridDim.x * blockDim.x / cols * cols;
  if (t >= n_threads) return;
  const uint32_t j = (uint32_t)(t % cols), cb = j / kPcaColsPerBlock, jj = j % kPcaColsPerBlock;
  const int s = pca_shift(max_bits[j]);
  const uint64_t n_words = k_stages * 8;
  long long sum = 0;
  for (uint64_t w = t / cols; w < n_words; w += n_threads / cols) {
    uint32_t dig[kPcaDigits] = {}, ind = 0;
    for (int i = 0; i < 16; ++i) {
      const uint64_t k = w * 16 + i;
      if (k >= k_count || (used && used[k] == 0)) continue;
      const long long q = pca_quant(F[k * cols + j], s);
      sum += q;
      const uint32_t f = (uint32_t)(q + kPcaOffset);
#pragma unroll
      for (int d = 0; d < kPcaDigits; ++d) dig[d] |= ((f >> (2 * d)) & 3u) << (2 * i);
      ind |= 1u << (2 * i);
    }
    const uint64_t row0 = (uint64_t)cb * kGramN;
#pragma unroll
    for (int d = 0; d < kPcaDigits; ++d) digits[gram_code_index(row0 + jj * kPcaDigits + d, w, k_stages)] = dig[d];
    if (jj == 0) {
      digits[gram_code_index(row0 + kPcaIndicatorRow, w, k_stages)] = ind;
      for (uint64_t r = kPcaIndicatorRow + 1; r < (uint64_t)kGramN; ++r) digits[gram_code_index(row0 + r, w, k_stages)] = 0u;
    }
  }
  atomicAdd(sums + j, (unsigned long long)sum);
}

// Pass 1, rows [row0, row0 + n_rows) of the loci, from the GX (and CX) digit runs (acc rows relative to row0, pitch ld): Y [L][cols]
// when Y is given (the loadings), otherwise WV [L][2 cols] = W | V, pass 2's input.
__global__ void __launch_bounds__(256)
k_pca_recombine_loci(const int32_t* __restrict__ acc_g, const int32_t* __restrict__ acc_c, uint64_t ld, uint64_t row0, uint64_t n_rows,
                     uint32_t cols, const double* __restrict__ p, const double* __restrict__ dl, const uint8_t* __restrict__ used,
                     const unsigned long long* __restrict__ max_bits, const unsigned long long* __restrict__ sums, double* __restrict__ Y,
                     double* __restrict__ WV) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_rows * cols) return;
  const uint64_t r = idx / cols, l = row0 + r;
  const uint32_t j = (uint32_t)(idx % cols), cb = j / kPcaColsPerBlock, jj = j % kPcaColsPerBlock;
  double y = 0.0, w = 0.0, v = 0.0;
  if (used[l]) {
    const long long gx = pca_digit_sum(acc_g + r * ld, cb, jj);
    const long long cx = acc_c ? pca_digit_sum(acc_c + r * ld, cb, jj) : 0;
    const double p2 = __dmul_rn(2.0, p[l]);
    const double num = __dsub_rn((double)gx, __dmul_rn(p2, (double)((long long)sums[j] - cx)));
    y = __dmul_rn(dl[l], ldexp(num, -pca_shift(max_bits[j])));
    w = __dmul_rn(dl[l], y);
    v = __dmul_rn(p2, w);
  }
  if (Y) {
    Y[l * cols + j] = y;
  } else {
    WV[l * 2 * cols + j] = w;
    WV[l * 2 * cols + cols + j] = v;
  }
}

// Pass 2: out [n_genomes][cols] = 2^-t GW - 2^-t' (T - CV); acc rows = genomes with pitch ld, W in blocks 0 .., V in blocks
// cols / 16 ..; max_bits / sums over the 2 cols columns of WV.
__global__ void __launch_bounds__(256)
k_pca_recombine_genomes(const int32_t* __restrict__ acc, uint64_t ld, uint64_t n_genomes, uint32_t cols, int with_c,
                        const unsigned long long* __restrict__ max_bits, const unsigned long long* __restrict__ sums, double* __restrict__ out) {
  const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_genomes * cols) return;
  const uint64_t g = idx / cols;
  const uint32_t j = (uint32_t)(idx % cols), cb = j / kPcaColsPerBlock, jj = j % kPcaColsPerBlock;
  const int32_t* row = acc + g * ld;
  const long long gw = pca_digit_sum(row, cb, jj);
  const long long cv = with_c ? pca_digit_sum(row, cols / kPcaColsPerBlock + cb, jj) : 0;
  out[idx] = __dsub_rn(ldexp((double)gw, -pca_shift(max_bits[j])),
                       ldexp((double)((long long)sums[cols + j] - cv), -pca_shift(max_bits[cols + j])));
}

// ---- host side of the subspace iteration: plain double, a fixed sequence of operations, so every run is reproducible ----

inline uint64_t pca_mix64(uint64_t z) {              // splitmix64 finaliser (synth.py mix64)
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// Start block entry (genome g, column j): Box-Muller on two splitmix64 draws keyed by (seed, g, j) -- a pure function of the
// three, whatever the population's size or the block's width.
inline double pca_start_entry(uint64_t seed, uint64_t g, uint64_t j) {
  const uint64_t h1 = pca_mix64(pca_mix64(seed) ^ ((g << 8) | j)), h2 = pca_mix64(h1 ^ 0xD6E8FEB86659FD93ull);
  const double u1 = (double)((h1 >> 11) + 1) * 0x1.0p-53, u2 = (double)(h2 >> 11) * 0x1.0p-53;
  return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2);
}

// a[k..n)[j0..b) -= beta v (v^T a[k..n)[j0..b)) for the reflector (v, beta) that starts at row k: two passes over the rows of the
// row-major block, all columns' dot products in the first.
inline void pca_reflect(std::vector<double>& a, uint64_t n, uint32_t b, const double* v, double beta, uint64_t k, uint32_t j0,
                        std::vector<double>& dot) {
  std::fill(dot.begin(), dot.end(), 0.0);
  for (uint64_t i = k; i < n; ++i) {
    const double* row = &a[i * b];
    for (uint32_t j = j0; j < b; ++j) dot[j] += v[i] * row[j];
  }
  for (uint32_t j = j0; j < b; ++j) dot[j] *= beta;
  for (uint64_t i = k; i < n; ++i) {
    double* row = &a[i * b];
    for (uint32_t j = j0; j < b; ++j) row[j] -= dot[j] * v[i];
  }
}

// Orthonormal basis of the columns of a [n][b] (row-major) by Householder QR; a is replaced by the thin Q.
inline void pca_orth(std::vector<double>& a, uint64_t n, uint32_t b) {
  std::vector<double> v((size_t)b * n), beta(b, 0.0), dot(b);
  for (uint32_t k = 0; k < b; ++k) {                   // reflector k zeroes column k below the diagonal
    double* vk = &v[(size_t)k * n];
    double norm2 = 0.0;
    for (uint64_t i = k; i < n; ++i) { vk[i] = a[i * b + k]; norm2 += vk[i] * vk[i]; }
    if (norm2 == 0.0) continue;
    vk[k] -= vk[k] >= 0.0 ? -std::sqrt(norm2) : std::sqrt(norm2);
    double vnorm2 = 0.0;
    for (uint64_t i = k; i < n; ++i) vnorm2 += vk[i] * vk[i];
    if (vnorm2 == 0.0) continue;
    beta[k] = 2.0 / vnorm2;
    pca_reflect(a, n, b, vk, beta[k], k, k, dot);
  }
  std::fill(a.begin(), a.end(), 0.0);                  // Q = H_0 H_1 ... H_{b-1} [I_b; 0]
  for (uint32_t j = 0; j < b; ++j) a[(size_t)j * b + j] = 1.0;
  for (int k = (int)b - 1; k >= 0; --k)
    if (beta[k] != 0.0) pca_reflect(a, n, b, &v[(size_t)k * n], beta[k], (uint64_t)k, 0, dot);
}

// Eigen-decomposition of the symmetric t [b][b] by cyclic Jacobi: t is left with the eigenvalues on its diagonal, u [b][b]
// (row-major) holds the eigenvectors as columns.
inline void pca_jacobi(std::vector<double>& t, uint32_t b, std::vector<double>& u) {
  u.assign((size_t)b * b, 0.0);
  for (uint32_t i = 0; i < b; ++i) u[(size_t)i * b + i] = 1.0;
  for (int sweep = 0; sweep < 100; ++sweep) {
    bool rotated = false;
    for (uint32_t p = 0; p + 1 < b; ++p)
      for (uint32_t q = p + 1; q < b; ++q) {
        const double apq = t[(size_t)p * b + q], app = t[(size_t)p * b + p], aqq = t[(size_t)q * b + q];
        if (std::fabs(apq) <= 1e-18 * std::sqrt(std::fabs(app * aqq)) || apq == 0.0) continue;
        rotated = true;
        const double theta = (aqq - app) / (2.0 * apq);
        const double tn = (theta >= 0.0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double cs = 1.0 / std::sqrt(tn * tn + 1.0), sn = tn * cs;
        for (uint32_t k = 0; k < b; ++k) {             // columns p, q
          const double xp = t[(size_t)k * b + p], xq = t[(size_t)k * b + q];
          t[(size_t)k * b + p] = cs * xp - sn * xq; t[(size_t)k * b + q] = sn * xp + cs * xq;
        }
        for (uint32_t k = 0; k < b; ++k) {             // rows p, q
          const double xp = t[(size_t)p * b + k], xq = t[(size_t)q * b + k];
          t[(size_t)p * b + k] = cs * xp - sn * xq; t[(size_t)q * b + k] = sn * xp + cs * xq;
        }
        t[(size_t)p * b + q] = t[(size_t)q * b + p] = 0.0;
        for (uint32_t k = 0; k < b; ++k) {
          const double xp = u[(size_t)k * b + p], xq = u[(size_t)k * b + q];
          u[(size_t)k * b + p] = cs * xp - sn * xq; u[(size_t)k * b + q] = sn * xp + cs * xq;
        }
      }
    if (!rotated) break;
  }
}

}  // namespace kgl
