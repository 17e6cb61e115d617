// kgl_b200_api.cu -- the C ABI (include/kgl_b200.h) over the sm_100a kernels. No CPU fallback anywhere in this file.
#include "../../include/kgl_b200.h"

#include "common.cuh"
#include "locus_kernels.cuh"
#include "stream_launch.cuh"
#include "sparse_events.cuh"
#include "sample_major.cuh"
#include "terms_fast.cuh"
#include "terms_moments.cuh"
#include "terms_moments_mma.cuh"
#include "misc_kernels.cuh"
#include "ibs_launch.cuh"
#include "tail_kernels.cuh"
#include "multi_allelic.cuh"
#include "gram_launch.cuh"
#include "ibs_gram.cuh"
#include "king.cuh"
#include "pca.cuh"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

using namespace kgl;

namespace {

thread_local std::string tl_create_error;

// Exchange regions exported by contexts of THIS process (kgl_b200_peer_export): a CUDA IPC handle cannot be opened by the
// process that created it, so kgl_b200_peer_attach maps such regions directly.
struct LocalPeerRegion { unsigned char handle[KGL_B200_PEER_HANDLE_BYTES]; void* ptr; int device; const void* owner; };
std::mutex g_peer_mu;
std::vector<LocalPeerRegion> g_peer_regions;

template <class T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;   // elements
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p) cudaFree(p); }
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T));
    if (e == cudaSuccess) cap = n;
    return e;
  }
  // For buffers whose size follows the selection window (the moment tables): a quarter of head room, so that a run of windows of
  // similar sizes reallocates once, not every time a window is a little larger than all before it.
  cudaError_t ensure_roomy(size_t n) { return n <= cap ? cudaSuccess : ensure(n + n / 4); }
};

// Event pairs around the launches of one kind since the last reset (kgl_b200_kernel_timer_read, kgl_b200_ibs_timer_read).
struct TimerRing {
  static constexpr int kSlots = 256;
  std::vector<cudaEvent_t> ev;
  int used = 0;
  TimerRing() = default;
  TimerRing(const TimerRing&) = delete;
  TimerRing& operator=(const TimerRing&) = delete;
  ~TimerRing() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
  // The next pair (its events are created on first use), or two null events when every slot has been used since the reset.
  cudaError_t next(cudaEvent_t& e0, cudaEvent_t& e1) {
    e0 = e1 = nullptr;
    if (used == kSlots) return cudaSuccess;
    while ((int)ev.size() < 2 * (used + 1)) {
      cudaEvent_t e = nullptr;
      const cudaError_t err = cudaEventCreate(&e);
      if (err != cudaSuccess) return err;
      ev.push_back(e);
    }
    e0 = ev[2 * used]; e1 = ev[2 * used + 1];
    ++used;
    return cudaSuccess;
  }
  // Milliseconds of the first min(used, capacity) pairs; the events must have completed.
  cudaError_t read(float* ms, uint32_t capacity, uint32_t* n) const {
    uint32_t k = 0;
    for (; k < (uint32_t)used && k < capacity; ++k) {
      const cudaError_t err = cudaEventElapsedTime(&ms[k], ev[2 * k], ev[2 * k + 1]);
      if (err != cudaSuccess) return err;
    }
    *n = k;
    return cudaSuccess;
  }
};

// Identifies the IBS tile list on the device: a repeated request (the benchmark loop, HallME-style reruns) neither builds nor
// uploads it again.
struct TileKey {
  enum Kind : uint64_t { kNone, kUpper, kBand, kList };
  Kind kind = kNone;
  uint64_t a = 0, b = 0;   // kUpper: first, stride; kBand: first and end tile row; kList: FNV-1a hash of the coordinates, tiles per side
  uint64_t n = 0;          // tiles
  bool operator==(const TileKey& o) const { return kind == o.kind && a == o.a && b == o.b && n == o.n; }
};

// A tile list: its key and, for a list of coordinates from the host, the coordinates. The tiles of a range of the upper triangle
// or of a band of tile rows follow from the key (tile_coords).
struct TileList {
  TileKey key;
  std::vector<uint2> coords;
};

}  // namespace

struct kgl_b200_ctx {
  int device = 0;
  int sm_count = 148;
  uint64_t total_memory = 0;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool ev_valid = false;
  TimerRing timer;                        // around every launch of the streaming kernel (bench.py's live roofline timing)
  cudaEvent_t last_e0 = nullptr, last_e1 = nullptr;
  std::string err;
  uint64_t launches = 0;

  // population. units = device row pitch in 128-bit units (>= host_units: wide populations are padded to 40-unit slices)
  uint64_t N = 0, L = 0, row_bytes = 0, host_units = 0, units = 0, Npad = 0, padded_rows = 0;
  uint32_t n_pop = 0;
  bool have_geno = false, have_loci = false, have_superpop = false, unphased = false;
  DevBuf<uint8_t> d_packed;
  DevBuf<float> d_af;
  DevBuf<uint8_t> d_superpop, d_sel, d_need32;
  DevBuf<uint64_t> d_popmask;
  // dropped-cell index (built once per uploaded matrix)
  DevBuf<DroppedKey> d_dropped;          // sorted keys (genome << 32 | row)
  DevBuf<uint64_t> d_dropped_seg;        // [Npad + 1] first key of every genome
  DevBuf<unsigned long long> d_dropped_counter;
  DevBuf<DroppedKey> d_dropped_unsorted;
  DevBuf<uint8_t> d_sort_temp;
  DevBuf<uint2> d_dropped_cells;         // per indexed cell {row, frequency float of the genome's population} (k_dropped_cells)
  uint64_t n_dropped = 0;
  bool dropped_indexed = false, dropped_valid = false;
  int dropped_cells_state = 0;           // 0: stale; 1: rows only (no frequencies uploaded yet); 2: rows + frequencies
  std::vector<uint32_t> h_offsets;     // host copy of the locus offsets (they arrive from the host): window -> row range
  uint64_t sel_row_lo = 0, sel_row_hi = ~0ull;   // rows that can be selected (the window of the last select_loci); [0, inf): unknown
  bool have_offsets = false;
  uint64_t loci_len = 0;               // n_loci of the uploaded AF table
  DevBuf<uint32_t> d_offsets;
  DevBuf<uint8_t> d_locus_keep;          // verdict of the variant-level filters per locus (kgl_b200_set_locus_filter)
  bool keep_valid = false;
  DevBuf<unsigned long long> d_sel_counts;
  DevBuf<uint32_t> d_chain_u32;          // spaced selection: next-valid table, two jump tables, block summaries
  DevBuf<uint8_t> d_chain_mark;
  std::vector<uint8_t> h_superpop;
  bool units_valid = false;

  // per-locus preparation
  // Outputs of k_locus_prepare, double-buffered: the preparation of pass i+1 runs on prep_stream while the tail kernel
  // of pass i still reads the buffers of pass i (ensure_prepared). acc: every accumulator of a preparation in one allocation,
  // zeroed with one memset -- {uint32 blocks with an unselected row, 3 x pad} | totals_fx u64[6][TOT_COUNT] |
  // ecorr_fx u64[Npad][2] | nz_rare u32[Npad].
  struct PrepSet {
    DevBuf<uint16_t> flags16, sum64;
    DevBuf<uint32_t> selw;
    DevBuf<uint8_t> acc;
    static constexpr size_t kTotalsOff = 16, kEcorrOff = 16 + kMaxPop * TOT_COUNT * 8;
    static size_t acc_bytes(uint64_t npad) { return kEcorrOff + (size_t)npad * 20; }
    uint32_t* unselected_blocks() const { return reinterpret_cast<uint32_t*>(acc.p); }
    unsigned long long* totals_fx() const { return reinterpret_cast<unsigned long long*>(acc.p + kTotalsOff); }
    unsigned long long* ecorr_fx() const { return reinterpret_cast<unsigned long long*>(acc.p + kEcorrOff); }
    uint32_t* nz_rare(uint64_t npad) const { return reinterpret_cast<uint32_t*>(acc.p + kEcorrOff + npad * 16); }
    double fx = 0.0;        // fixed-point scale of this set's sums (fx_scale_for the rows of the selection window it was prepared for)
  } prep[2];
  int par = 0;                                  // the set the current selection was prepared into
  // Three streams per pass (DESIGN 4): the streaming kernel on the context stream; the preparation of the NEXT pass and the
  // tail of the PREVIOUS pass on two side streams, where they run next to the streaming kernel's CTAs (72 registers x 608
  // threads leave room for one 256-thread block of either on every SM).
  cudaStream_t prep_stream = nullptr, tail_stream = nullptr, copy_stream = nullptr;
  std::vector<cudaEvent_t> chunk_ev;      // chunked upload: one event per row chunk
  cudaEvent_t prep_done = nullptr, inputs_ready = nullptr;
  cudaEvent_t readers_main[2] = {nullptr, nullptr}, readers_tail[2] = {nullptr, nullptr};   // readers of prep[par] so far
  bool readers_marked[2] = {false, false};
  cudaEvent_t stream_done[2] = {nullptr, nullptr}, tail_done[2] = {nullptr, nullptr};       // per cta_counts buffer
  bool tail_marked[2] = {false, false};
  int cbuf = 0;                                 // the cta_counts buffer of the most recent pass
  bool tail_pending = false;                    // a tail runs on tail_stream that the context stream has not been ordered after
  bool inputs_async = false;                    // d_sel was last written by a kernel on the main stream without a host sync
  bool prep_valid = false, prep_has_w0 = false, prep_has_selw = false;

  // multi-allelic loci (multi_allelic.cuh): rows of the locus table, per-slot frequencies, side cells, per-selection table
  uint64_t n_multi = 0;
  DevBuf<uint32_t> d_multi_rows, d_multi_counts;
  DevBuf<float> d_multi_af;
  DevBuf<uint8_t> d_multi_cells;
  DevBuf<MultiLocus> d_multi_tab;
  DevBuf<double> d_multi_out;

  // sample-major copy
  DevBuf<uint32_t> d_sm_lo, d_sm_hi;
  DevBuf<uint2> d_sm_codes;             // interleaved codes of the same cells (terms_fast.cuh)
  uint64_t n_gblocks = 0, n_words = 0;
  bool sm_valid = false, codes_valid = false;

  // fused pass outputs
  DevBuf<uint32_t> d_locus_counts, d_cta_counts[2];
  DevBuf<uint8_t> d_scratch;            // per-genome accumulators of one pass, zeroed with a single memset
  uint32_t *d_gcounts = nullptr, *d_n3 = nullptr;
  unsigned long long* d_ecorr_scan = nullptr;   // fallback path (code-3 cells not indexed): k_dropped_scan's fixed-point sums
  DevBuf<double> d_partials, d_iter, d_f, d_bracket, d_chunk_out, d_inbreeding, d_grid;
  DevBuf<uint32_t> d_done;
  DevBuf<unsigned long long> d_flag;
  // table-driven estimator sweeps (terms_fast.cuh): per-genome limits of the feasible region, lane states of the last
  // Newton sweep, chunk outputs of the exact fallback
  DevBuf<double> d_limits, d_slow_out;
  DevBuf<uint8_t> d_lane_state;
  // peer-memory exchange of the locus-sharded step (misc_kernels.cuh, k_peer_exchange)
  DevBuf<unsigned char> d_xchg;
  uint64_t xchg_npad = 0, peer_epoch = 0;
  uint32_t peer_rank = 0, peer_world = 0;
  std::vector<void*> peer_base;           // mapped exchange regions of the other ranks (nullptr for our own slot)
  std::vector<uint8_t> peer_ipc;          // 1: peer_base[r] was opened with cudaIpcOpenMemHandle (closed on detach)
  DevBuf<unsigned int> d_peer_error;      // set by k_peer_exchange when a peer did not arrive in time
  uint64_t peer_timeout_ms = 10000;
  bool peer_results = false;              // d_results / d_locus_counts were produced by a peer step: the fetches check d_peer_error
  double* partials_target = nullptr;      // where the moment kernels write (d_partials unless a peer step redirects them)
  DevBuf<double2> d_terms_table;         // per-run table constants of the HALL / NEWTON sweeps (terms_fast.cuh)
  int table_mode = -1;                   // mode the table was built for (-1: none); reset by inbreed_begin
  DevBuf<uint32_t> d_list_count;         // length of d_list on the device (sweeps between two host checks shrink it)
  DevBuf<uint32_t> d_n_slow, d_list;    // d_list: genomes whose root search is still running (late Newton sweeps)
  uint64_t list_len = 0;
  bool limits_valid = false;
  // moment tables of the iterative estimators (terms_moments.cuh), built once per selection
  DevBuf<uint64_t> d_mom_keys, d_mom_keys2, d_mom_base;
  DevBuf<uint32_t> d_mom_rows, d_mom_rows2, d_mom_pop_begin, d_mom_cnt, d_mom_totals;
  DevBuf<int> d_mom_stats;
  DevBuf<long long> d_mom_pm, d_mom_mi;
  DevBuf<uint2> d_mom_offs;
  DevBuf<uint32_t> d_mom_bounds, d_mom_bounds2, d_mom_unit_out, d_mom_unit_cnt, d_mom_unit_offs;
  DevBuf<MomUnit> d_mom_units;
  DevBuf<uint2> d_mom_unit_range;
  DevBuf<unsigned long long> d_mom_pop_cmin;
  DevBuf<unsigned char> d_mom_btiles;
  DevBuf<uint32_t> d_mom_rare_bits;
  uint32_t mom_mma_tile_lo[kMaxPop] = {}, mom_mma_tile_hi[kMaxPop] = {}, mom_mma_tiles = 1;
  bool mom_used_mma = false, mom_cnt_valid = false;
  uint32_t mom_n_units = 0;
  DevBuf<double> d_mom_list, d_mom_limits, d_mom_rr;
  DevBuf<uint8_t> d_mom_tmp;
  bool mom_valid = false, mom_lists = false, mom_supported = false, used_moments = false;
  int mom_b_lo = 0, mom_nbt = 0;
  DevBuf<uint64_t> d_genome_counts;
  DevBuf<kgl_b200_locus_results> d_results;
  DevBuf<uint32_t> d_ibs;
  // pairwise IBS (ibs_tile.cuh): planes of the dense kernel, tile list, accumulators, compact tile results
  DevBuf<uint32_t> d_ibs_lo, d_ibs_hi, d_sm_valid, d_ibs_acc, d_ibs_tiles_out;
  DevBuf<uint2> d_ibs_tiles;
  int ibs_mode = -1;                 // 0: no code-3 cell; 1: in-kernel validity plane; 2: pre-masked planes + sparse repair
  TimerRing ibs_timer;
  uint64_t ibs_last_count = 0;
  TileKey ibs_tiles_key;                 // the tile list on the device
  // AF-bin passes (CalcFWS): row mask, its 64-row summaries, the all-genomes population tables
  DevBuf<uint16_t> d_bin_flags, d_bin_sum64;
  DevBuf<uint32_t> d_bin_popmask32, d_bin_state;   // d_bin_state: [0] all-selected flag (always 0), [1] rows in the bin
  DevBuf<uint8_t> d_bin_need32, d_zero_superpop;
  DevBuf<uint64_t> d_bin_out;
  uint64_t bin_tables_n = 0, bin_tables_units = 0;
  // K5 (gram_i8.cuh): 2-bit code matrix (code 3 kept) in row-block-major layout, tile list, int32 Gram matrix, rank-one terms
  DevBuf<uint32_t> d_codes16;
  DevBuf<int32_t> d_gram, d_gram_hh, d_gram_aa;
  DevBuf<uint2> d_ibs_blocks;          // 256 x 256 Gram blocks the current IBS tile list needs (ibs_gram.cuh)
  DevBuf<uint32_t> d_ibs_tile_block;   // per tile: index of its block | 1 << 31 when mirrored
  uint32_t ibs_n_blocks = 0;
  DevBuf<int32_t> d_ibs_class;         // {heterozygous, hom-alt} cells per genome on the IBS planes
  bool ibs_class_valid = false;
  bool ibs_tensor_enabled = true, ibs_used_tensor = false;
  DevBuf<uint2> d_gram_tiles;
  DevBuf<double> d_gp_chunks, d_gp;
  DevBuf<uint8_t> d_gram_out;
  uint64_t gram_tiles_ld = 0, gram_n_tiles = 0, gram_first = 0, gram_stride = 1;
  bool codes16_valid = false;
  bool gram_valid = false;             // d_gram holds the last kgl_b200_enqueue_gram[_tiles] result (the IBS tensor form lends it out)
  cudaEvent_t gram_e0 = nullptr, gram_e1 = nullptr;
  // KING-robust kinship (king.cuh): M = H C^T blocks, dense slab, pair list and its sort
  DevBuf<int32_t> d_king_m;
  DevBuf<double> d_king_out;
  DevBuf<kgl_b200_king_pair> d_king_pairs, d_king_sorted;
  DevBuf<unsigned long long> d_king_keys, d_king_keys2, d_king_cursor;
  DevBuf<uint32_t> d_king_index, d_king_index2;
  DevBuf<uint8_t> d_king_sort_temp;
  // genotype PCA (pca.cuh): loci-major codes (code 3 kept), per-locus p / d / used, the product's blocks, digits and Gram outputs
  DevBuf<uint32_t> d_codes_loci;
  bool codes_loci_valid = false;
  DevBuf<uint8_t> d_pca_keep, d_pca_used;
  DevBuf<uint32_t> d_pca_counts;            // raw per-locus counts of PCA's own counting pass (d_locus_counts stays the caller's)
  DevBuf<double> d_pca_p, d_pca_d, d_pca_x, d_pca_y, d_pca_wv, d_pca_out;
  DevBuf<uint32_t> d_pca_digits;
  DevBuf<int32_t> d_pca_acc;
  DevBuf<unsigned long long> d_pca_stats;   // max bits and sums of X (2 x 48), of W | V (2 x 96), |U|
  DevBuf<uint2> d_pca_tiles;

  // iterative estimator state
  int algo = -1, phase = 0, iteration = 0;
  kgl_b200_inbreed_options opt{};
  std::vector<double> hall_start;

  ~kgl_b200_ctx();
};

namespace {

int fail(kgl_b200_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg; else tl_create_error = msg;
  return code;
}

#define KGL_CUDA(c, call)                                                                                   \
  do {                                                                                                      \
    cudaError_t e_ = (call);                                                                                \
    if (e_ != cudaSuccess)                                                                                  \
      return fail((c), e_ == cudaErrorMemoryAllocation ? KGL_B200_ERR_NOMEM : KGL_B200_ERR_CUDA,            \
                  std::string(#call) + ": " + cudaGetErrorString(e_));                                      \
  } while (0)

#define KGL_LAUNCH_CHECK(c)                                                                                 \
  do {                                                                                                      \
    ++(c)->launches;                                                                                        \
    cudaError_t e_ = cudaGetLastError();                                                                    \
    if (e_ != cudaSuccess) return fail((c), KGL_B200_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e_)); \
  } while (0)

void peer_detach(kgl_b200_ctx* c) {
  for (size_t r = 0; r < c->peer_base.size(); ++r)
    if (c->peer_base[r] && r < c->peer_ipc.size() && c->peer_ipc[r]) cudaIpcCloseMemHandle(c->peer_base[r]);
  c->peer_base.clear(); c->peer_ipc.clear(); c->peer_world = 0;
}

void peer_unregister(const kgl_b200_ctx* c) {
  std::lock_guard<std::mutex> lock(g_peer_mu);
  for (size_t i = 0; i < g_peer_regions.size();)
    if (g_peer_regions[i].owner == c) g_peer_regions.erase(g_peer_regions.begin() + i); else ++i;
}

inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// Orders the context stream after the tail of the last pass (no host synchronisation).
int join_tail(kgl_b200_ctx* c) {
  if (c->tail_pending) {
    KGL_CUDA(c, cudaStreamWaitEvent(c->stream, c->tail_done[c->cbuf], 0));
    c->tail_pending = false;
  }
  return KGL_B200_OK;
}

// Every entry point starts here. Only the resident pass (kgl_b200_enqueue_count_and_inbreed[_peer]) leaves its tail running on
// the side stream; whatever is called next is ordered after it first -- unless it is another such pass (join = false).
int use_device(kgl_b200_ctx* c, bool join = true) {
  KGL_CUDA(c, cudaSetDevice(c->device));
  return join ? join_tail(c) : KGL_B200_OK;
}

int ensure_side_streams(kgl_b200_ctx* c) {
  if (c->prep_stream) return KGL_B200_OK;
  int least = 0, greatest = 0;
  KGL_CUDA(c, cudaDeviceGetStreamPriorityRange(&least, &greatest));
  // The side kernels run NEXT to the streaming kernel, whose 180 KB of dynamic shared memory force the largest shared-memory
  // carve-out on the SM: they ask for the same carve-out, so that an SM never has to be drained to switch configurations.
  const int max_shared = cudaSharedmemCarveoutMaxShared;
  KGL_CUDA(c, cudaFuncSetAttribute(k_locus_prepare<false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, max_shared));
  KGL_CUDA(c, cudaFuncSetAttribute(k_locus_prepare<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, max_shared));
  KGL_CUDA(c, cudaFuncSetAttribute(k_locus_prepare<true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, max_shared));
  KGL_CUDA(c, cudaFuncSetAttribute(k_locus_prepare<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, max_shared));
  KGL_CUDA(c, cudaFuncSetAttribute(k_tail, cudaFuncAttributePreferredSharedMemoryCarveout, max_shared));
  KGL_CUDA(c, cudaFuncSetAttribute(k_peer_publish, cudaFuncAttributePreferredSharedMemoryCarveout, max_shared));
  KGL_CUDA(c, cudaFuncSetAttribute(k_peer_exchange, cudaFuncAttributePreferredSharedMemoryCarveout, max_shared));
  KGL_CUDA(c, cudaStreamCreateWithPriority(&c->prep_stream, cudaStreamNonBlocking, least));
  KGL_CUDA(c, cudaStreamCreateWithPriority(&c->tail_stream, cudaStreamNonBlocking, least));
  KGL_CUDA(c, cudaEventCreateWithFlags(&c->prep_done, cudaEventDisableTiming));
  KGL_CUDA(c, cudaEventCreateWithFlags(&c->inputs_ready, cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) {
    KGL_CUDA(c, cudaEventCreateWithFlags(&c->readers_main[i], cudaEventDisableTiming));
    KGL_CUDA(c, cudaEventCreateWithFlags(&c->readers_tail[i], cudaEventDisableTiming));
    KGL_CUDA(c, cudaEventCreateWithFlags(&c->stream_done[i], cudaEventDisableTiming));
    KGL_CUDA(c, cudaEventCreateWithFlags(&c->tail_done[i], cudaEventDisableTiming));
  }
  return KGL_B200_OK;
}

// Per-population genome masks of every 128-bit unit (read as 32-bit halves by the streaming kernel) and the populations
// present in every 32-genome group.
int build_unit_tables(kgl_b200_ctx* c) {
  if (c->units_valid) return KGL_B200_OK;
  const uint64_t units = c->units;
  std::vector<uint8_t> need32(units * 2, 0);
  std::vector<uint64_t> popmask((size_t)KGL_B200_MAX_POP * units, 0);
  for (uint64_t g = 0; g < c->N; ++g) {
    const int k = c->h_superpop[g];
    popmask[(size_t)k * units + (g >> 6)] |= 1ull << (g & 63);
    need32[g >> 5] |= (uint8_t)(1u << k);
  }
  KGL_CUDA(c, c->d_need32.ensure(need32.size()));
  KGL_CUDA(c, c->d_popmask.ensure(popmask.size()));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_need32.p, need32.data(), need32.size(), cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_popmask.p, popmask.data(), popmask.size() * 8, cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  c->units_valid = true;
  return KGL_B200_OK;
}

int require_population(kgl_b200_ctx* c, bool need_loci) {
  if (!c->have_geno) return fail(c, KGL_B200_ERR_STATE, "no genotype matrix uploaded");
  if (need_loci) {
    if (!c->have_loci) return fail(c, KGL_B200_ERR_STATE, "no allele frequencies uploaded (kgl_b200_upload_loci)");
    if (!c->have_superpop) return fail(c, KGL_B200_ERR_STATE, "no genome super-populations set (kgl_b200_set_genome_superpop)");
    if (c->loci_len != c->L) return fail(c, KGL_B200_ERR_STATE, "locus selection does not match the genotype matrix");
    for (uint64_t g = 0; g < c->N; ++g)
      if (c->h_superpop[g] >= c->n_pop) return fail(c, KGL_B200_ERR_INVALID, "genome super-population index out of range");
  }
  return KGL_B200_OK;
}

// First row of the locus table at or after offset `lower` (the offsets are sorted).
uint64_t first_row_at(const kgl_b200_ctx* c, uint64_t lower) {
  return std::lower_bound(c->h_offsets.begin(), c->h_offsets.end(), lower, [](uint32_t o, uint64_t v) { return (uint64_t)o < v; }) -
         c->h_offsets.begin();
}

uint64_t term_words(uint64_t n_loci) {
  const uint64_t nw = (n_loci + 31) / 32;
  return (nw + kTermTileWords - 1) / kTermTileWords * kTermTileWords;
}

// Selection flags, 64-row summaries, packed selection words, rare-major rows and dense totals (once per selection).
int ensure_prepared(kgl_b200_ctx* c, bool want_w0 = false, bool want_selw = false) {
  if (c->prep_valid && (c->prep_has_w0 || !want_w0) && (c->prep_has_selw || !want_selw)) return KGL_B200_OK;
  want_w0 = want_w0 || (c->prep_valid && c->prep_has_w0);          // a repeat keeps what the earlier one produced
  want_selw = want_selw || (c->prep_valid && c->prep_has_selw);
  int rc = build_unit_tables(c); if (rc) return rc;
  const uint64_t L = c->L;
  c->n_words = term_words(L);
  const uint64_t span = std::max<uint64_t>(c->padded_rows, c->n_words * 32);
  const uint64_t n_tiles = std::max<uint64_t>(1, (span + kPrepLociPerBlock - 1) / kPrepLociPerBlock);
  const unsigned nb = (unsigned)std::min<uint64_t>(n_tiles, (uint64_t)c->sm_count * 2);
  rc = ensure_side_streams(c); if (rc) return rc;
  // Everything enqueued so far may read the current set (the streaming kernels on the context stream, the tails on the tail
  // stream): mark both, switch to the other set, and let the preparation start as soon as the readers of THAT set (marked one
  // switch ago) are done. It does not wait for the streaming kernel of the pass before it: it runs next to it.
  KGL_CUDA(c, cudaEventRecord(c->readers_main[c->par], c->stream));
  KGL_CUDA(c, cudaEventRecord(c->readers_tail[c->par], c->tail_stream));
  c->readers_marked[c->par] = true;
  c->par ^= 1;
  kgl_b200_ctx::PrepSet& S = c->prep[c->par];
  KGL_CUDA(c, S.flags16.ensure(c->padded_rows));
  KGL_CUDA(c, S.sum64.ensure(c->padded_rows / 64));
  if (want_selw) KGL_CUDA(c, S.selw.ensure((size_t)KGL_B200_MAX_POP * c->n_words));
  const size_t acc_bytes = kgl_b200_ctx::PrepSet::acc_bytes(c->Npad);
  KGL_CUDA(c, S.acc.ensure(acc_bytes));
  cudaStream_t ps = c->prep_stream;
  if (c->readers_marked[c->par]) {
    KGL_CUDA(c, cudaStreamWaitEvent(ps, c->readers_main[c->par], 0));
    KGL_CUDA(c, cudaStreamWaitEvent(ps, c->readers_tail[c->par], 0));
  }
  if (c->inputs_async) {            // the selection mask / frequency table was just written on the context stream without a host sync
    KGL_CUDA(c, cudaEventRecord(c->inputs_ready, c->stream));
    KGL_CUDA(c, cudaStreamWaitEvent(ps, c->inputs_ready, 0));
    c->inputs_async = false;
  }
  KGL_CUDA(c, cudaMemsetAsync(S.acc.p, 0, acc_bytes, ps));
  const uint4* packed = reinterpret_cast<const uint4*>(c->d_packed.p);
  // at most one term per row of the selection window: a narrow window of a long contig keeps its low-order bits
  const uint64_t window_rows = c->sel_row_hi == ~0ull ? L : std::min<uint64_t>(L, c->sel_row_hi) - std::min<uint64_t>(L, c->sel_row_lo);
  const double fx = fx_scale_for(std::max<uint64_t>(window_rows, 1));
  S.fx = fx;
#define KGL_PREP(W0, SELW)                                                                                                          \
  k_locus_prepare<W0, SELW><<<nb, kPrepThreads, 0, ps>>>(c->d_af.p, c->d_sel.p, L, c->padded_rows, n_tiles, (int)c->n_pop,         \
      S.flags16.p, S.sum64.p, SELW ? S.selw.p : nullptr, c->n_words, packed, (uint32_t)c->units, c->d_popmask.p,                   \
      S.nz_rare(c->Npad), S.ecorr_fx(), fx, S.totals_fx(), S.unselected_blocks())
  if (want_w0 && want_selw) KGL_PREP(true, true);
  else if (want_w0) KGL_PREP(true, false);
  else if (want_selw) KGL_PREP(false, true);
  else KGL_PREP(false, false);
#undef KGL_PREP
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaEventRecord(c->prep_done, ps));
  KGL_CUDA(c, cudaStreamWaitEvent(c->stream, c->prep_done, 0));
  c->prep_valid = true; c->prep_has_w0 = want_w0; c->prep_has_selw = want_selw;
  c->mom_valid = false;             // the moment tables belong to the selection that was prepared before
  return KGL_B200_OK;
}

int ensure_sample_major(kgl_b200_ctx* c) {
  if (c->sm_valid) return KGL_B200_OK;
  c->n_gblocks = c->units * 2;
  const uint64_t nw = term_words(c->L);
  c->n_words = nw;
  const size_t n = (size_t)c->n_gblocks * nw * 32;
  KGL_CUDA(c, c->d_sm_lo.ensure(n));
  KGL_CUDA(c, c->d_sm_hi.ensure(n));
  dim3 grid((unsigned)nw, (unsigned)((c->n_gblocks + 7) / 8));
  k_to_sample_major<<<grid, 256, 0, c->stream>>>(reinterpret_cast<const uint32_t*>(c->d_packed.p), c->units * 4, c->L,
                                                  c->n_gblocks, nw, c->d_sm_lo.p, c->d_sm_hi.p);
  KGL_LAUNCH_CHECK(c);
  c->sm_valid = true;
  return KGL_B200_OK;
}

// The side list of code-3 cells (SURVEY flattener contract), built on the device once per uploaded matrix.
// Populations with more than ~1.5% code-3 cells are not indexed: every pass scans the matrix for them instead.
uint64_t dropped_index_limit(const kgl_b200_ctx* c) { return std::max<uint64_t>(1u << 16, c->N * c->L / 64); }   // indexed iff total <= limit

// Keys of the code-3 cells of n128 128-bit units from unit first on into d_dropped_unsorted (at most cap of them; the cursor
// d_dropped_counter[1] counts them all).
int launch_dropped_index(kgl_b200_ctx* c, uint64_t first, uint64_t n128, uint64_t cap) {
  const unsigned grid = (unsigned)std::min<uint64_t>((n128 + 255) / 256, (uint64_t)c->sm_count * 16);
  k_dropped_index<<<grid, 256, 0, c->stream>>>(reinterpret_cast<const uint4*>(c->d_packed.p) + first, n128, first, (uint32_t)c->units,
                                                c->d_dropped_counter.p + 1, c->d_dropped_unsorted.p, cap);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

// Sort + segment table of the n keys in d_dropped_unsorted (n <= its capacity), or the "not indexed" verdict.
int finish_dropped_index(kgl_b200_ctx* c, unsigned long long total) {
  c->n_dropped = total;
  c->dropped_indexed = total <= dropped_index_limit(c);
  if (c->dropped_indexed) {
    KGL_CUDA(c, c->d_dropped.ensure(std::max<uint64_t>(total, 1)));
    KGL_CUDA(c, c->d_dropped_seg.ensure(c->Npad + 1));
    if (total > 0) {
      DevBuf<DroppedKey>& unsorted = c->d_dropped_unsorted;   // kept: re-uploads of the same shape allocate nothing
      DevBuf<uint8_t>& temp = c->d_sort_temp;
      int end_bit = 33;
      while (end_bit < 64 && (c->Npad >> (end_bit - 32)) != 0) ++end_bit;
      size_t temp_bytes = 0;
      cudaError_t e = cub::DeviceRadixSort::SortKeys(nullptr, temp_bytes, unsorted.p, c->d_dropped.p, (uint64_t)total, 0, end_bit, c->stream);
      if (e == cudaSuccess) e = temp.ensure(temp_bytes);
      if (e == cudaSuccess) e = cub::DeviceRadixSort::SortKeys(temp.p, temp_bytes, unsorted.p, c->d_dropped.p, (uint64_t)total, 0, end_bit, c->stream);
      KGL_CUDA(c, e);
      c->launches += 2;
    }
    k_dropped_segments<<<blocks_for(c->Npad + 1, 256), 256, 0, c->stream>>>(c->d_dropped.p, total, c->Npad, c->d_dropped_seg.p);
    KGL_LAUNCH_CHECK(c);
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  c->dropped_valid = true; c->dropped_cells_state = 0;
  return KGL_B200_OK;
}

// The side list of code-3 cells, built once per matrix that is already resident (device-generated populations; uploads index
// while they copy, see kgl_b200_upload_genotypes).
int build_dropped_index(kgl_b200_ctx* c) {
  if (c->dropped_valid) return KGL_B200_OK;
  const uint64_t n128 = c->L * c->units;
  const unsigned grid = (unsigned)std::min<uint64_t>((n128 + 255) / 256, (uint64_t)c->sm_count * 16);
  KGL_CUDA(c, c->d_dropped_counter.ensure(2));
  KGL_CUDA(c, cudaMemsetAsync(c->d_dropped_counter.p, 0, 16, c->stream));
  k_dropped_count<<<grid, 256, 0, c->stream>>>(reinterpret_cast<const uint4*>(c->d_packed.p), n128, c->d_dropped_counter.p);
  KGL_LAUNCH_CHECK(c);
  unsigned long long total = 0;
  KGL_CUDA(c, cudaMemcpyAsync(&total, c->d_dropped_counter.p, 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  if (total > 0 && total <= dropped_index_limit(c)) {
    KGL_CUDA(c, c->d_dropped_unsorted.ensure(total));
    int rc = launch_dropped_index(c, 0, n128, total); if (rc) return rc;
  }
  return finish_dropped_index(c, total);
}

// Device storage of the genotype matrix: rows padded to a multiple of 256 (zero rows), row pitch c->units.
int alloc_matrix(kgl_b200_ctx* c) {
  c->padded_rows = (c->L + 255) / 256 * 256;
  const size_t bytes = (size_t)c->padded_rows * c->units * 16;
  KGL_CUDA(c, c->d_packed.ensure(bytes));
  if (c->units != c->host_units) {
    KGL_CUDA(c, cudaMemsetAsync(c->d_packed.p, 0, bytes, c->stream));
  } else {
    KGL_CUDA(c, cudaMemsetAsync(c->d_packed.p + (size_t)c->L * c->units * 16, 0, (size_t)(c->padded_rows - c->L) * c->units * 16, c->stream));
  }
  return KGL_B200_OK;
}

// Per-cell side list {row, frequency float of the genome's population} of the indexed code-3 cells, for k_tail. Follows the
// key index (once per matrix) and the frequency table / super-populations (rebuilt when either is uploaded again).
int ensure_dropped_cells(kgl_b200_ctx* c, bool want_af) {
  if (!c->dropped_indexed || c->n_dropped == 0) return KGL_B200_OK;
  const bool have_af = c->have_loci && c->have_superpop && c->loci_len == c->L;
  if (want_af && !have_af) return fail(c, KGL_B200_ERR_STATE, "internal: the code-3 side list needs the allele frequencies");
  const int want_state = have_af ? 2 : 1;
  if (c->dropped_cells_state >= want_state) return KGL_B200_OK;
  KGL_CUDA(c, c->d_dropped_cells.ensure(c->n_dropped));
  k_dropped_cells<<<blocks_for(c->n_dropped, 256), 256, 0, c->stream>>>(c->d_dropped.p, c->n_dropped, have_af ? c->d_superpop.p : nullptr,
                                                                        c->d_af.p, c->L, c->d_dropped_cells.p);
  KGL_LAUNCH_CHECK(c);
  c->dropped_cells_state = want_state;
  return KGL_B200_OK;
}

// End of what a pass put on the tail stream: the event later passes (reuse of the cta_counts buffer) and joins wait for.
int mark_tail(kgl_b200_ctx* c, bool join) {
  KGL_CUDA(c, cudaEventRecord(c->tail_done[c->cbuf], c->tail_stream));
  c->tail_marked[c->cbuf] = true;
  return join ? join_tail(c) : KGL_B200_OK;
}

DenseTotals dense_totals(const kgl_b200_ctx* c, const kgl_b200_ctx::PrepSet& S) {
  const double fx = S.fx > 0.0 ? S.fx : fx_scale_for(c->L);      // a set that was never prepared: the totals are not read
  return DenseTotals{S.totals_fx(), 1.0 / fx, 128.0 / fx};
}

// The fused streaming pass + its tail. raw: allele_count over all loci; otherwise over the selected loci.
// Row mask that replaces the per-population selection flags of a pass: every genome belongs to "population 0" and a row
// counts iff bit 0 of flags16 is set (the AF-bin passes of kgl_b200_run_binned_genome_counts).
struct MaskOverride {
  const uint16_t* flags16; const uint16_t* sum64; const uint32_t* popmask32; const uint8_t* need32;
  const uint8_t* zero_superpop;
};

// want_moments: the tail assembles the moment partials of every genome (d_partials; + the Simple closed form into d_results
// when simple_results); otherwise it leaves the raw per-genome counts d_gcounts {set lo bits, set hi bits} and d_n3.
// defer_join: the tail stays on the tail stream and the context stream is NOT ordered after it (the resident pass: the next
// pass's streaming kernel may start while this tail runs); the next entry point joins (use_device).
// counts: where the per-locus counts go (null = d_locus_counts, the buffer kgl_b200_fetch_locus_counts reads).
int launch_count(kgl_b200_ctx* c, bool raw, bool want_locus_counts, bool want_genome, bool simple_results = false, bool want_moments = false,
                 const MaskOverride* mo = nullptr, bool defer_join = false, DevBuf<uint32_t>* counts = nullptr) {
  DevBuf<uint32_t>& lc = counts ? *counts : c->d_locus_counts;
  int rc = mo ? KGL_B200_OK : build_unit_tables(c);
  if (rc) return rc;
  rc = build_dropped_index(c);
  if (rc) return rc;
  const StreamPlan pl = plan_stream(c->units, c->L, c->sm_count);
  if (pl.padded_rows > c->padded_rows) return fail(c, KGL_B200_ERR_STATE, "internal: stream plan needs more padded rows than allocated");
  if (want_locus_counts) {
    KGL_CUDA(c, lc.ensure((size_t)c->L * 4));
    if (pl.slices > 1) KGL_CUDA(c, cudaMemsetAsync(lc.p, 0, (size_t)c->L * 16, c->stream));
  }
  const bool indexed = c->dropped_indexed || c->n_dropped == 0;
  rc = ensure_side_streams(c); if (rc) return rc;
  if (want_genome) {
    // the tail of the pass before the last one may still read the buffer this pass writes
    if (c->tail_pending && !defer_join) { rc = join_tail(c); if (rc) return rc; }
    c->cbuf ^= 1;
    if (c->tail_marked[c->cbuf]) KGL_CUDA(c, cudaStreamWaitEvent(c->stream, c->tail_done[c->cbuf], 0));
    KGL_CUDA(c, c->d_cta_counts[c->cbuf].ensure((size_t)pl.n_ctas * 2 * c->Npad));
    // scratch: gcounts u32[Npad][2] | n3 u32[Npad] | pad u32[Npad] | ecorr_scan u64[Npad][2] (fallback path only)
    KGL_CUDA(c, c->d_scratch.ensure((size_t)c->Npad * 32));
    c->d_gcounts = reinterpret_cast<uint32_t*>(c->d_scratch.p);
    c->d_n3 = c->d_gcounts + c->Npad * 2;
    c->d_ecorr_scan = reinterpret_cast<unsigned long long*>(c->d_scratch.p + (size_t)c->Npad * 16);
    if (!indexed) KGL_CUDA(c, cudaMemsetAsync(c->d_scratch.p, 0, (size_t)c->Npad * 32, c->stream));
    if (indexed) { rc = ensure_dropped_cells(c, want_moments); if (rc) return rc; }
  }
  StreamParams P{};
  fill_stream_params(P, pl);
  P.packed = reinterpret_cast<const uint4*>(c->d_packed.p);
  P.units = (uint32_t)c->units; P.n_loci = (uint32_t)c->L; P.n_genomes = (uint32_t)c->N;
  P.flags16 = mo ? mo->flags16 : (raw ? nullptr : c->prep[c->par].flags16.p);
  P.sum64 = mo ? mo->sum64 : (raw ? nullptr : c->prep[c->par].sum64.p);
  P.popmask32 = mo ? mo->popmask32 : reinterpret_cast<const uint32_t*>(c->d_popmask.p);     // little endian: u64 mask = {low half, high half}
  P.need32 = mo ? mo->need32 : c->d_need32.p;
  P.n_pop = (raw || mo) ? 1 : c->n_pop;
  P.locus_counts = want_locus_counts ? lc.p : nullptr;
  P.cta_counts = want_genome ? c->d_cta_counts[c->cbuf].p : nullptr;
  P.n_genomes_padded = (uint32_t)c->Npad;
  stream_make_tensor_map(P, pl, c->padded_rows);          // wide populations: one 2-D TMA box per stage
  cudaEvent_t e0, e1;
  KGL_CUDA(c, c->timer.next(e0, e1));
  if (!e0) { e0 = c->ev0; e1 = c->ev1; }       // the ring is full: kgl_b200_last_stream_kernel_ms still times this launch
  KGL_CUDA(c, cudaEventRecord(e0, c->stream));
  KGL_CUDA(c, launch_stream(P, pl, want_locus_counts, want_genome, c->stream));
  ++c->launches;
  KGL_CUDA(c, cudaEventRecord(e1, c->stream));
  c->ev_valid = true;
  c->last_e0 = e0; c->last_e1 = e1;
  if (want_locus_counts && pl.slices > 1) {
    k_fix_locus_n0<<<blocks_for(c->L, 256), 256, 0, c->stream>>>(lc.p, c->L, (uint32_t)c->N);
    KGL_LAUNCH_CHECK(c);
  }
  if (!want_genome) return KGL_B200_OK;
  const uint16_t* fl = mo ? mo->flags16 : (raw ? nullptr : c->prep[c->par].flags16.p);
  const kgl_b200_ctx::PrepSet& S = c->prep[c->par];
  const bool prepared = !raw && !mo;
  const double fx = prepared ? S.fx : fx_scale_for(c->L);
  if (indexed) {
    // the tail runs on its own stream, behind this pass's streaming kernel
    KGL_CUDA(c, cudaEventRecord(c->stream_done[c->cbuf], c->stream));
    KGL_CUDA(c, cudaStreamWaitEvent(c->tail_stream, c->stream_done[c->cbuf], 0));
    TailParams T{};
    T.cta_counts = c->d_cta_counts[c->cbuf].p; T.n_ctas = pl.n_ctas; T.n_genomes_padded = c->Npad;
    T.cells = c->n_dropped ? c->d_dropped_cells.p : nullptr; T.seg = c->d_dropped_seg.p;
    T.row_lo = 0; T.row_hi = 0xFFFFFFFFu;
    if (prepared && c->sel_row_hi != ~0ull && (c->sel_row_lo > 0 || c->sel_row_hi < c->L)) {   // a proper window
      T.row_lo = (uint32_t)c->sel_row_lo; T.row_hi = (uint32_t)std::min<uint64_t>(c->sel_row_hi, 0xFFFFFFFEull);
    }
    T.n_genomes = c->N; T.flags16 = fl;
    T.unselected_blocks = prepared ? S.unselected_blocks() : nullptr;
    T.superpop = mo ? mo->zero_superpop : c->d_superpop.p;
    T.want_moments = want_moments ? 1 : 0; T.unphased = c->unphased ? 1 : 0;
    T.nz_rare = prepared ? S.nz_rare(c->Npad) : nullptr; T.ecorr_rare_fx = prepared ? S.ecorr_fx() : nullptr; T.fx_inv = 1.0 / fx;
    T.totals = dense_totals(c, S); T.partials = c->partials_target ? c->partials_target : c->d_partials.p;
    T.results = simple_results ? c->d_results.p : nullptr;
    T.gcounts = c->d_gcounts; T.n3 = c->d_n3;
    k_tail<<<blocks_for(c->N, kTailGenomesPerBlock), 256, 0, c->tail_stream>>>(T);
    KGL_LAUNCH_CHECK(c);
    c->tail_pending = true;
    if (!defer_join) return mark_tail(c, true);
    return KGL_B200_OK;              // the caller adds what else belongs on the tail stream and calls mark_tail(c, false)
  }
  // populations whose code-3 cells are too many to index: separate kernels, the matrix is scanned for the cells
  k_sum_cta_counts<<<blocks_for(c->Npad, 256), 256, 0, c->stream>>>(c->d_cta_counts[c->cbuf].p, pl.n_ctas, c->Npad, c->d_gcounts);
  KGL_LAUNCH_CHECK(c);
  const uint64_t n128 = c->L * c->units;
  const unsigned grid = (unsigned)std::min<uint64_t>((n128 + 255) / 256, (uint64_t)c->sm_count * 16);
  k_dropped_scan<<<grid, 256, 0, c->stream>>>(reinterpret_cast<const uint4*>(c->d_packed.p), n128, (uint32_t)c->units, fl,
                                               mo ? mo->zero_superpop : c->d_superpop.p, c->d_af.p, c->L, c->d_n3, c->d_ecorr_scan, fx);
  KGL_LAUNCH_CHECK(c);
  if (want_moments) {
    k_moment_partials<<<blocks_for(c->N, 256), 256, 0, c->stream>>>(c->d_gcounts, c->d_n3, dense_totals(c, S), c->d_ecorr_scan, S.nz_rare(c->Npad),
                                                                    S.ecorr_fx(), 1.0 / fx, c->d_superpop.p, c->N, c->unphased ? 1 : 0,
                                                                    c->partials_target ? c->partials_target : c->d_partials.p,
                                                                    simple_results ? c->d_results.p : nullptr);
    KGL_LAUNCH_CHECK(c);
  }
  return KGL_B200_OK;
}

// Moments of all genomes over the selected loci into d_partials (phase 0 of every estimator).
int enqueue_moments(kgl_b200_ctx* c, bool want_locus_counts, bool simple_results = false, bool want_w0 = false, bool want_selw = false,
                    bool defer_join = false) {
  int rc = ensure_prepared(c, want_w0, want_selw);
  if (rc) return rc;
  KGL_CUDA(c, c->d_partials.ensure((size_t)c->Npad * PART_COUNT));
  return launch_count(c, false, want_locus_counts, true, simple_results, true, nullptr, defer_join);
}

// ---- multi-allelic loci: their share of a pass, added to what the dense path left on the context stream -----------------
int multi_launch_prepare(kgl_b200_ctx* c) {
  KGL_CUDA(c, c->d_multi_tab.ensure((size_t)c->n_pop * c->n_multi));
  k_multi_prepare<<<blocks_for(c->n_multi * c->n_pop, 128), 128, 0, c->stream>>>(c->d_multi_rows.p, c->d_multi_af.p, c->d_sel.p, c->n_multi,
                                                                                 (int)c->n_pop, c->d_multi_tab.p);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

template <int MODE>
int multi_launch_terms(kgl_b200_ctx* c, const double* d_grid, int n_grid, uint64_t& n_chunks) {
  n_chunks = (c->n_multi + kMultiChunk - 1) / kMultiChunk;
  KGL_CUDA(c, c->d_multi_out.ensure((size_t)n_chunks * c->Npad * multi_n_out(MODE)));
  MultiParams P{};
  P.cells = c->d_multi_cells.p; P.n_multi = c->n_multi; P.n_genomes = c->N; P.n_genomes_padded = c->Npad;
  P.tab = c->d_multi_tab.p; P.superpop = c->d_superpop.p; P.unphased = c->unphased ? 1 : 0;
  P.f = c->d_f.p; P.grid = d_grid; P.n_grid = n_grid; P.out = c->d_multi_out.p;
  k_multi_terms<MODE><<<dim3(blocks_for(c->N, 128), (unsigned)n_chunks), 128, 0, c->stream>>>(P);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

// MOMENTS into the partial sums (after everything the dense path writes there), HALL / NEWTON into the iteration terms.
template <int MODE>
int multi_add(kgl_b200_ctx* c, double* target, kgl_b200_locus_results* results = nullptr) {
  if (c->n_multi == 0) return KGL_B200_OK;
  int rc = KGL_B200_OK;
  if (MODE == MULTI_MOMENTS) { rc = multi_launch_prepare(c); if (rc) return rc; }
  uint64_t n_chunks = 0;
  rc = multi_launch_terms<MODE>(c, nullptr, 0, n_chunks); if (rc) return rc;
  k_multi_add<MODE><<<blocks_for(c->N, 128), 128, 0, c->stream>>>(c->d_multi_out.p, n_chunks, c->Npad, c->N, target, results);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

struct TermLaunch { dim3 grid; uint32_t words_per_chunk; uint64_t n_chunks; };

TermLaunch plan_terms(const kgl_b200_ctx* c) {
  TermLaunch t;
  const uint64_t gx = (c->n_gblocks + kTermWarps - 1) / kTermWarps;
  // aim for ~4 waves of CTAs; chunks are multiples of the shared-memory tile
  uint64_t want_chunks = std::max<uint64_t>(1, ((uint64_t)c->sm_count * 8 + gx - 1) / gx);
  uint64_t wpc = (c->n_words + want_chunks - 1) / want_chunks;
  wpc = std::max<uint64_t>(kTermTileWords, (wpc + kTermTileWords - 1) / kTermTileWords * kTermTileWords);
  t.words_per_chunk = (uint32_t)wpc;
  t.n_chunks = (c->n_words + wpc - 1) / wpc;
  t.grid = dim3((unsigned)gx, (unsigned)t.n_chunks);
  return t;
}

// What a k_genome_terms launch of either mode reads; its chunk outputs go to out ([tl.n_chunks][Npad][n_out]).
TermParams term_params(const kgl_b200_ctx* c, const TermLaunch& tl, double* out, int n_out) {
  TermParams P{};
  P.sm_lo = c->d_sm_lo.p; P.sm_hi = c->d_sm_hi.p;
  P.n_gblocks = c->n_gblocks; P.n_words = c->n_words; P.n_loci = c->L; P.n_genomes = c->N;
  P.selw = c->prep[c->par].selw.p; P.af = c->d_af.p; P.superpop = c->d_superpop.p; P.n_pop = (int)c->n_pop;
  P.unphased = c->unphased ? 1 : 0; P.words_per_chunk = tl.words_per_chunk;
  P.f = c->d_f.p; P.out = out; P.n_out = n_out; P.n_genomes_padded = c->Npad;
  return P;
}

// The log-likelihood at the n_grid values of d_grid, per genome and chunk of words, into d_chunk_out.
int launch_grid_terms(kgl_b200_ctx* c, const double* d_grid, int n_grid, TermLaunch& tl) {
  int rc = ensure_sample_major(c);
  if (rc) return rc;
  tl = plan_terms(c);
  KGL_CUDA(c, c->d_chunk_out.ensure((size_t)tl.n_chunks * c->Npad * kGridMax));
  TermParams P = term_params(c, tl, c->d_chunk_out.p, kGridMax);
  P.grid = d_grid; P.n_grid = n_grid;
  k_genome_terms<TERM_GRID><<<tl.grid, kTermWarps * 32, 0, c->stream>>>(P);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

// Interleaved 2-bit copy of the sample-major planes for the table-driven sweeps (built on first use, as the planes are).
int ensure_sample_codes(kgl_b200_ctx* c) {
  int rc = ensure_sample_major(c);
  if (rc) return rc;
  if (c->codes_valid) return KGL_B200_OK;
  const size_t n = (size_t)c->n_gblocks * c->n_words * 32;
  KGL_CUDA(c, c->d_sm_codes.ensure(n));
  k_to_sample_codes<<<blocks_for(n, 256), 256, 0, c->stream>>>(c->d_sm_lo.p, c->d_sm_hi.p, n, c->d_sm_codes.p);
  KGL_LAUNCH_CHECK(c);
  c->codes_valid = true;
  return KGL_B200_OK;
}

// Table-driven sweeps (terms_fast.cuh). One CTA per SM walks a contiguous range of 128-locus tiles over all genome blocks.
struct FastLaunch { dim3 grid; uint32_t tiles_per_chunk, slots; uint64_t n_chunks; };

template <int MODE>
int launch_fast(kgl_b200_ctx* c, FastLaunch& fl, uint64_t list_len = 0) {
  int rc = ensure_sample_major(c);
  if (rc) return rc;
  const uint64_t gblocks = list_len ? (list_len + 31) / 32 : std::min<uint64_t>(c->n_gblocks, (c->N + 31) / 32);
  // warps per CTA: of 16..32 the count that leaves the fewest genome-block slots empty (more warps on a tie)
  int warps = 16; double best = -1.0;
  for (int w = 16; w <= kFastMaxWarps; ++w) {
    const uint64_t sl = std::min<uint64_t>(8, (gblocks + w - 1) / w);
    const uint64_t rows = (gblocks + (uint64_t)w * sl - 1) / ((uint64_t)w * sl);
    const double filled = (double)gblocks / (double)(rows * sl * w);
    if (filled >= best) { best = filled; warps = w; }
  }
  // A handful of genome blocks (late Newton sweeps over the list of unfinished genomes, small populations) cannot fill 16
  // warps: small CTAs instead, four of them per SM, each with a quarter of the tiles -- the sweep is then bound by the
  // per-tile latency of a few warps, and four CTAs per SM overlap it.
  int ctas_per_sm = 1;
  if (gblocks <= 8) { warps = gblocks <= 4 ? 4 : 8; ctas_per_sm = 4; }
  const uint32_t slots = (uint32_t)std::min<uint64_t>(8, (gblocks + warps - 1) / warps);
  const uint64_t gy = (gblocks + (uint64_t)warps * slots - 1) / ((uint64_t)warps * slots);
  // only the tiles of the selection window are swept (a contig is usually analysed in many short windows)
  const uint64_t all_tiles = (c->n_words + kFastTileWords - 1) / kFastTileWords;
  const uint64_t tile_begin = std::min<uint64_t>(all_tiles, c->sel_row_lo / kFastTile);
  const uint64_t tile_end = std::max<uint64_t>(tile_begin, std::min<uint64_t>(all_tiles, c->sel_row_hi == ~0ull ? all_tiles : (c->sel_row_hi + kFastTile - 1) / kFastTile));
  const uint64_t n_tiles = std::max<uint64_t>(1, tile_end - tile_begin);
  const uint64_t want = std::max<uint64_t>(1, (uint64_t)c->sm_count * ctas_per_sm / gy);
  const uint64_t tpc = std::max<uint64_t>(1, (n_tiles + want - 1) / want);
  fl.tiles_per_chunk = (uint32_t)tpc; fl.slots = slots;
  fl.n_chunks = (n_tiles + tpc - 1) / tpc;
  fl.grid = dim3((unsigned)fl.n_chunks, (unsigned)gy);
  constexpr int NACC = FastAcc<MODE>::N;
  KGL_CUDA(c, c->d_chunk_out.ensure((size_t)fl.n_chunks * c->Npad * NACC));
  rc = ensure_sample_codes(c);
  if (rc) return rc;
  FastParams P{};
  P.codes = c->d_sm_codes.p;
  P.n_gblocks = gblocks; P.n_words = c->n_words; P.n_loci = c->L; P.n_genomes = c->N; P.n_genomes_padded = c->Npad;
  P.selw = c->prep[c->par].selw.p; P.af = c->d_af.p; P.superpop = c->d_superpop.p; P.n_pop = (int)c->n_pop;
  P.unphased = c->unphased ? 1 : 0; P.tiles_per_chunk = fl.tiles_per_chunk; P.slots = slots;
  P.tile_begin = tile_begin; P.tile_end = tile_end;
  P.f = c->d_f.p; P.out = c->d_chunk_out.p;
  P.list = list_len ? c->d_list.p : nullptr; P.n_list = list_len; P.n_list_dev = list_len ? c->d_list_count.p : nullptr;
  if (MODE == FAST_HALL || MODE == FAST_NEWTON) {
    // the per-locus constants of the run: built before its first sweep, reused by every later one
    if (c->table_mode != MODE) {
      KGL_CUDA(c, c->d_terms_table.ensure((size_t)c->n_pop * c->n_words * 32));
      k_terms_table<MODE><<<dim3(blocks_for(c->n_words * 32, 256), c->n_pop), 256, 0, c->stream>>>(
          c->prep[c->par].selw.p, c->d_af.p, c->L, c->n_words, (int)c->n_pop, c->unphased ? 1 : 0, c->d_terms_table.p);
      KGL_LAUNCH_CHECK(c);
      c->table_mode = MODE;
    }
    P.table = c->d_terms_table.p;
  }
  const size_t smem = fast_smem_bytes(MODE, slots, warps);
  KGL_CUDA(c, cudaFuncSetAttribute(k_terms_fast<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_terms_fast<MODE><<<fl.grid, warps * 32, smem, c->stream>>>(P);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

// The exact cell-by-cell evaluation for the genomes a Newton reduction marked (none in the normal case: the kernels then
// return at once).
int newton_exact_tail(kgl_b200_ctx* c) {
  const unsigned nb = blocks_for(c->N, 256);
  TermLaunch tl = plan_terms(c);
  KGL_CUDA(c, c->d_slow_out.ensure((size_t)tl.n_chunks * c->Npad * 4));
  TermParams P = term_params(c, tl, c->d_slow_out.p, 4);
  P.lane_state = c->d_lane_state.p; P.n_slow = c->d_n_slow.p;
  k_genome_terms<TERM_NEWTON><<<tl.grid, kTermWarps * 32, 0, c->stream>>>(P);
  KGL_LAUNCH_CHECK(c);
  k_newton_add_slow<<<nb, 256, 0, c->stream>>>(c->d_slow_out.p, tl.n_chunks, c->Npad, c->N, c->d_lane_state.p, c->d_n_slow.p, c->d_iter.p);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

// The end of every Newton sweep: the reduction of its chunk outputs in d_chunk_out (n_out per genome and chunk; the sums hold
// for f >= valid_min) and the exact evaluation for the genomes the reduction marks.
int newton_reduce(kgl_b200_ctx* c, int n_out, uint64_t n_chunks, double valid_min) {
  KGL_CUDA(c, cudaMemsetAsync(c->d_n_slow.p, 0, 4, c->stream));
  k_newton_reduce<<<blocks_for((c->list_len ? c->list_len : c->N) * 8, 256), 256, 0, c->stream>>>(
      c->d_chunk_out.p, n_out, n_chunks, c->Npad, c->N, c->list_len ? c->d_list.p : nullptr, c->list_len,
      c->list_len ? c->d_list_count.p : nullptr, c->d_f.p,
      c->d_limits.p, c->d_done.p, valid_min, c->d_iter.p, c->d_lane_state.p, c->d_n_slow.p);
  KGL_LAUNCH_CHECK(c);
  return newton_exact_tail(c);
}

// One Newton sweep of the log-likelihood root search on the table-driven kernel.
template <int MODE>
int newton_sweep(kgl_b200_ctx* c) {
  FastLaunch fl;
  int rc = launch_fast<MODE>(c, fl, c->list_len); if (rc) return rc;
  return newton_reduce(c, FastAcc<MODE>::N, fl.n_chunks, -kHuge);
}

// ---- moment tables (terms_moments.cuh) ------------------------------------------------------------------------------------
__global__ void k_mom_stats_init(int* stats) { stats[0] = kMomBinsMax; stats[1] = -1; stats[2] = 0; stats[3] = 0; }
__global__ void k_mom_copy_limits(const double* __restrict__ src, uint64_t n, double* __restrict__ limits) {
  const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n) { limits[g * 3 + 0] = src[g * 3 + 0]; limits[g * 3 + 1] = src[g * 3 + 1]; }
}

// Whether the estimator run may sweep from the moment tables (ensure_moments may still find them unsupported). HallME: every
// start lies in [0,1] -- the tables cover f >= 0 without the lists, and a start there stays there (calc.cpp:285). The root
// search: phased genotypes only.
bool moments_enabled(const kgl_b200_ctx* c) {
  if (c->opt.exact_sweeps) return false;
  if (c->algo != KGL_B200_ALGO_HALLME) return !c->unphased;
  for (double v : c->hall_start) if (!(v >= 0.0 && v <= 1.0)) return false;
  return true;
}

// The root search's limits of the feasible region, from the moment lists.
int copy_moment_limits(kgl_b200_ctx* c) {
  k_mom_copy_limits<<<blocks_for(c->N, 256), 256, 0, c->stream>>>(c->d_mom_limits.p, c->N, c->d_limits.p);
  KGL_LAUNCH_CHECK(c);
  c->limits_valid = true;
  return KGL_B200_OK;
}

// Tiles (of tile_genomes genomes) that hold a genome of each population, from the host copy of the assignment; returns the widest range.
uint32_t moment_tile_ranges(const kgl_b200_ctx* c, uint32_t tile_genomes, uint32_t (&lo)[kMaxPop], uint32_t (&hi)[kMaxPop]) {
  uint32_t widest = 1;
  for (int k = 0; k < kMaxPop; ++k) { lo[k] = 0xFFFFFFFFu; hi[k] = 0; }
  for (uint64_t g = 0; g < c->N; ++g) {
    const int k = g < c->h_superpop.size() ? c->h_superpop[g] : 0;
    if (k >= kMaxPop) continue;
    const uint32_t t = (uint32_t)(g / tile_genomes);
    lo[k] = std::min(lo[k], t); hi[k] = std::max(hi[k], t + 1);
  }
  for (int k = 0; k < kMaxPop; ++k) { if (hi[k] == 0) lo[k] = 0; widest = std::max(widest, hi[k] - lo[k]); }
  return widest;
}

// The lists of rare homozygous cells and the limits of the feasible region, after either builder has left the per-genome list
// lengths in d_mom_totals: the list offsets (k_mom_base), the list sized on the host, fill() (the builder's own fill kernel), the
// limits.
template <class Fill>
int moments_lists(kgl_b200_ctx* c, Fill fill) {
  cudaStream_t st = c->stream;
  k_mom_base<<<1, 1024, 0, st>>>(c->d_mom_totals.p, c->N, c->d_mom_base.p);
  KGL_LAUNCH_CHECK(c);
  uint64_t list_len = 0;
  KGL_CUDA(c, cudaMemcpyAsync(&list_len, c->d_mom_base.p + c->N, 8, cudaMemcpyDeviceToHost, st));
  KGL_CUDA(c, cudaStreamSynchronize(st));
  KGL_CUDA(c, c->d_mom_list.ensure_roomy(std::max<uint64_t>(1, list_len)));
  int rc = fill(); if (rc) return rc;
  k_mom_list_limits<<<blocks_for(c->N, 256), 256, 0, st>>>(c->d_mom_list.p, c->d_mom_base.p, c->d_mom_totals.p, c->d_superpop.p,
                                                           c->d_mom_pop_cmin.p, c->N, c->d_mom_limits.p);
  KGL_LAUNCH_CHECK(c);
  c->mom_lists = true;
  return KGL_B200_OK;
}

// The lists from the per-unit counts the tensor-core builder left.
int moments_build_lists(kgl_b200_ctx* c) {
  cudaStream_t st = c->stream;
  const uint64_t N = c->N, npad = c->Npad;
  KGL_CUDA(c, c->d_mom_unit_offs.ensure_roomy((size_t)c->mom_n_units * npad));
  k_mom_unit_scan<<<blocks_for(N, 32), 256, 0, st>>>(c->d_mom_unit_cnt.p, c->d_mom_units.p, c->d_mom_unit_range.p, c->d_superpop.p, N, npad,
                                                     c->d_mom_unit_offs.p, c->d_mom_totals.p);
  KGL_LAUNCH_CHECK(c);
  int rc = moments_lists(c, [&] {
    MomFillParams F{};
    F.packed = reinterpret_cast<const uint4*>(c->d_packed.p); F.units = c->units; F.rr = c->d_mom_rr.p;
    F.superpop = c->d_superpop.p; F.n_genomes = N; F.n_genomes_padded = npad; F.rows = c->d_mom_rows2.p; F.unit_table = c->d_mom_units.p;
    F.cnt = c->d_mom_unit_cnt.p; F.offs = c->d_mom_unit_offs.p; F.totals = c->d_mom_totals.p; F.base = c->d_mom_base.p; F.list = c->d_mom_list.p;
    const uint32_t fill_tiles = moment_tile_ranges(c, kMomTile, F.tile_lo, F.tile_hi);
    F.tiles_per_unit = fill_tiles;
    F.rare_bits = c->d_mom_rare_bits.p; F.mma_tiles_per_unit = c->mom_mma_tiles;
    for (int k = 0; k < kMaxPop; ++k) { F.mma_tile_lo[k] = c->mom_mma_tile_lo[k]; F.mma_tile_hi[k] = c->mom_mma_tile_hi[k]; }
    k_mom_unit_fill<<<(unsigned)((uint64_t)fill_tiles * c->mom_n_units), kMomTile, 0, st>>>(F);
    KGL_LAUNCH_CHECK(c);
    return KGL_B200_OK;
  });
  if (rc) return rc;
  c->launches += 4;
  return KGL_B200_OK;
}

// Builds the per-genome moment tables of the current selection (and, for the root search, the lists of rare homozygous cells
// and the limits of the feasible region). mom_supported = false afterwards: the selection has a frequency outside the bins, or
// the tables would not fit -- the caller then sweeps with the exact kernels.
int ensure_moments(kgl_b200_ctx* c, bool want_lists) {
  if (c->mom_valid && (!c->mom_supported || c->mom_lists || !want_lists)) return KGL_B200_OK;
  if (c->mom_valid && c->mom_supported && c->mom_used_mma && c->mom_cnt_valid) return moments_build_lists(c);   // tables of an earlier HallME run: only the lists are missing
  c->mom_valid = true; c->mom_lists = false; c->mom_supported = false; c->mom_used_mma = false; c->mom_cnt_valid = false;
  int rc = ensure_sample_major(c); if (rc) return rc;       // the exact fallback reads the sample-major planes
  const uint64_t L = c->L, N = c->N, npad = c->Npad;
  const uint64_t row_lo = std::min<uint64_t>(L, c->sel_row_lo), row_hi = c->sel_row_hi == ~0ull ? L : std::min<uint64_t>(L, c->sel_row_hi);
  const uint64_t W = row_hi > row_lo ? row_hi - row_lo : 0, n_items = W * c->n_pop;
  if (W == 0 || n_items >= 0xFFFFFFFFull || !c->prep[c->par].selw.p) return KGL_B200_OK;
  cudaStream_t st = c->stream;
  const int unph = c->unphased ? 1 : 0;
  KGL_CUDA(c, c->d_mom_keys.ensure_roomy(n_items)); KGL_CUDA(c, c->d_mom_keys2.ensure_roomy(n_items));
  KGL_CUDA(c, c->d_mom_rows.ensure_roomy(n_items)); KGL_CUDA(c, c->d_mom_rows2.ensure_roomy(n_items));
  KGL_CUDA(c, c->d_mom_stats.ensure_roomy(4)); KGL_CUDA(c, c->d_mom_pop_begin.ensure_roomy(kMaxPop + 2));
  KGL_CUDA(c, c->d_mom_pop_cmin.ensure_roomy(kMaxPop));
  KGL_CUDA(c, c->d_mom_bounds.ensure_roomy(kMomMaxUnits)); KGL_CUDA(c, c->d_mom_bounds2.ensure_roomy(kMomMaxUnits));
  KGL_CUDA(c, c->d_mom_units.ensure_roomy(kMomMaxUnits)); KGL_CUDA(c, c->d_mom_unit_range.ensure_roomy(kMaxPop));
  KGL_CUDA(c, c->d_mom_unit_out.ensure_roomy(4));
  k_mom_stats_init<<<1, 1, 0, st>>>(c->d_mom_stats.p);
  KGL_CUDA(c, cudaMemsetAsync(c->d_mom_pop_cmin.p, 0xFF, kMaxPop * 8, st));
  KGL_CUDA(c, cudaMemsetAsync(c->d_mom_bounds.p, 0xFF, kMomMaxUnits * 4, st));
  KGL_CUDA(c, cudaMemsetAsync(c->d_mom_unit_out.p, 0, 16, st));
  k_mom_keys<<<dim3(blocks_for(W, 256), (unsigned)c->n_pop), 256, 0, st>>>(c->prep[c->par].selw.p, c->d_af.p, L, c->n_words, row_lo, W, unph,
                                                                           c->d_mom_keys.p, c->d_mom_rows.p, c->d_mom_stats.p, c->d_mom_pop_cmin.p);
  KGL_LAUNCH_CHECK(c);
  size_t temp_bytes = 0, temp2 = 0;
  KGL_CUDA(c, cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, c->d_mom_keys.p, c->d_mom_keys2.p, c->d_mom_rows.p, c->d_mom_rows2.p,
                                              n_items, 0, 35, st));
  KGL_CUDA(c, cub::DeviceRadixSort::SortKeys(nullptr, temp2, c->d_mom_bounds.p, c->d_mom_bounds2.p, (uint64_t)kMomMaxUnits, 0, 32, st));
  KGL_CUDA(c, c->d_mom_tmp.ensure_roomy(std::max(temp_bytes, temp2)));
  KGL_CUDA(c, cub::DeviceRadixSort::SortPairs(c->d_mom_tmp.p, temp_bytes, c->d_mom_keys.p, c->d_mom_keys2.p, c->d_mom_rows.p, c->d_mom_rows2.p,
                                              n_items, 0, 35, st));
  k_mom_ranges<<<1, 32, 0, st>>>(c->d_mom_keys2.p, n_items, (int)c->n_pop, c->d_mom_pop_begin.p);
  KGL_LAUNCH_CHECK(c);
  // units of the tensor-core builder: boundaries, sorted, then the unit table
  uint32_t* d_n_bounds = c->d_mom_unit_out.p + 3;
  k_mom_bounds<<<blocks_for(n_items, 256), 256, 0, st>>>(c->d_mom_keys2.p, c->d_mom_rows2.p, c->d_mom_pop_begin.p, (int)c->n_pop, c->d_af.p, L,
                                                         unph, c->d_mom_bounds.p, d_n_bounds);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cub::DeviceRadixSort::SortKeys(c->d_mom_tmp.p, temp2, c->d_mom_bounds.p, c->d_mom_bounds2.p, (uint64_t)kMomMaxUnits, 0, 32, st));
  k_mom_units<<<1, 1024, 0, st>>>(c->d_mom_bounds2.p, d_n_bounds, c->d_mom_keys2.p, c->d_mom_rows2.p, c->d_mom_pop_begin.p, (int)c->n_pop,
                                  c->d_af.p, L, unph, c->d_mom_units.p, c->d_mom_unit_range.p, c->d_mom_unit_out.p);
  KGL_LAUNCH_CHECK(c);
  int stats[4]; uint32_t pop_begin[kMaxPop + 2]; uint32_t unit_out[4];
  KGL_CUDA(c, cudaMemcpyAsync(stats, c->d_mom_stats.p, sizeof stats, cudaMemcpyDeviceToHost, st));
  KGL_CUDA(c, cudaMemcpyAsync(pop_begin, c->d_mom_pop_begin.p, (c->n_pop + 1) * 4, cudaMemcpyDeviceToHost, st));
  KGL_CUDA(c, cudaMemcpyAsync(unit_out, c->d_mom_unit_out.p, sizeof unit_out, cudaMemcpyDeviceToHost, st));
  KGL_CUDA(c, cudaStreamSynchronize(st));
  if (stats[2] > 0 || stats[1] < stats[0]) return KGL_B200_OK;      // a frequency outside the bins / nothing selected: exact kernels
  const int b_lo = stats[0], nbt = stats[1] - stats[0] + 2;           // + the a == 1 class
  static const uint64_t limit_bytes = [] { const char* e = std::getenv("KGL_B200_MOMENT_BYTES"); return e ? std::strtoull(e, nullptr, 10) : (16ull << 30); }();
  if ((uint64_t)npad * nbt * kMomJ * 8 > limit_bytes) return KGL_B200_OK;
  uint32_t longest = 0;
  for (uint32_t k = 0; k < c->n_pop; ++k) longest = std::max(longest, pop_begin[k + 1] - pop_begin[k]);
  int sbits = 61; for (uint64_t v = longest; v; v >>= 1) --sbits;
  const double scale = std::ldexp(1.0, std::min(sbits, 46));          // the tensor-core payload has six 8-bit limbs for U + 2^s
  const uint32_t n_units = unit_out[0], n_btiles = unit_out[1];
  // scratch of the tensor-core builder (payload tiles, per-unit counts and offsets)
  // (a quarter of the device's memory, from the properties read at kgl_b200_create: cudaMemGetInfo stalls the host for milliseconds)
  const uint64_t scratch_limit = std::max<uint64_t>(4ull << 30, c->total_memory / 4);
  const bool use_mma = !c->opt.moments_on_cuda_cores && unit_out[2] <= kMomMaxUnits && n_units > 0 &&
                       (uint64_t)n_btiles * 2 * kMmaBTile + (want_lists ? (uint64_t)n_units * npad * 8 : 0) <= scratch_limit;
  KGL_CUDA(c, c->d_mom_pm.ensure_roomy((size_t)c->n_pop * nbt * kMomJ));
  KGL_CUDA(c, c->d_mom_mi.ensure_roomy((size_t)npad * nbt * kMomJ));
  KGL_CUDA(c, c->d_mom_totals.ensure_roomy((size_t)npad * 2));
  KGL_CUDA(c, c->d_mom_limits.ensure_roomy((size_t)npad * 3));
  KGL_CUDA(c, c->d_mom_base.ensure_roomy(N + 1));
  KGL_CUDA(c, cudaMemsetAsync(c->d_mom_pm.p, 0, (size_t)c->n_pop * nbt * kMomJ * 8, st));
  KGL_CUDA(c, cudaMemsetAsync(c->d_mom_mi.p, 0, (size_t)npad * nbt * kMomJ * 8, st));
  if (!use_mma) {              // the tensor-core path sums the population's moments while it writes the payload tiles (k_mom_btiles)
    k_mom_dense<<<blocks_for(pop_begin[c->n_pop], 256), 256, 0, st>>>(c->d_mom_keys2.p, c->d_mom_rows2.p, c->d_mom_pop_begin.p, (int)c->n_pop,
                                                                      c->d_af.p, L, unph, b_lo, nbt, scale, c->d_mom_pm.p);
    KGL_LAUNCH_CHECK(c);
  }
  if (use_mma) {
    KGL_CUDA(c, c->d_mom_btiles.ensure_roomy((size_t)std::max<uint32_t>(1, n_btiles) * 2 * kMmaBTile));
    KGL_CUDA(c, c->d_mom_rr.ensure_roomy(n_items));
    k_mom_btiles<<<n_units, kMmaK, 0, st>>>(c->d_mom_units.p, c->d_mom_rows2.p, c->d_af.p, L, unph, scale, c->d_mom_btiles.p, c->d_mom_rr.p, b_lo, nbt, c->d_mom_pm.p);
    KGL_LAUNCH_CHECK(c);
    if (want_lists) { KGL_CUDA(c, c->d_mom_unit_cnt.ensure_roomy((size_t)n_units * npad)); KGL_CUDA(c, c->d_mom_unit_offs.ensure_roomy((size_t)n_units * npad)); }
    const bool keep_counts = want_lists || (uint64_t)n_units * npad * 8 <= (2ull << 30);     // lets a later root search add its lists to these tables
    if (keep_counts) KGL_CUDA(c, c->d_mom_unit_cnt.ensure_roomy((size_t)n_units * npad));
    MomMmaParams M{};
    const uint32_t mma_tiles = moment_tile_ranges(c, kMmaM, M.tile_lo, M.tile_hi);
    M.packed = reinterpret_cast<const uint4*>(c->d_packed.p); M.units = c->units;
    M.superpop = c->d_superpop.p; M.n_genomes = N; M.n_genomes_padded = npad;
    M.rows = c->d_mom_rows2.p; M.unit_table = c->d_mom_units.p; M.btiles = c->d_mom_btiles.p;
    M.b_lo = b_lo; M.nbt = nbt; M.scale = scale; M.mi = c->d_mom_mi.p; M.cnt = keep_counts ? c->d_mom_unit_cnt.p : nullptr;
    M.tiles_per_unit = mma_tiles;
    M.rare_bits = nullptr;
    if (keep_counts) {          // the bitmap of the rows the list pass has to load
      KGL_CUDA(c, c->d_mom_rare_bits.ensure_roomy((size_t)std::max<uint32_t>(1, n_btiles) * mma_tiles * 4));
      KGL_CUDA(c, cudaMemsetAsync(c->d_mom_rare_bits.p, 0, (size_t)std::max<uint32_t>(1, n_btiles) * mma_tiles * 16, st));
      M.rare_bits = c->d_mom_rare_bits.p;
    }
    for (int k = 0; k < kMaxPop; ++k) { c->mom_mma_tile_lo[k] = M.tile_lo[k]; c->mom_mma_tile_hi[k] = M.tile_hi[k]; }
    c->mom_mma_tiles = mma_tiles;
    k_mom_mma<<<(unsigned)((uint64_t)mma_tiles * n_units), kMmaM, 0, st>>>(M);
    KGL_LAUNCH_CHECK(c);
    c->mom_n_units = n_units; c->mom_cnt_valid = keep_counts;
    if (want_lists) { rc = moments_build_lists(c); if (rc) return rc; }
    c->mom_used_mma = true;
  } else {
    const uint32_t chunks_per_pop = (longest + kMomChunk - 1) / kMomChunk;
    KGL_CUDA(c, c->d_mom_cnt.ensure_roomy((size_t)chunks_per_pop * npad));
    if (want_lists) KGL_CUDA(c, c->d_mom_offs.ensure_roomy((size_t)chunks_per_pop * npad));
    MomParams P{};
    P.packed = reinterpret_cast<const uint4*>(c->d_packed.p); P.units = c->units;
    P.af = c->d_af.p; P.n_loci = L; P.n_pop = (int)c->n_pop; P.unphased = unph;
    P.superpop = c->d_superpop.p; P.n_genomes = N; P.n_genomes_padded = npad;
    P.rows = c->d_mom_rows2.p; P.pop_begin = c->d_mom_pop_begin.p; P.chunks_per_pop = chunks_per_pop;
    P.b_lo = b_lo; P.nbt = nbt; P.scale = scale;
    P.mi = c->d_mom_mi.p; P.cnt = c->d_mom_cnt.p;
    const dim3 grid((unsigned)(c->n_pop * chunks_per_pop), (unsigned)((N + kMomTile - 1) / kMomTile));
    k_mom_build<<<grid, kMomTile, 0, st>>>(P);          // the limits of the root search come from the lists (k_mom_list_limits)
    KGL_LAUNCH_CHECK(c);
    k_mom_scan<<<blocks_for(N, 256), 256, 0, st>>>(c->d_mom_cnt.p, c->d_mom_pop_begin.p, c->d_superpop.p, N, npad, c->d_mom_totals.p,
                                                   want_lists ? c->d_mom_offs.p : nullptr);
    KGL_LAUNCH_CHECK(c);
    if (want_lists) {
      rc = moments_lists(c, [&] {
        P.base = c->d_mom_base.p; P.offs = c->d_mom_offs.p; P.list = c->d_mom_list.p;
        k_mom_fill<<<grid, kMomTile, 0, st>>>(P, c->d_mom_totals.p);
        KGL_LAUNCH_CHECK(c);
        return KGL_B200_OK;
      });
      if (rc) return rc;
    }
  }
  k_mom_finalize<<<blocks_for(N * (uint64_t)nbt, 256), 256, 0, st>>>(c->d_mom_mi.p, c->d_mom_pm.p, c->d_superpop.p, N, nbt, 1.0 / scale);
  KGL_LAUNCH_CHECK(c);
  c->launches += 12;
  c->mom_b_lo = b_lo; c->mom_nbt = nbt; c->mom_supported = true;
  return KGL_B200_OK;
}

// One Newton sweep from the moment tables: one chunk of two sums per genome.
int newton_sweep_moments(kgl_b200_ctx* c) {
  KGL_CUDA(c, c->d_chunk_out.ensure((size_t)c->Npad * 2));
  k_mom_eval<FAST_NEWTON><<<(unsigned)(c->list_len ? c->list_len : c->N), 128, 0, c->stream>>>(
      reinterpret_cast<const double*>(c->d_mom_mi.p), c->mom_b_lo, c->mom_nbt, c->d_f.p, c->list_len ? c->d_list.p : nullptr, c->list_len,
      c->list_len ? c->d_list_count.p : nullptr, c->N, c->d_mom_list.p, c->d_mom_base.p, c->d_mom_totals.p, c->d_chunk_out.p, nullptr);
  KGL_LAUNCH_CHECK(c);
  return newton_reduce(c, 2, 1, kMomValidMin);
}

// ---- pairwise IBS ----------------------------------------------------------------------------------------------------
// Planes of the dense kernel. No code-3 cell: the sample-major copy as it is. Indexed code-3 cells: pre-masked copies, the
// sparse repair kernel does the rest. Otherwise: a validity plane and the three-plane kernel.
int ensure_ibs_planes(kgl_b200_ctx* c) {
  int rc = ensure_sample_major(c); if (rc) return rc;
  rc = build_dropped_index(c); if (rc) return rc;
  if (c->ibs_mode >= 0) return KGL_B200_OK;
  const size_t n = (size_t)c->n_gblocks * c->n_words * 32;
  const unsigned nb = blocks_for(n / 4, 256);
  if (c->n_dropped == 0) {
    c->ibs_mode = 0;
  } else if (c->dropped_indexed) {
    KGL_CUDA(c, c->d_ibs_lo.ensure(n));
    KGL_CUDA(c, c->d_ibs_hi.ensure(n));
    k_ibs_premask<<<nb, 256, 0, c->stream>>>(reinterpret_cast<const uint4*>(c->d_sm_lo.p), reinterpret_cast<const uint4*>(c->d_sm_hi.p), n / 4,
                                              reinterpret_cast<uint4*>(c->d_ibs_lo.p), reinterpret_cast<uint4*>(c->d_ibs_hi.p));
    KGL_LAUNCH_CHECK(c);
    c->ibs_mode = 2;
  } else {
    KGL_CUDA(c, c->d_sm_valid.ensure(n));
    k_valid_plane<<<nb, 256, 0, c->stream>>>(reinterpret_cast<const uint4*>(c->d_sm_lo.p), reinterpret_cast<const uint4*>(c->d_sm_hi.p), n / 4,
                                              reinterpret_cast<uint4*>(c->d_sm_valid.p));
    KGL_LAUNCH_CHECK(c);
    c->ibs_mode = 1;
  }
  return KGL_B200_OK;
}

uint64_t ibs_side(const kgl_b200_ctx* c) { return (c->N + kIbsT - 1) / kIbsT; }

// Row pitch of the Gram matrices and code matrices (gram_i8.cuh), and the k-stages of a Gram run over all loci.
uint64_t gram_ld(const kgl_b200_ctx* c) { return (c->N + kGramN - 1) / kGramN * kGramN; }
uint32_t gram_k_stages(const kgl_b200_ctx* c) { return (uint32_t)((c->L + kGramK - 1) / kGramK); }

// t-th tile of the row-major upper triangle (ti <= tj) of a side x side tile grid.
uint2 ibs_upper_tile(uint64_t t, uint64_t side) {
  // row ti starts at ti*side - ti*(ti-1)/2
  uint64_t lo = 0, hi = side - 1;
  while (lo < hi) {
    const uint64_t mid = (lo + hi + 1) / 2;
    const uint64_t start = mid * side - mid * (mid - 1) / 2;
    if (start <= t) lo = mid; else hi = mid - 1;
  }
  const uint64_t start = lo * side - lo * (lo - 1) / 2;
  return make_uint2((uint32_t)lo, (uint32_t)(lo + (t - start)));
}

constexpr uint64_t kIbsMaxTilesPerLaunch = 8192;     // 384 MB of accumulators

// Tiles first, first + stride, ... (count of them) of the row-major upper triangle.
TileList upper_tiles(uint64_t first, uint64_t stride, uint64_t count) { return {{TileKey::kUpper, first, stride, count}, {}}; }

// Every tile of the tile rows [tr0, tr1).
TileList band_tiles(uint64_t tr0, uint64_t tr1, uint64_t side) { return {{TileKey::kBand, tr0, tr1, (tr1 - tr0) * side}, {}}; }

// count tiles {row, column} from the host, each inside the grid and, when upper_only, not below the diagonal.
int listed_tiles(kgl_b200_ctx* c, const uint32_t* coords, uint64_t count, bool upper_only, TileList& out) {
  const uint64_t side = ibs_side(c);
  uint64_t hash = 1469598103934665603ull;
  out.coords.resize(count);
  for (uint64_t i = 0; i < count; ++i) {
    const uint32_t ti = coords[2 * i], tj = coords[2 * i + 1];
    if (ti >= side || tj >= side) return fail(c, KGL_B200_ERR_INVALID, "tile coordinate outside the grid");
    if (upper_only && ti > tj) return fail(c, KGL_B200_ERR_INVALID, "tile below the diagonal (need tile row <= tile column)");
    out.coords[i] = make_uint2(ti, tj);
    hash = (hash ^ ti) * 1099511628211ull; hash = (hash ^ tj) * 1099511628211ull;
  }
  out.key = {TileKey::kList, hash, side, count};
  return KGL_B200_OK;
}

std::vector<uint2> tile_coords(const TileList& list, uint64_t side) {
  const TileKey& k = list.key;
  if (k.kind == TileKey::kList) return list.coords;
  std::vector<uint2> tiles;
  tiles.reserve(k.n);
  if (k.kind == TileKey::kUpper) {
    for (uint64_t i = 0; i < k.n; ++i) tiles.push_back(ibs_upper_tile(k.a + i * k.b, side));
  } else {
    for (uint64_t ta = k.a; ta < k.b; ++ta)
      for (uint64_t tb = 0; tb < side; ++tb) tiles.push_back(make_uint2((uint32_t)ta, (uint32_t)tb));
  }
  return tiles;
}

// The 2-bit code matrix of every Gram run in row-block-major layout, once per upload. Code 3 is kept: each run's byte table
// reads it as 0, except the code-3 indicator of KING's M = H C^T and of PCA's code-3 run.
int ensure_codes(kgl_b200_ctx* c) {
  int rc = ensure_sample_major(c); if (rc) return rc;
  if (c->codes16_valid) return KGL_B200_OK;
  const uint64_t ld = gram_ld(c), k_stages = gram_k_stages(c);
  const size_t words = (size_t)ld * k_stages * 8;
  KGL_CUDA(c, c->d_codes16.ensure(words));
  KGL_CUDA(c, cudaMemsetAsync(c->d_codes16.p, 0, words * 4, c->stream));
  k_codes16<<<blocks_for((uint64_t)c->n_gblocks * c->n_words * 32, 256), 256, 0, c->stream>>>(c->d_sm_lo.p, c->d_sm_hi.p, c->n_gblocks,
                                                                                              c->n_words, k_stages, ld, c->d_codes16.p);
  KGL_LAUNCH_CHECK(c);
  c->codes16_valid = true;
  return KGL_B200_OK;
}

// One Gram run, table_a x table_b, over the 256 x 256 blocks under the current IBS tile list, into compact blocks: plan, clear
// the output when the run is chunked (the chunks add into it), launch.
int run_gram_blocks(kgl_b200_ctx* c, const uint32_t* codes, uint32_t table_a, uint32_t table_b, int32_t* out) {
  const uint32_t k_stages = gram_k_stages(c);
  const GramPlan gp = plan_gram(std::max<uint32_t>(c->ibs_n_blocks, 1), k_stages, c->sm_count);
  GramParams G{};
  G.codes = codes; G.k_stages = k_stages; G.tiles = c->d_ibs_blocks.p; G.n_tiles = c->ibs_n_blocks;
  G.stages_per_chunk = gp.stages_per_chunk; G.n_chunks = gp.n_chunks; G.out = out; G.ld = gram_ld(c); G.compact = 1;
  G.table_a = table_a; G.table_b = table_b;
  if (gp.n_chunks > 1) KGL_CUDA(c, cudaMemsetAsync(out, 0, (size_t)c->ibs_n_blocks * kGramM * kGramN * 4, c->stream));
  KGL_CUDA(c, launch_gram(G, gp, c->stream));
  ++c->launches;
  return KGL_B200_OK;
}

// The genomes' heterozygous / hom-alt cells on the IBS planes (code 3 in neither), once per upload.
int ensure_ibs_class(kgl_b200_ctx* c) {
  if (c->ibs_class_valid) return KGL_B200_OK;
  const size_t n_rows = (size_t)std::max<uint64_t>(c->n_gblocks * 32, gram_ld(c));
  KGL_CUDA(c, c->d_ibs_class.ensure(n_rows * 2));
  KGL_CUDA(c, cudaMemsetAsync(c->d_ibs_class.p, 0, n_rows * 2 * 4, c->stream));
  const uint32_t wpc = 4096;
  k_ibs_class_counts<<<dim3((unsigned)c->n_gblocks, (unsigned)((c->n_words + wpc - 1) / wpc)), 256, 0, c->stream>>>(
      c->ibs_mode == 2 ? c->d_ibs_lo.p : c->d_sm_lo.p, c->ibs_mode == 2 ? c->d_ibs_hi.p : c->d_sm_hi.p, c->n_words, wpc, c->d_ibs_class.p);
  KGL_LAUNCH_CHECK(c);
  c->ibs_class_valid = true;
  return KGL_B200_OK;
}

// Dense kernel (+ sparse repair) over a tile list; leaves acc[n][3][4096] in d_ibs_acc. n <= kIbsMaxTilesPerLaunch.
// want_blocks: build the 256 x 256 block list under the tiles also when the popcount kernel runs (KING's Gram runs use it).
int ibs_compute_tiles(kgl_b200_ctx* c, const TileList& list, bool want_blocks = false) {
  const uint32_t n = (uint32_t)list.key.n;
  KGL_CUDA(c, c->d_ibs_tiles.ensure(n));
  KGL_CUDA(c, c->d_ibs_acc.ensure((size_t)n * 3 * kIbsTileCells));
  // Tensor-core form of the dense part: populations whose code-3 cells are indexed (or absent), n_loci < 2^29
  const bool tensor = c->ibs_tensor_enabled && c->ibs_mode != 1 && c->L < (1ull << 29);
  const bool need_blocks = tensor || want_blocks;
  if (tensor) {
    int rc = ensure_codes(c); if (rc) return rc;
    rc = ensure_ibs_class(c); if (rc) return rc;
  }
  if (!(list.key == c->ibs_tiles_key) || (need_blocks && c->ibs_n_blocks == 0)) {
    const std::vector<uint2> tiles = tile_coords(list, ibs_side(c));
    KGL_CUDA(c, cudaMemcpyAsync(c->d_ibs_tiles.p, tiles.data(), (size_t)n * sizeof(uint2), cudaMemcpyHostToDevice, c->stream));
    std::vector<uint2> blocks;
    std::vector<uint32_t> tile_block;
    c->ibs_n_blocks = 0;                 // a list uploaded without its blocks must not inherit the block count of the one before
    if (need_blocks) {
      // the 256 x 256 Gram blocks under the tiles (upper triangle of the block grid; a tile below the diagonal uses the mirror block)
      std::unordered_map<uint64_t, uint32_t> index;
      tile_block.resize(tiles.size());
      for (size_t t = 0; t < tiles.size(); ++t) {
        uint32_t bi = tiles[t].x / kIbsTilesPerBlock, bj = tiles[t].y / kIbsTilesPerBlock;
        const bool mirrored = bi > bj;
        if (mirrored) std::swap(bi, bj);
        const uint64_t k2 = ((uint64_t)bi << 32) | bj;
        auto it = index.find(k2);
        if (it == index.end()) { it = index.emplace(k2, (uint32_t)blocks.size()).first; blocks.push_back(make_uint2(bi, bj)); }
        tile_block[t] = it->second | (mirrored ? 0x80000000u : 0u);
      }
      KGL_CUDA(c, c->d_ibs_blocks.ensure(blocks.size()));
      KGL_CUDA(c, c->d_ibs_tile_block.ensure(tile_block.size()));
      KGL_CUDA(c, cudaMemcpyAsync(c->d_ibs_blocks.p, blocks.data(), blocks.size() * sizeof(uint2), cudaMemcpyHostToDevice, c->stream));
      KGL_CUDA(c, cudaMemcpyAsync(c->d_ibs_tile_block.p, tile_block.data(), tile_block.size() * 4, cudaMemcpyHostToDevice, c->stream));
      c->ibs_n_blocks = (uint32_t)blocks.size();
    }
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));     // the lists are pageable host memory
    c->ibs_tiles_key = list.key;
  }
  if (tensor) {
    const size_t block_cells = (size_t)c->ibs_n_blocks * kGramM * kGramN;
    c->gram_valid = false;                                  // d_gram holds the dosage blocks from here on
    KGL_CUDA(c, c->d_gram.ensure(block_cells));             // (also kgl_b200_run_gram's matrix: that call sizes it for itself)
    KGL_CUDA(c, c->d_gram_hh.ensure(block_cells));
    KGL_CUDA(c, c->d_gram_aa.ensure(block_cells));
  }
  const uint32_t words_used = (uint32_t)(((c->L + 31) / 32 + 1) / 2 * 2);
  const IbsPlan pl = plan_ibs(n, words_used, c->sm_count);
  IbsParams P{};
  const bool premasked = c->ibs_mode == 2;
  P.plane[0] = premasked ? c->d_ibs_lo.p : c->d_sm_lo.p;
  P.plane[1] = premasked ? c->d_ibs_hi.p : c->d_sm_hi.p;
  P.plane[2] = c->ibs_mode == 1 ? c->d_sm_valid.p : nullptr;
  P.n_words = c->n_words; P.words_used = words_used; P.tiles = c->d_ibs_tiles.p; P.n_tiles = n;
  P.words_per_chunk = pl.words_per_chunk; P.n_chunks = pl.n_chunks; P.acc = c->d_ibs_acc.p;
  if (pl.n_chunks > 1) KGL_CUDA(c, cudaMemsetAsync(c->d_ibs_acc.p, 0, (size_t)n * 3 * kIbsTileCells * 4, c->stream));
  cudaEvent_t e0, e1;
  KGL_CUDA(c, c->ibs_timer.next(e0, e1));
  if (e0) KGL_CUDA(c, cudaEventRecord(e0, c->stream));
  if (tensor) {
    // dense part on the tensor cores: three Gram matrices over the blocks the tile list touches, then the tile cells (ibs_gram.cuh)
    int32_t* outs[3] = {c->d_gram.p, c->d_gram_hh.p, c->d_gram_aa.p};
    const uint32_t tables[3] = {kGramTableDosage, kGramTableHet, kGramTableHomAlt};
    for (int m = 0; m < 3; ++m) {
      int rc = run_gram_blocks(c, c->d_codes16.p, tables[m], tables[m], outs[m]); if (rc) return rc;
    }
    k_ibs_from_grams<<<blocks_for((uint64_t)n * kIbsTileCells, 256), 256, 0, c->stream>>>(c->d_gram.p, c->d_gram_hh.p, c->d_gram_aa.p,
                                                                                         c->d_ibs_class.p, c->d_ibs_tiles.p, c->d_ibs_tile_block.p, n, c->d_ibs_acc.p);
    KGL_LAUNCH_CHECK(c);
    ++c->launches;
  } else {
    KGL_CUDA(c, launch_ibs(P, pl, c->ibs_mode == 1, c->stream));
    ++c->launches;
  }
  c->ibs_used_tensor = tensor;
  if (e1) KGL_CUDA(c, cudaEventRecord(e1, c->stream));
  if (c->ibs_mode == 2) {
    // every genome's dropped rows are cut into segments so that the repair fills the GPU also when few tiles are dealt to it
    // (multi-GPU): about eight 128-thread CTAs per SM, and no segment shorter than ~256 rows on average
    const uint64_t avg_rows = c->n_dropped / std::max<uint64_t>(1, c->N);
    uint32_t segs = (uint32_t)std::max<uint64_t>(1, ((uint64_t)c->sm_count * 8 + n - 1) / n);
    segs = (uint32_t)std::min<uint64_t>(segs, std::max<uint64_t>(1, avg_rows / 256));
    segs = std::min<uint32_t>(segs, 64);
    if (segs > 1 && pl.n_chunks == 1)      // plane 2 (J) is accumulated atomically then: clear it (the whole buffer is cleared when chunked)
      KGL_CUDA(c, cudaMemset2DAsync(c->d_ibs_acc.p + 2 * kIbsTileCells, (size_t)3 * kIbsTileCells * 4, 0, (size_t)kIbsTileCells * 4, n, c->stream));
    k_ibs_missing_fix<<<dim3(n, segs), 128, 0, c->stream>>>(reinterpret_cast<const uint4*>(c->d_packed.p), (uint32_t)c->units, c->d_dropped.p,
                                                             c->d_dropped_seg.p, c->N, c->d_ibs_tiles.p, c->d_ibs_acc.p);
    KGL_LAUNCH_CHECK(c);
  }
  return KGL_B200_OK;
}

int ibs_finalize(kgl_b200_ctx* c, uint32_t n_tiles, int mode, uint64_t row_begin, uint64_t row_end, int mirror, uint32_t* d_out) {
  k_ibs_finalize<<<blocks_for((uint64_t)n_tiles * kIbsTileCells, 256), 256, 0, c->stream>>>(
      c->d_ibs_acc.p, c->d_ibs_tiles.p, n_tiles, c->ibs_mode, c->ibs_mode == 2 ? c->d_dropped_seg.p : nullptr, (uint32_t)c->L, mode, c->N,
      row_begin, row_end, mirror, d_out);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

// The tiles of `list` for kgl_b200_ibs_tiles_buffer (kgl_b200_enqueue_ibs_tiles, kgl_b200_enqueue_ibs_tile_list).
int ibs_enqueue_tiles(kgl_b200_ctx* c, const TileList& list) {
  int rc = ibs_compute_tiles(c, list); if (rc) return rc;
  const uint64_t count = list.key.n;
  KGL_CUDA(c, c->d_ibs_tiles_out.ensure((size_t)count * kIbsTileCells * 4));
  rc = ibs_finalize(c, (uint32_t)count, 0, 0, 0, 0, c->d_ibs_tiles_out.p); if (rc) return rc;
  c->ibs_last_count = count;
  return KGL_B200_OK;
}

// count tiles to the host in calls of at most kIbsMaxTilesPerLaunch: enqueue(done, n) computes tiles [done, done + n) of them.
template <class Enqueue>
int ibs_run_tiles(kgl_b200_ctx* c, uint64_t count, uint32_t* out, Enqueue enqueue) {
  for (uint64_t done = 0; done < count; done += kIbsMaxTilesPerLaunch) {
    const uint64_t n = std::min<uint64_t>(kIbsMaxTilesPerLaunch, count - done);
    int rc = enqueue(done, n); if (rc) return rc;
    KGL_CUDA(c, cudaMemcpyAsync(out + (size_t)done * kIbsTileCells * 4, c->d_ibs_tiles_out.p, (size_t)n * kIbsTileCells * 16, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return KGL_B200_OK;
}

// Dense pairwise output of genomes [row_begin, row_end) against all genomes, per_pair values of T a pair, through the device
// buffer `buf` to `out`. The whole matrix when it takes at most 2 GiB: the upper-triangle tiles, every tile also written
// transposed. Otherwise slabs of whole tile rows that keep the device result under ~1 GiB. slab(tiles, r0, r1, mirror) writes
// rows [r0, r1) of buf from one tile list of at most kIbsMaxTilesPerLaunch tiles.
template <class T, class Slab>
int run_pairwise(kgl_b200_ctx* c, uint64_t row_begin, uint64_t row_end, uint64_t per_pair, DevBuf<T>& buf, T* out, Slab slab) {
  const uint64_t N = c->N, side = ibs_side(c), bytes = per_pair * sizeof(T);
  if (row_begin == 0 && row_end == N && N * N * bytes <= (2ull << 30)) {
    KGL_CUDA(c, buf.ensure((size_t)N * N * per_pair));
    for (uint64_t t0 = 0, n_upper = side * (side + 1) / 2; t0 < n_upper; t0 += kIbsMaxTilesPerLaunch) {
      int rc = slab(upper_tiles(t0, 1, std::min(n_upper - t0, kIbsMaxTilesPerLaunch)), 0, N, 1); if (rc) return rc;
    }
    KGL_CUDA(c, cudaMemcpyAsync(out, buf.p, (size_t)N * N * bytes, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    return KGL_B200_OK;
  }
  const uint64_t slab_tile_rows = std::max<uint64_t>(1, std::min<uint64_t>((1ull << 30) / (N * bytes * kIbsT), kIbsMaxTilesPerLaunch / side));
  for (uint64_t tr0 = row_begin / kIbsT; tr0 * kIbsT < row_end; tr0 += slab_tile_rows) {
    const uint64_t tr1 = std::min((row_end + kIbsT - 1) / kIbsT, tr0 + slab_tile_rows);
    const uint64_t r0 = std::max(row_begin, tr0 * kIbsT), r1 = std::min(row_end, tr1 * kIbsT);
    KGL_CUDA(c, buf.ensure((size_t)(r1 - r0) * N * per_pair));
    int rc = slab(band_tiles(tr0, tr1, side), r0, r1, 0); if (rc) return rc;
    KGL_CUDA(c, cudaMemcpyAsync(out + (size_t)(r0 - row_begin) * N * per_pair, buf.p, (size_t)(r1 - r0) * N * bytes, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  return KGL_B200_OK;
}

// ---- KING-robust kinship (king.cuh) -------------------------------------------------------------------------------------
// One slab of tiles (<= kIbsMaxTilesPerLaunch): the IBS counts by ibs_compute_tiles in whichever form it picks, HH (already
// filled by the tensor form, otherwise one Gram run) and, with code-3 cells, M = H C^T over the same blocks. Fills K.
int king_compute_tiles(kgl_b200_ctx* c, const TileList& list, KingTiles& K) {
  int rc = ibs_compute_tiles(c, list, true); if (rc) return rc;
  rc = ensure_ibs_class(c); if (rc) return rc;
  rc = ensure_codes(c); if (rc) return rc;
  const size_t block_cells = (size_t)c->ibs_n_blocks * kGramM * kGramN;
  if (!c->ibs_used_tensor) {                       // the popcount kernel ran: HH is not there yet
    KGL_CUDA(c, c->d_gram_hh.ensure(block_cells));
    rc = run_gram_blocks(c, c->d_codes16.p, kGramTableHet, kGramTableHet, c->d_gram_hh.p); if (rc) return rc;
  }
  if (c->n_dropped > 0) {
    KGL_CUDA(c, c->d_king_m.ensure(block_cells));
    rc = run_gram_blocks(c, c->d_codes16.p, kGramTableHet, kGramTableCode3, c->d_king_m.p); if (rc) return rc;
  }
  K = KingTiles{};
  K.acc = c->d_ibs_acc.p; K.tiles = c->d_ibs_tiles.p; K.n_tiles = (uint32_t)list.key.n;
  K.valid_mode = c->ibs_mode; K.seg = c->ibs_mode == 2 ? c->d_dropped_seg.p : nullptr; K.n_loci = (uint32_t)c->L; K.n_genomes = c->N;
  K.hh = c->d_gram_hh.p; K.m = c->n_dropped > 0 ? c->d_king_m.p : nullptr; K.tile_block = c->d_ibs_tile_block.p; K.counts = c->d_ibs_class.p;
  return KGL_B200_OK;
}

int king_check(kgl_b200_ctx* c) {
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  if (c->L >= (1ull << 29)) return fail(c, KGL_B200_ERR_INVALID, "KING: more than 2^29 loci would overflow the int32 Gram accumulators");
  return ensure_ibs_planes(c);
}

// Tiles first, first + stride, ... of the upper-triangle tile list (rank r of R: first = r, stride = R); the rest of the
// matrix is left zero so that a SUM all-reduce of the int32 matrix over the ranks assembles it.
// Not run_gram_blocks: the tiles are those of the whole ld x ld matrix, the matrix is also cleared when only some of its tiles
// run (stride > 1), and kgl_b200_last_gram_kernel_ms times the launch alone, without that clear.
int gram_compute(kgl_b200_ctx* c, uint64_t first = 0, uint64_t stride = 1) {
  int rc = ensure_codes(c); if (rc) return rc;
  c->gram_valid = false;
  const uint64_t ld = gram_ld(c);
  if (c->gram_tiles_ld != ld || c->gram_first != first || c->gram_stride != stride) {
    const std::vector<uint2> all = gram_upper_tiles(ld);
    std::vector<uint2> tiles;
    for (uint64_t t = first; t < all.size(); t += stride) tiles.push_back(all[t]);
    if (tiles.empty()) tiles.push_back(all[0]);              // more ranks than tiles: nothing is launched (gram_n_tiles = 0)
    c->gram_first = first; c->gram_stride = stride;
    KGL_CUDA(c, c->d_gram_tiles.ensure(tiles.size()));
    KGL_CUDA(c, cudaMemcpyAsync(c->d_gram_tiles.p, tiles.data(), tiles.size() * sizeof(uint2), cudaMemcpyHostToDevice, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    c->gram_tiles_ld = ld; c->gram_n_tiles = first < all.size() ? tiles.size() : 0;
  }
  KGL_CUDA(c, c->d_gram.ensure((size_t)ld * ld));
  const uint32_t k_stages = gram_k_stages(c);
  const GramPlan pl = plan_gram((uint32_t)std::max<uint64_t>(c->gram_n_tiles, 1), k_stages, c->sm_count);
  GramParams P{};
  P.codes = c->d_codes16.p; P.k_stages = k_stages; P.tiles = c->d_gram_tiles.p; P.n_tiles = (uint32_t)c->gram_n_tiles;
  P.stages_per_chunk = pl.stages_per_chunk; P.n_chunks = pl.n_chunks; P.out = c->d_gram.p; P.ld = ld;
  P.table_a = P.table_b = kGramTableDosage;
  if (pl.n_chunks > 1 || stride > 1) KGL_CUDA(c, cudaMemsetAsync(c->d_gram.p, 0, (size_t)ld * ld * 4, c->stream));
  if (!c->gram_e0) { KGL_CUDA(c, cudaEventCreate(&c->gram_e0)); KGL_CUDA(c, cudaEventCreate(&c->gram_e1)); }
  KGL_CUDA(c, cudaEventRecord(c->gram_e0, c->stream));
  if (c->gram_n_tiles > 0) { KGL_CUDA(c, launch_gram(P, pl, c->stream)); ++c->launches; }
  KGL_CUDA(c, cudaEventRecord(c->gram_e1, c->stream));
  c->gram_valid = true;
  return KGL_B200_OK;
}

// Raw counting needs no super-populations: without them everyone counts as population 0.
int default_superpop(kgl_b200_ctx* c) {
  if (c->have_superpop) return KGL_B200_OK;
  std::vector<uint8_t> zeros(c->N, 0);
  int rc = kgl_b200_set_genome_superpop(c, c->N, zeros.data()); if (rc) return rc;
  c->have_superpop = false;
  return KGL_B200_OK;
}

// ---- genotype PCA (pca.cuh) ---------------------------------------------------------------------------------------------
constexpr uint64_t kPcaSlabBytes = 1ull << 30;     // int32 outputs of one slab of pass-1 loci (both runs)
// d_pca_stats: max bits and sums of the X block, of the W | V block, and |U|
constexpr size_t kPcaStatX = 0, kPcaStatXSum = kPcaMaxCols, kPcaStatWV = 2 * kPcaMaxCols, kPcaStatWVSum = 4 * kPcaMaxCols,
                 kPcaStatUsed = 6 * kPcaMaxCols, kPcaStats = 6 * kPcaMaxCols + 1;

// Loci-major codes of the pass-1 runs (K = genomes), once per upload.
int ensure_codes_loci(kgl_b200_ctx* c) {
  if (c->codes_loci_valid) return KGL_B200_OK;
  const uint64_t ks = (c->N + kGramK - 1) / kGramK, words = c->padded_rows * ks * 8;
  KGL_CUDA(c, c->d_codes_loci.ensure(words));
  k_codes16_loci<<<blocks_for(words, 256), 256, 0, c->stream>>>(reinterpret_cast<const uint32_t*>(c->d_packed.p), c->units, c->padded_rows, ks,
                                                                c->d_codes_loci.p);
  KGL_LAUNCH_CHECK(c);
  c->codes_loci_valid = true;
  return KGL_B200_OK;
}

// p_l, d_l and the used loci for the keep mask (NULL = every locus) from one raw counting pass; m = |U|.
int pca_prepare(kgl_b200_ctx* c, const uint8_t* keep, uint64_t& m) {
  if (c->L >= (1ull << 28)) return fail(c, KGL_B200_ERR_INVALID, "PCA: n_loci must be < 2^28 (int32 digit accumulators)");
  int rc = default_superpop(c); if (rc) return rc;
  rc = launch_count(c, true, true, false, false, false, nullptr, false, &c->d_pca_counts); if (rc) return rc;
  if (keep) {
    KGL_CUDA(c, c->d_pca_keep.ensure(c->L));
    KGL_CUDA(c, cudaMemcpyAsync(c->d_pca_keep.p, keep, c->L, cudaMemcpyHostToDevice, c->stream));
  }
  KGL_CUDA(c, c->d_pca_p.ensure(c->L));
  KGL_CUDA(c, c->d_pca_d.ensure(c->L));
  KGL_CUDA(c, c->d_pca_used.ensure(c->L));
  KGL_CUDA(c, c->d_pca_stats.ensure(kPcaStats));
  KGL_CUDA(c, cudaMemsetAsync(c->d_pca_stats.p + kPcaStatUsed, 0, 8, c->stream));
  k_pca_loci<<<blocks_for(c->L, 256), 256, 0, c->stream>>>(c->d_pca_counts.p, keep ? c->d_pca_keep.p : nullptr, c->L, c->d_pca_p.p, c->d_pca_d.p,
                                                           c->d_pca_used.p, c->d_pca_stats.p + kPcaStatUsed);
  KGL_LAUNCH_CHECK(c);
  unsigned long long used = 0;
  KGL_CUDA(c, cudaMemcpyAsync(&used, c->d_pca_stats.p + kPcaStatUsed, 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  m = used;
  return KGL_B200_OK;
}

// Column maxima and digits of F [k_count][cols] into d_pca_digits (B operand of k_stages), sums next to the maxima.
int pca_digits(kgl_b200_ctx* c, const double* F, uint64_t k_count, uint32_t cols, const uint8_t* used, uint64_t k_stages,
               unsigned long long* max_bits, unsigned long long* sums) {
  KGL_CUDA(c, cudaMemsetAsync(max_bits, 0, cols * 8, c->stream));
  KGL_CUDA(c, cudaMemsetAsync(sums, 0, cols * 8, c->stream));
  k_pca_colmax<<<dim3((unsigned)std::min<uint64_t>(blocks_for(k_count, 256), 64), cols), 256, 0, c->stream>>>(F, k_count, cols, max_bits);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, c->d_pca_digits.ensure((size_t)cols / kPcaColsPerBlock * kGramN * k_stages * 8));
  const uint64_t threads = (uint64_t)cols * k_stages * 8;
  k_pca_digits<<<(unsigned)std::min<uint64_t>(blocks_for(threads, 256), (uint64_t)c->sm_count * 16), 256, 0, c->stream>>>(
      F, k_count, cols, max_bits, used, k_stages, c->d_pca_digits.p, sums);
  KGL_LAUNCH_CHECK(c);
  return KGL_B200_OK;
}

// One digit Gram run: A rows of `codes` (tiles' rows) against the digit blocks, into out with row pitch ld.
int pca_gram(kgl_b200_ctx* c, const uint32_t* codes, uint32_t table_a, uint64_t k_stages, const uint2* tiles, uint32_t n_tiles, const GramPlan& pl,
             int32_t* out, uint64_t ld) {
  GramParams G{};
  G.codes = codes; G.codes_b = c->d_pca_digits.p; G.k_stages = (uint32_t)k_stages; G.tiles = tiles; G.n_tiles = n_tiles;
  G.stages_per_chunk = pl.stages_per_chunk; G.n_chunks = pl.n_chunks; G.out = out; G.ld = ld;
  G.table_a = table_a; G.table_b = kPcaTableDigit;
  KGL_CUDA(c, launch_gram(G, pl, c->stream));
  ++c->launches;
  return KGL_B200_OK;
}

// y = Z^T Z x for x [N][n_in] (host, n_in <= 48) after pca_prepare. With loci_out: only pass 1, Y = Z x [L][n_in] to loci_out.
int pca_apply(kgl_b200_ctx* c, uint32_t n_in, const double* x, double* y, double* loci_out) {
  const uint32_t nb = (n_in + kPcaColsPerBlock - 1) / kPcaColsPerBlock, cols = nb * kPcaColsPerBlock;
  const uint64_t N = c->N, L = c->L, ld1 = (uint64_t)cols / kPcaColsPerBlock * kGramN, ld2 = 2 * ld1, ldg = gram_ld(c);
  const uint64_t ks1 = (N + kGramK - 1) / kGramK, ks2 = gram_k_stages(c);
  const bool code3 = c->n_dropped > 0;
  const int runs = code3 ? 2 : 1;
  int rc = ensure_codes_loci(c); if (rc) return rc;
  if (!loci_out) { rc = ensure_codes(c); if (rc) return rc; }
  // tile lists: a pass-1 slab (loci tiles x digit blocks), then pass 2 against the W blocks and against the V blocks
  const uint64_t slab = std::min<uint64_t>(c->padded_rows, std::max<uint64_t>(kGramM, kPcaSlabBytes / (runs * ld1 * 4) / kGramM * kGramM));
  std::vector<uint2> tiles;
  for (uint32_t ti = 0; ti < slab / kGramM; ++ti)
    for (uint32_t tj = 0; tj < nb; ++tj) tiles.push_back(make_uint2(ti, tj));
  const size_t n1 = tiles.size();
  for (uint32_t part = 0; part < 2; ++part)
    for (uint32_t ti = 0; ti < ldg / kGramM; ++ti)
      for (uint32_t tj = 0; tj < nb; ++tj) tiles.push_back(make_uint2(ti, part * nb + tj));
  const uint32_t n2 = (uint32_t)(ldg / kGramM * nb);
  std::vector<double> xp((size_t)N * cols, 0.0);
  for (uint64_t g = 0; g < N; ++g) std::copy(x + g * n_in, x + (g + 1) * n_in, xp.begin() + g * cols);
  KGL_CUDA(c, c->d_pca_tiles.ensure(tiles.size()));
  KGL_CUDA(c, c->d_pca_x.ensure(xp.size()));
  if (loci_out) KGL_CUDA(c, c->d_pca_y.ensure((size_t)L * cols));
  else KGL_CUDA(c, c->d_pca_wv.ensure((size_t)L * 2 * cols));
  KGL_CUDA(c, c->d_pca_acc.ensure(std::max<uint64_t>(runs * slab * ld1, ldg * ld2)));
  KGL_CUDA(c, c->d_pca_out.ensure((size_t)N * cols));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_pca_tiles.p, tiles.data(), tiles.size() * sizeof(uint2), cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_pca_x.p, xp.data(), xp.size() * 8, cudaMemcpyHostToDevice, c->stream));
  unsigned long long* st = c->d_pca_stats.p;
  int32_t* acc = c->d_pca_acc.p;

  // pass 1: Y = Z X over slabs of loci; K = genomes
  rc = pca_digits(c, c->d_pca_x.p, N, cols, nullptr, ks1, st + kPcaStatX, st + kPcaStatXSum); if (rc) return rc;
  for (uint64_t r0 = 0; r0 < L; r0 += slab) {
    const uint64_t rows = std::min<uint64_t>(slab, c->padded_rows - r0);
    const uint32_t n_tiles = (uint32_t)(rows / kGramM * nb);
    const GramPlan pl = plan_gram(n_tiles, (uint32_t)ks1, c->sm_count);
    if (pl.n_chunks > 1) KGL_CUDA(c, cudaMemsetAsync(acc, 0, (size_t)runs * slab * ld1 * 4, c->stream));
    for (int run = 0; run < runs; ++run) {
      rc = pca_gram(c, c->d_codes_loci.p + r0 / 128 * ks1 * 1024, run ? kGramTableCode3 : kGramTableDosage, ks1, c->d_pca_tiles.p, n_tiles, pl,
                    acc + (size_t)run * slab * ld1, ld1);
      if (rc) return rc;
    }
    const uint64_t n = std::min<uint64_t>(rows, L - r0);
    k_pca_recombine_loci<<<blocks_for(n * cols, 256), 256, 0, c->stream>>>(acc, code3 ? acc + slab * ld1 : nullptr, ld1, r0, n, cols, c->d_pca_p.p,
                                                                           c->d_pca_d.p, c->d_pca_used.p, st + kPcaStatX, st + kPcaStatXSum,
                                                                           loci_out ? c->d_pca_y.p : nullptr, c->d_pca_wv.p);
    KGL_LAUNCH_CHECK(c);
  }
  if (loci_out) {
    KGL_CUDA(c, cudaMemcpy2DAsync(loci_out, n_in * 8, c->d_pca_y.p, cols * 8, n_in * 8, L, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    return KGL_B200_OK;
  }

  // pass 2: X' = Z^T Y from the digits of W | V; K = loci, the used ones count
  rc = pca_digits(c, c->d_pca_wv.p, L, 2 * cols, c->d_pca_used.p, ks2, st + kPcaStatWV, st + kPcaStatWVSum); if (rc) return rc;
  const GramPlan pl = plan_gram(n2, (uint32_t)ks2, c->sm_count);
  if (pl.n_chunks > 1) KGL_CUDA(c, cudaMemsetAsync(acc, 0, (size_t)ldg * ld2 * 4, c->stream));
  rc = pca_gram(c, c->d_codes16.p, kGramTableDosage, ks2, c->d_pca_tiles.p + n1, n2, pl, acc, ld2); if (rc) return rc;
  if (code3) { rc = pca_gram(c, c->d_codes16.p, kGramTableCode3, ks2, c->d_pca_tiles.p + n1 + n2, n2, pl, acc, ld2); if (rc) return rc; }
  k_pca_recombine_genomes<<<blocks_for(N * cols, 256), 256, 0, c->stream>>>(acc, ld2, N, cols, code3 ? 1 : 0, st + kPcaStatWV, st + kPcaStatWVSum,
                                                                            c->d_pca_out.p);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaMemcpy2DAsync(y, n_in * 8, c->d_pca_out.p, cols * 8, n_in * 8, N, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

}  // namespace

// The device buffers free themselves (DevBuf) after this body, the peer regions that map d_xchg must be gone by then.
kgl_b200_ctx::~kgl_b200_ctx() {
  cudaSetDevice(device);
  for (cudaStream_t s : {stream, tail_stream, prep_stream}) if (s) cudaStreamSynchronize(s);
  peer_detach(this); peer_unregister(this);
  for (cudaEvent_t e : {ev0, ev1, gram_e0, gram_e1, prep_done, inputs_ready}) if (e) cudaEventDestroy(e);
  for (int i = 0; i < 2; ++i)
    for (cudaEvent_t e : {readers_main[i], readers_tail[i], stream_done[i], tail_done[i]}) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : chunk_ev) cudaEventDestroy(e);
  for (cudaStream_t s : {prep_stream, tail_stream, copy_stream, own_stream}) if (s) cudaStreamDestroy(s);
}

// ---------------------------------------------------------------------------------------------------------------------
extern "C" {

const char* kgl_b200_version(void) { return "kgl_b200 0.1 (sm_100a)"; }

int kgl_b200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int kgl_b200_create(int device, kgl_b200_ctx** out) {
  if (!out) return fail(nullptr, KGL_B200_ERR_INVALID, "ctx out pointer is null");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return fail(nullptr, KGL_B200_ERR_NO_DEVICE, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                                 " (kgl_b200 has no CPU fallback)");
  }
  if (device < 0 || device >= n) return fail(nullptr, KGL_B200_ERR_INVALID, "device index out of range");
  cudaDeviceProp prop{};
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, KGL_B200_ERR_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10) {
    char buf[160];
    std::snprintf(buf, sizeof buf, "device %d (%s, sm_%d%d) is not a Blackwell sm_100 GPU; this library ships sm_100a code only",
                  device, prop.name, prop.major, prop.minor);
    return fail(nullptr, KGL_B200_ERR_NO_DEVICE, buf);
  }
  auto* c = new kgl_b200_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->total_memory = prop.totalGlobalMem;
  // the context stream carries the streaming kernel: highest priority, so that its CTAs are placed before the blocks of the
  // side streams (preparation, tail) when both are ready
  int pr_least = 0, pr_greatest = 0;
  cudaDeviceGetStreamPriorityRange(&pr_least, &pr_greatest);
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithPriority(&c->own_stream, cudaStreamNonBlocking, pr_greatest) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
    std::string m = std::string("context setup failed: ") + cudaGetErrorString(cudaGetLastError());
    delete c;
    return fail(nullptr, KGL_B200_ERR_CUDA, m);
  }
  c->stream = c->own_stream;
  *out = c;
  return KGL_B200_OK;
}

void kgl_b200_destroy(kgl_b200_ctx* c) { delete c; }

const char* kgl_b200_last_error(const kgl_b200_ctx* c) { return c ? c->err.c_str() : tl_create_error.c_str(); }

int kgl_b200_set_stream(kgl_b200_ctx* c, void* s) {
  if (!c) return KGL_B200_ERR_INVALID;
  c->stream = s ? static_cast<cudaStream_t>(s) : c->own_stream;
  return KGL_B200_OK;
}

int kgl_b200_synchronize(kgl_b200_ctx* c) {
  if (!c) return KGL_B200_ERR_INVALID;
  int rc = use_device(c); if (rc) return rc;
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

uint64_t kgl_b200_launch_count(const kgl_b200_ctx* c) { return c ? c->launches : 0; }

// Milliseconds from e0 to e1 once e1 has completed; -1 on a CUDA error.
static float event_ms(const kgl_b200_ctx* c, cudaEvent_t e0, cudaEvent_t e1) {
  if (cudaSetDevice(c->device) != cudaSuccess || cudaEventSynchronize(e1) != cudaSuccess) return -1.0f;
  float ms = -1.0f;
  if (cudaEventElapsedTime(&ms, e0, e1) != cudaSuccess) return -1.0f;
  return ms;
}

float kgl_b200_last_stream_kernel_ms(kgl_b200_ctx* c) { return c && c->ev_valid ? event_ms(c, c->last_e0, c->last_e1) : -1.0f; }

int kgl_b200_kernel_timer_reset(kgl_b200_ctx* c) {
  if (!c) return KGL_B200_ERR_INVALID;
  c->timer.used = 0;
  return KGL_B200_OK;
}

int kgl_b200_kernel_timer_read(kgl_b200_ctx* c, float* ms, uint32_t capacity, uint32_t* n) {
  if (!c || !ms || !n) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  KGL_CUDA(c, c->timer.read(ms, capacity, n));
  return KGL_B200_OK;
}

static int set_shape(kgl_b200_ctx* c, uint64_t n_genomes, uint64_t n_loci, uint64_t row_bytes) {
  if (n_genomes == 0 || n_loci == 0) return fail(c, KGL_B200_ERR_INVALID, "empty genotype matrix");
  if (row_bytes != 16 * ((n_genomes + 63) / 64)) return fail(c, KGL_B200_ERR_INVALID, "row_bytes must be 16*ceil(n_genomes/64)");
  if (n_genomes >= (1ull << 32) || n_loci >= (1ull << 32)) return fail(c, KGL_B200_ERR_INVALID, "dimension too large");
  // A matrix of a different shape starts a new population: stale loci / super-populations must be uploaded again
  // (require_population reports what is missing at run time).
  if (c->have_loci && c->loci_len != n_loci) { c->have_loci = false; c->prep_valid = false; }
  if (c->have_superpop && c->h_superpop.size() != n_genomes) c->have_superpop = false;
  c->N = n_genomes; c->L = n_loci; c->row_bytes = row_bytes; c->host_units = row_bytes / 16;
  c->n_multi = 0;                    // the side cells belong to the matrix: kgl_b200_upload_multi_allelic comes after it
  c->units = stream_units_padded(c->host_units); c->Npad = c->units * 64;
  c->sm_valid = false; c->codes_valid = false; c->units_valid = false; c->dropped_valid = false; c->dropped_cells_state = 0; c->prep_valid = false; c->ibs_mode = -1; c->ibs_tiles_key = TileKey{}; c->ibs_n_blocks = 0; c->ibs_class_valid = false;
  c->codes16_valid = false; c->gram_valid = false; c->codes_loci_valid = false;
  return KGL_B200_OK;
}

int kgl_b200_upload_genotypes(kgl_b200_ctx* c, uint64_t n_genomes, uint64_t n_loci, uint64_t row_bytes, const void* packed) {
  if (!c || !packed) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = set_shape(c, n_genomes, n_loci, row_bytes); if (rc) return rc;
  rc = alloc_matrix(c); if (rc) return rc;
  c->have_geno = true;
  if (c->units != c->host_units) {        // padded device pitch (wide populations): one strided copy, then the index
    KGL_CUDA(c, cudaMemcpy2DAsync(c->d_packed.p, c->units * 16, packed, row_bytes, row_bytes, n_loci, cudaMemcpyHostToDevice, c->stream));
    return build_dropped_index(c);        // synchronises the stream
  }
  // The matrix crosses PCIe in row chunks on a copy stream; the code-3 cells of a chunk are listed (k_dropped_index) as soon
  // as it has landed, i.e. while the next chunk is still copying. The key buffer is sized for 0.25 % code-3 cells; a
  // population with more is indexed again with the exact size (the cursor has counted them all).
  if (!c->copy_stream) KGL_CUDA(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  constexpr int kChunks = 16;
  while ((int)c->chunk_ev.size() < kChunks) {
    cudaEvent_t ev = nullptr;
    KGL_CUDA(c, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    c->chunk_ev.push_back(ev);
  }
  const uint64_t limit = dropped_index_limit(c);
  const uint64_t cap = std::min<uint64_t>(limit, std::max<uint64_t>(1u << 16, c->N * c->L / 400));
  KGL_CUDA(c, c->d_dropped_unsorted.ensure(cap));
  KGL_CUDA(c, c->d_dropped_counter.ensure(2));
  KGL_CUDA(c, cudaMemsetAsync(c->d_dropped_counter.p, 0, 16, c->stream));
  // the copy stream must not overtake work already queued on the context stream (the memsets of alloc_matrix)
  KGL_CUDA(c, cudaEventRecord(c->chunk_ev[0], c->stream));
  KGL_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->chunk_ev[0], 0));
  const uint64_t rows_per_chunk = ((n_loci + kChunks - 1) / kChunks + 255) / 256 * 256;
  int ci = 0;
  for (uint64_t r0 = 0; r0 < n_loci; r0 += rows_per_chunk, ++ci) {
    const uint64_t rows = std::min<uint64_t>(rows_per_chunk, n_loci - r0);
    KGL_CUDA(c, cudaMemcpyAsync(c->d_packed.p + r0 * row_bytes, static_cast<const uint8_t*>(packed) + r0 * row_bytes, rows * row_bytes,
                                cudaMemcpyHostToDevice, c->copy_stream));
    KGL_CUDA(c, cudaEventRecord(c->chunk_ev[ci], c->copy_stream));
    KGL_CUDA(c, cudaStreamWaitEvent(c->stream, c->chunk_ev[ci], 0));
    rc = launch_dropped_index(c, r0 * c->units, rows * c->units, cap); if (rc) return rc;
  }
  unsigned long long total = 0;
  KGL_CUDA(c, cudaMemcpyAsync(&total, c->d_dropped_counter.p + 1, 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));      // every chunk has landed: the host buffer is free again
  if (total > cap && total <= limit) {
    KGL_CUDA(c, c->d_dropped_unsorted.ensure(total));
    KGL_CUDA(c, cudaMemsetAsync(c->d_dropped_counter.p, 0, 16, c->stream));
    rc = launch_dropped_index(c, 0, c->L * c->units, total); if (rc) return rc;
  }
  return finish_dropped_index(c, total);
}

int kgl_b200_upload_loci(kgl_b200_ctx* c, uint64_t n_loci, uint32_t n_pop, const float* af, const uint32_t* offsets) {
  if (!c || !af) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (n_pop == 0 || n_pop > KGL_B200_MAX_POP) return fail(c, KGL_B200_ERR_INVALID, "n_pop must be 1..6");
  if (n_loci == 0) return fail(c, KGL_B200_ERR_INVALID, "n_loci is 0");
  if (c->have_geno && c->L != n_loci) c->have_geno = false;   // new population: the old matrix no longer applies
  int rc = use_device(c); if (rc) return rc;
  c->have_offsets = offsets != nullptr; c->loci_len = n_loci;
  c->n_pop = n_pop;
  if (!c->have_geno) c->L = n_loci;
  KGL_CUDA(c, c->d_af.ensure((size_t)n_pop * n_loci));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_af.p, af, (size_t)n_pop * n_loci * 4, cudaMemcpyHostToDevice, c->stream));
  if (offsets) {
    KGL_CUDA(c, c->d_offsets.ensure(n_loci));
    KGL_CUDA(c, cudaMemcpyAsync(c->d_offsets.p, offsets, n_loci * 4, cudaMemcpyHostToDevice, c->stream));
    c->h_offsets.assign(offsets, offsets + n_loci);
  }
  c->sel_row_lo = 0; c->sel_row_hi = ~0ull;
  KGL_CUDA(c, c->d_sel.ensure(n_loci));
  KGL_CUDA(c, cudaMemsetAsync(c->d_sel.p, 0, n_loci, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  c->have_loci = true; c->prep_valid = false; c->dropped_cells_state = 0;
  c->n_multi = 0;                    // ... and after the frequency table
  c->keep_valid = false;
  return KGL_B200_OK;
}

int kgl_b200_set_genome_superpop(kgl_b200_ctx* c, uint64_t n_genomes, const uint8_t* superpop) {
  if (!c || !superpop) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (c->have_geno && c->N != n_genomes) c->have_geno = false;   // new population
  for (uint64_t g = 0; g < n_genomes; ++g)
    if (superpop[g] >= KGL_B200_MAX_POP) return fail(c, KGL_B200_ERR_INVALID, "super-population index must be 0..5");
  int rc = use_device(c); if (rc) return rc;
  c->h_superpop.assign(superpop, superpop + n_genomes);
  KGL_CUDA(c, c->d_superpop.ensure(n_genomes));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_superpop.p, superpop, n_genomes, cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  c->have_superpop = true; c->units_valid = false; c->dropped_cells_state = 0; c->prep_valid = false;
  if (!c->have_geno) c->N = n_genomes;
  return KGL_B200_OK;
}

int kgl_b200_upload_multi_allelic(kgl_b200_ctx* c, uint64_t n_multi, const uint32_t* rows, const float* af, const uint8_t* cells) {
  if (!c) return KGL_B200_ERR_INVALID;
  int rc = use_device(c); if (rc) return rc;
  if (!c->have_geno || !c->have_loci || c->loci_len != c->L)
    return fail(c, KGL_B200_ERR_STATE, "upload the genotype matrix and the allele frequencies before the multi-allelic loci");
  c->n_multi = 0; c->prep_valid = false;
  if (n_multi == 0) return KGL_B200_OK;
  if (!rows || !af || !cells) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  for (uint64_t m = 0; m < n_multi; ++m)
    if (rows[m] >= c->L || (m > 0 && rows[m] <= rows[m - 1])) return fail(c, KGL_B200_ERR_INVALID, "multi-allelic rows must be ascending rows of the locus table");
  KGL_CUDA(c, c->d_multi_rows.ensure(n_multi));
  KGL_CUDA(c, c->d_multi_af.ensure((size_t)c->n_pop * n_multi * kMultiSlots));
  KGL_CUDA(c, c->d_multi_cells.ensure((size_t)n_multi * c->N));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_multi_rows.p, rows, n_multi * 4, cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_multi_af.p, af, (size_t)c->n_pop * n_multi * kMultiSlots * 4, cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_multi_cells.p, cells, (size_t)n_multi * c->N, cudaMemcpyHostToDevice, c->stream));
  k_multi_mask_af<<<blocks_for(n_multi * c->n_pop, 128), 128, 0, c->stream>>>(c->d_multi_rows.p, n_multi, (int)c->n_pop, c->L, c->d_af.p);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  c->n_multi = n_multi; c->dropped_cells_state = 0;
  return KGL_B200_OK;
}

int kgl_b200_run_multi_allele_count(kgl_b200_ctx* c, uint32_t* counts) {
  if (!c || !counts) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  if (c->n_multi == 0) return fail(c, KGL_B200_ERR_STATE, "no multi-allelic loci uploaded");
  KGL_CUDA(c, c->d_multi_counts.ensure(c->n_multi * kMultiSlots * 3));
  k_multi_allele_count<<<(unsigned)c->n_multi, 256, 0, c->stream>>>(c->d_multi_cells.p, c->N, c->d_multi_counts.p);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaMemcpyAsync(counts, c->d_multi_counts.p, c->n_multi * kMultiSlots * 3 * 4, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

int kgl_b200_set_unphased(kgl_b200_ctx* c, int unphased) {
  if (!c) return KGL_B200_ERR_INVALID;
  if (c->unphased != (unphased != 0)) c->mom_valid = false;
  c->unphased = unphased != 0;
  return KGL_B200_OK;
}

int kgl_b200_set_locus_selection(kgl_b200_ctx* c, uint64_t n_loci, const uint8_t* selected) {
  if (!c || !selected) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->have_loci) return fail(c, KGL_B200_ERR_STATE, "upload_loci first");
  if (n_loci != c->L) return fail(c, KGL_B200_ERR_INVALID, "selection length differs from n_loci");
  int rc = use_device(c); if (rc) return rc;
  c->sel_row_lo = 0; c->sel_row_hi = ~0ull;
  KGL_CUDA(c, cudaMemcpyAsync(c->d_sel.p, selected, n_loci, cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  c->prep_valid = false;
  return KGL_B200_OK;
}

int kgl_b200_get_locus_selection(kgl_b200_ctx* c, uint64_t n_loci, uint8_t* selected) {
  if (!c || !selected) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->have_loci || n_loci != c->loci_len) return fail(c, KGL_B200_ERR_INVALID, "selection length differs from n_loci");
  int rc = use_device(c); if (rc) return rc;
  KGL_CUDA(c, cudaMemcpyAsync(selected, c->d_sel.p, n_loci, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

// RetrieveLociiVector::getAllelesFromTo (kga_analysis_inbreed_locus.cpp:21-72) per super-population.
//  * spacing == 0: every locus decides for itself -> one kernel over the device tables (k_select_dense), nothing crosses PCIe
//    but six counters.
//  * spacing  > 0: the same kernel marks the candidates; the rule "at least `spacing` after the previously ACCEPTED locus" is a
//    sequential chain per population, marked for all populations on the device by pointer doubling (k_chain_*, locus_kernels.cuh).
int kgl_b200_select_loci(kgl_b200_ctx* c, uint64_t lower, uint64_t upper, uint64_t spacing, double min_af, double max_af,
                         uint64_t* n_selected) {
  if (!c) return KGL_B200_ERR_INVALID;
  if (!c->have_loci) return fail(c, KGL_B200_ERR_STATE, "upload_loci first");
  if (!c->have_offsets) return fail(c, KGL_B200_ERR_STATE, "select_loci needs the locus offsets (upload_loci with offsets)");
  int rc = use_device(c, false); if (rc) return rc;     // the selection mask is not read by a tail that may still be running
  min_af = std::min(std::max(min_af, 0.0), 1.0);     // LociiVectorArguments clamps (kga_analysis_inbreed_args.h:85-86)
  max_af = std::min(std::max(max_af, 0.0), 1.0);
  const uint64_t L = c->loci_len;
  // rows of the window [lower, upper] (the offsets are sorted): what the spaced chain walks and the estimator sweeps visit
  const uint64_t l_begin = first_row_at(c, lower);
  const uint64_t l_end = std::upper_bound(c->h_offsets.begin(), c->h_offsets.end(), upper,
                                          [](uint64_t v, uint32_t o) { return v < (uint64_t)o; }) - c->h_offsets.begin();
  c->sel_row_lo = l_begin; c->sel_row_hi = std::max(l_begin, l_end);
  KGL_CUDA(c, c->d_sel_counts.ensure(kMaxPop));
  KGL_CUDA(c, cudaMemsetAsync(c->d_sel_counts.p, 0, kMaxPop * 8, c->stream));
  k_select_dense<<<blocks_for(L, 256), 256, 0, c->stream>>>(c->d_af.p, c->d_offsets.p, L, (int)c->n_pop, lower, upper, min_af, max_af,
                                                            c->keep_valid ? c->d_locus_keep.p : nullptr, c->d_sel.p, c->d_sel_counts.p);
  KGL_LAUNCH_CHECK(c);
  if (c->n_multi) {          // the multi-allelic loci, which also take part in the accept chain like any locus
    k_multi_select<<<blocks_for(c->n_multi, 128), 128, 0, c->stream>>>(c->d_multi_rows.p, c->d_multi_af.p, c->d_offsets.p, c->n_multi, (int)c->n_pop,
                                                                       lower, upper, min_af, max_af, c->keep_valid ? c->d_locus_keep.p : nullptr, c->d_sel.p, c->d_sel_counts.p);
    KGL_LAUNCH_CHECK(c);
  }
  if (spacing > 0) {       // the accept chain over the rows of the window only: a contig is usually swept in many short windows
    const uint64_t span = l_end > l_begin ? l_end - l_begin : 0;
    KGL_CUDA(c, cudaMemsetAsync(c->d_sel_counts.p, 0, kMaxPop * 8, c->stream));
    if (span) {
      const uint64_t n_blocks = (span + kChainBlock - 1) / kChainBlock;
      KGL_CUDA(c, c->d_chain_u32.ensure((size_t)c->n_pop * (3 * span + 2 * n_blocks)));
      KGL_CUDA(c, c->d_chain_mark.ensure((size_t)c->n_pop * span));
      uint32_t* next_valid = c->d_chain_u32.p;
      uint32_t* jump_a = next_valid + (size_t)c->n_pop * span;
      uint32_t* jump_b = jump_a + (size_t)c->n_pop * span;
      uint32_t* block_first = jump_b + (size_t)c->n_pop * span;
      uint32_t* block_after = block_first + (size_t)c->n_pop * n_blocks;
      uint8_t* sel_w = c->d_sel.p + l_begin;                 // all tables below are indexed relative to the window
      const uint32_t* off_w = c->d_offsets.p + l_begin;
      KGL_CUDA(c, cudaMemsetAsync(c->d_chain_mark.p, 0, (size_t)c->n_pop * span, c->stream));
      const dim3 grid_l(blocks_for(span, 256), c->n_pop);
      k_chain_next_valid<<<dim3((unsigned)n_blocks, c->n_pop), kChainBlock, 0, c->stream>>>(sel_w, span, n_blocks, next_valid, block_first);
      KGL_LAUNCH_CHECK(c);
      k_chain_block_suffix<<<c->n_pop, 32, 0, c->stream>>>(block_first, n_blocks, block_after);
      KGL_LAUNCH_CHECK(c);
      k_chain_successor<<<grid_l, 256, 0, c->stream>>>(sel_w, off_w, span, n_blocks, spacing, next_valid, block_after, jump_a, c->d_chain_mark.p);
      KGL_LAUNCH_CHECK(c);
      int rounds = 1;
      while ((1ull << rounds) < span + 1) ++rounds;
      for (int r = 0; r < rounds; ++r) {
        k_chain_round<<<grid_l, 256, 0, c->stream>>>(sel_w, span, jump_a, jump_b, c->d_chain_mark.p);
        KGL_LAUNCH_CHECK(c);
        std::swap(jump_a, jump_b);
      }
      k_chain_finish<<<blocks_for(span, 256), 256, 0, c->stream>>>(c->d_chain_mark.p, span, (int)c->n_pop, sel_w, c->d_sel_counts.p);
      KGL_LAUNCH_CHECK(c);
    }
  }
  c->prep_valid = false; c->inputs_async = true;
  if (n_selected) {
    unsigned long long counts[kMaxPop];
    KGL_CUDA(c, cudaMemcpyAsync(counts, c->d_sel_counts.p, kMaxPop * 8, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    for (uint32_t k = 0; k < c->n_pop; ++k) n_selected[k] = counts[k];
  }
  return KGL_B200_OK;
}

int kgl_b200_set_locus_filter(kgl_b200_ctx* c, uint64_t n_loci, const uint8_t* keep) {
  if (!c) return KGL_B200_ERR_INVALID;
  if (!c->have_loci) return fail(c, KGL_B200_ERR_STATE, "upload_loci first");
  int rc = use_device(c); if (rc) return rc;
  c->keep_valid = false; c->prep_valid = false;
  if (!keep) return KGL_B200_OK;
  if (n_loci != c->loci_len) return fail(c, KGL_B200_ERR_INVALID, "filter length differs from n_loci");
  KGL_CUDA(c, c->d_locus_keep.ensure(n_loci));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_locus_keep.p, keep, n_loci, cudaMemcpyHostToDevice, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  c->keep_valid = true;
  return KGL_B200_OK;
}

// RetrieveLociiVector::getLociiCount (kga_analysis_inbreed_locus.cpp:159-183 over getAllelesCount, :105-156): the first `count`
// accepted loci of one super-population from `lower` on. The accept rule is the one of kgl_b200_select_loci (same kernels); the
// rows are searched in growing spans until `count` loci are found or the contig ends -- accepting a locus only depends on the
// loci before it, so a truncated span gives the same prefix. Leaves the selection of the last span in place.
int kgl_b200_count_loci(kgl_b200_ctx* c, uint32_t pop, uint64_t lower, uint64_t spacing, uint64_t count, double min_af, double max_af,
                        uint64_t* n_found, uint64_t* last_offset) {
  if (!c || !n_found || !last_offset) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->have_loci || !c->have_offsets) return fail(c, KGL_B200_ERR_STATE, "upload_loci (with offsets) first");
  if (pop >= c->n_pop) return fail(c, KGL_B200_ERR_INVALID, "population index out of range");
  *n_found = 0; *last_offset = 0;
  const uint64_t L = c->loci_len;
  const uint64_t l_begin = first_row_at(c, lower);
  if (l_begin >= L || count == 0) return KGL_B200_OK;
  KGL_CUDA(c, c->d_sel_counts.ensure(kMaxPop));
  uint64_t span = std::max<uint64_t>(4096, std::min<uint64_t>(L, count * 16));
  for (;;) {
    const uint64_t l_end = std::min<uint64_t>(L, l_begin + span);
    int rc = kgl_b200_select_loci(c, lower, c->h_offsets[l_end - 1], spacing, min_af, max_af, nullptr); if (rc) return rc;
    unsigned long long* out = c->d_sel_counts.p;            // reused as {found, last row}
    k_rank_find<<<1, 1024, 0, c->stream>>>(c->d_sel.p, l_begin, l_end, (int)pop, count, out);
    KGL_LAUNCH_CHECK(c);
    unsigned long long h[2] = {0, 0};
    KGL_CUDA(c, cudaMemcpyAsync(h, out, 16, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    if (h[0] >= count || l_end == L) {
      *n_found = h[0];
      if (h[0] > 0) *last_offset = c->h_offsets[h[1]];
      return KGL_B200_OK;
    }
    span *= 8;
  }
}

int kgl_b200_synth_genotypes(kgl_b200_ctx* c, uint64_t seed, uint64_t n_genomes, uint64_t n_loci, uint64_t locus_base,
                             const double* inbreeding, double missing_rate) {
  if (!c || !inbreeding) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->have_loci || !c->have_superpop) return fail(c, KGL_B200_ERR_STATE, "upload_loci and set_genome_superpop first");
  if (c->h_superpop.size() != n_genomes || c->loci_len != n_loci)
    return fail(c, KGL_B200_ERR_INVALID, "shape differs from the uploaded loci / super-populations");
  int rc = use_device(c); if (rc) return rc;
  const uint64_t row_bytes = 16 * ((n_genomes + 63) / 64);
  rc = set_shape(c, n_genomes, n_loci, row_bytes);
  if (rc) return rc;
  rc = alloc_matrix(c); if (rc) return rc;
  KGL_CUDA(c, c->d_inbreeding.ensure(n_genomes));
  KGL_CUDA(c, cudaMemcpyAsync(c->d_inbreeding.p, inbreeding, n_genomes * 8, cudaMemcpyHostToDevice, c->stream));
  const uint64_t total = n_loci * c->units;
  k_synth<<<blocks_for(total, 256), 256, 0, c->stream>>>(seed, n_genomes, n_loci, locus_base, c->units, c->d_af.p, c->d_superpop.p,
                                                        c->d_inbreeding.p, (uint64_t)(missing_rate * 16777216.0),
                                                        reinterpret_cast<uint4*>(c->d_packed.p));
  KGL_LAUNCH_CHECK(c);
  c->have_geno = true;
  return build_dropped_index(c);     // synchronises the stream
}

int kgl_b200_download_genotypes(kgl_b200_ctx* c, uint64_t n_bytes, void* packed) {
  if (!c || !packed) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->have_geno) return fail(c, KGL_B200_ERR_STATE, "no genotype matrix on the device");
  if (n_bytes != c->L * c->row_bytes) return fail(c, KGL_B200_ERR_INVALID, "n_bytes must be n_loci*row_bytes");
  int rc = use_device(c); if (rc) return rc;
  KGL_CUDA(c, cudaMemcpy2DAsync(packed, c->row_bytes, c->d_packed.p, c->units * 16, c->row_bytes, c->L, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

int kgl_b200_run_allele_count(kgl_b200_ctx* c, uint32_t* locus_counts, uint64_t* genome_counts) {
  if (!c) return KGL_B200_ERR_INVALID;
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  rc = default_superpop(c); if (rc) return rc;
  if (genome_counts) KGL_CUDA(c, c->d_genome_counts.ensure((size_t)c->N * 4));
  rc = launch_count(c, true, locus_counts != nullptr, genome_counts != nullptr); if (rc) return rc;
  if (locus_counts)
    KGL_CUDA(c, cudaMemcpyAsync(locus_counts, c->d_locus_counts.p, (size_t)c->L * 16, cudaMemcpyDeviceToHost, c->stream));
  if (genome_counts) {
    k_genome_counts_raw<<<blocks_for(c->N, 256), 256, 0, c->stream>>>(c->d_gcounts, c->d_n3, c->N, c->L, c->d_genome_counts.p);
    KGL_LAUNCH_CHECK(c);
    KGL_CUDA(c, cudaMemcpyAsync(genome_counts, c->d_genome_counts.p, (size_t)c->N * 32, cudaMemcpyDeviceToHost, c->stream));
  }
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

int kgl_b200_run_hetero_homo(kgl_b200_ctx* c, int other_allele_entries, uint64_t* out) {
  if (!c || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  rc = default_superpop(c); if (rc) return rc;
  rc = launch_count(c, true, false, true); if (rc) return rc;
  KGL_CUDA(c, c->d_genome_counts.ensure((size_t)c->N * 7));
  k_hetero_homo<<<blocks_for(c->N, 128), 128, 0, c->stream>>>(c->d_gcounts, c->d_n3, c->n_multi ? c->d_multi_cells.p : nullptr, c->n_multi, c->N,
                                                              other_allele_entries ? 1u : 0u, c->d_genome_counts.p);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaMemcpyAsync(out, c->d_genome_counts.p, (size_t)c->N * 56, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

// HeteroHomoZygous::UpdateSampleLocation (kga_PfEMP/kga_analysis_PfEMP_heterozygous.cpp:362-412) on the records of
// kgl_b200_run_hetero_homo. Host arithmetic over n_genomes records (no device work): the location aggregates of
// HeteroHomoZygous::location_summary (:266-358: sums over the location's samples, radii_samples_OK_ = its QC-pass samples), the
// city -> country fallback below MINIMUM_LOCATION_SAMPLES_ (:375-388) and Wright's F_IS = (H_exp - H_obs) / H_exp.
int kgl_b200_location_fis(uint64_t n_genomes, const uint64_t* hetero_homo, uint32_t n_locations, const uint64_t* location_begin,
                          const uint32_t* location_members, const uint32_t* city_of_genome, const uint32_t* country_of_genome,
                          const uint8_t* qc_pass, uint32_t min_location_samples, double* fis) {
  if (!hetero_homo || !location_begin || !location_members || !city_of_genome || !country_of_genome || !fis) return KGL_B200_ERR_INVALID;
  std::vector<uint64_t> total(n_locations, 0), het(n_locations, 0), ok(n_locations, 0);
  for (uint32_t loc = 0; loc < n_locations; ++loc)
    for (uint64_t i = location_begin[loc]; i < location_begin[loc + 1]; ++i) {
      const uint32_t g = location_members[i];
      if (g >= n_genomes) return KGL_B200_ERR_INVALID;
      total[loc] += hetero_homo[(size_t)g * 7 + 0];
      het[loc] += hetero_homo[(size_t)g * 7 + 4] + hetero_homo[(size_t)g * 7 + 5];
      ok[loc] += (!qc_pass || qc_pass[g]) ? 1u : 0u;
    }
  for (uint64_t g = 0; g < n_genomes; ++g) {
    fis[g] = 0.0;
    uint32_t loc = city_of_genome[g];
    if (loc >= n_locations) continue;                        // no location record: the reference logs an error and leaves 0
    if (ok[loc] < min_location_samples) {
      loc = country_of_genome[g];
      if (loc >= n_locations) continue;
    }
    const uint64_t g_total = hetero_homo[g * 7 + 0], g_het = hetero_homo[g * 7 + 4] + hetero_homo[g * 7 + 5];
    if (total[loc] > 0 && g_total > 0) {
      const double expected_heterozygosity = static_cast<double>(het[loc]) / static_cast<double>(total[loc]);
      const double observed_heterozygosity = static_cast<double>(g_het) / static_cast<double>(g_total);
      fis[g] = (expected_heterozygosity - observed_heterozygosity) / expected_heterozygosity;
    }
  }
  return KGL_B200_OK;
}

int kgl_b200_enqueue_count_and_inbreed(kgl_b200_ctx* c) {
  if (!c) return KGL_B200_ERR_INVALID;
  int rc = use_device(c, false); if (rc) return rc;      // the tail of the pass before may still be running: it is not waited for
  rc = require_population(c, true); if (rc) return rc;
  c->prep_valid = false;   // the AF vectors are an input of the pass: the per-locus preparation is part of every step
  c->peer_results = false;
  KGL_CUDA(c, c->d_results.ensure(c->Npad));
  rc = enqueue_moments(c, true, true, false, false, true); if (rc) return rc;
  rc = mark_tail(c, false); if (rc) return rc;
  if (c->n_multi) {            // their share follows the tail on the context stream (no overlap with the next pass then)
    rc = join_tail(c); if (rc) return rc;
    rc = multi_add<MULTI_MOMENTS>(c, c->d_partials.p, c->d_results.p); if (rc) return rc;
  }
  c->algo = KGL_B200_ALGO_SIMPLE; c->phase = 0;     // kgl_b200_inbreed_fetch copies d_results
  return KGL_B200_OK;
}

int kgl_b200_flush(kgl_b200_ctx* c) {
  if (!c) return KGL_B200_ERR_INVALID;
  return use_device(c);
}

// ---- locus-sharded step with the exchange over peer memory -----------------------------------------------------------
static size_t xchg_bytes(uint64_t npad) { return (size_t)2 * npad * PART_COUNT * 8 + kPeerMaxRanks * 8; }

int kgl_b200_peer_export(kgl_b200_ctx* c, void* handle) {
  if (!c || !handle) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  if (c->Npad == 0) return fail(c, KGL_B200_ERR_STATE, "upload the genotype matrix (or synthesise it) before exporting the exchange region");
  static_assert(sizeof(cudaIpcMemHandle_t) == KGL_B200_PEER_HANDLE_BYTES, "handle size");
  peer_detach(c); peer_unregister(c);
  KGL_CUDA(c, c->d_xchg.ensure(xchg_bytes(c->Npad)));
  KGL_CUDA(c, c->d_peer_error.ensure(1));
  KGL_CUDA(c, cudaMemsetAsync(c->d_xchg.p, 0, xchg_bytes(c->Npad), c->stream));
  KGL_CUDA(c, cudaMemsetAsync(c->d_peer_error.p, 0, 4, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  c->xchg_npad = c->Npad; c->peer_epoch = 0; c->peer_results = false;
  cudaIpcMemHandle_t h;
  KGL_CUDA(c, cudaIpcGetMemHandle(&h, c->d_xchg.p));
  std::memcpy(handle, &h, sizeof h);
  LocalPeerRegion reg{};
  std::memcpy(reg.handle, &h, sizeof h);
  reg.ptr = c->d_xchg.p; reg.device = c->device; reg.owner = c;
  std::lock_guard<std::mutex> lock(g_peer_mu);
  g_peer_regions.push_back(reg);
  return KGL_B200_OK;
}

int kgl_b200_peer_attach(kgl_b200_ctx* c, uint32_t rank, uint32_t world, const void* handles) {
  if (!c || !handles) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (world == 0 || world > (uint32_t)kPeerMaxRanks || rank >= world) return fail(c, KGL_B200_ERR_INVALID, "bad rank / world");
  if (c->d_xchg.p == nullptr || c->xchg_npad != c->Npad) return fail(c, KGL_B200_ERR_STATE, "kgl_b200_peer_export first");
  int rc = use_device(c); if (rc) return rc;
  peer_detach(c);
  c->peer_base.assign(world, nullptr);
  c->peer_ipc.assign(world, 0);
  for (uint32_t r = 0; r < world; ++r) {
    if (r == rank) continue;
    const unsigned char* hb = static_cast<const unsigned char*>(handles) + (size_t)r * KGL_B200_PEER_HANDLE_BYTES;
    void* p = nullptr;
    int peer_device = -1;
    {
      std::lock_guard<std::mutex> lock(g_peer_mu);
      for (const LocalPeerRegion& reg : g_peer_regions)
        if (std::memcmp(reg.handle, hb, KGL_B200_PEER_HANDLE_BYTES) == 0) { p = reg.ptr; peer_device = reg.device; break; }
    }
    if (p) {                                   // a region of this process: mapped already; another GPU needs peer access
      if (peer_device != c->device) {
        cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
        KGL_CUDA(c, e);
      }
    } else {
      cudaIpcMemHandle_t h;
      std::memcpy(&h, hb, sizeof h);
      KGL_CUDA(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      c->peer_ipc[r] = 1;
    }
    c->peer_base[r] = p;
  }
  c->peer_rank = rank; c->peer_world = world;
  return KGL_B200_OK;
}

int kgl_b200_peer_set_timeout_ms(kgl_b200_ctx* c, uint64_t milliseconds) {
  if (!c || milliseconds == 0) return fail(c, KGL_B200_ERR_INVALID, "timeout must be positive");
  c->peer_timeout_ms = milliseconds;
  return KGL_B200_OK;
}

int kgl_b200_enqueue_count_and_inbreed_peer(kgl_b200_ctx* c) {
  if (!c) return KGL_B200_ERR_INVALID;
  int rc = use_device(c, false); if (rc) return rc;
  rc = require_population(c, true); if (rc) return rc;
  if (c->peer_world == 0 || c->xchg_npad != c->Npad) return fail(c, KGL_B200_ERR_STATE, "kgl_b200_peer_export / kgl_b200_peer_attach first");
  c->prep_valid = false;   // the AF vectors are an input of the pass, as in kgl_b200_enqueue_count_and_inbreed
  KGL_CUDA(c, c->d_results.ensure(c->Npad));
  KGL_CUDA(c, c->d_partials.ensure((size_t)c->Npad * PART_COUNT));
  const uint64_t epoch = ++c->peer_epoch;
  const uint64_t parity_doubles = c->Npad * PART_COUNT;
  c->partials_target = reinterpret_cast<double*>(c->d_xchg.p) + (epoch & 1ull) * parity_doubles;
  rc = enqueue_moments(c, true, false, false, false, true);
  if (!rc && c->n_multi) {
    rc = mark_tail(c, true);
    if (!rc) rc = multi_add<MULTI_MOMENTS>(c, c->partials_target);
  }
  c->partials_target = nullptr;
  if (rc) return rc;
  // the exchange follows the tail on the tail stream (the context stream when the population's code-3 cells are not indexed)
  cudaStream_t xs = c->tail_pending ? c->tail_stream : c->stream;
  PeerParams P{};
  for (uint32_t r = 0; r < c->peer_world; ++r) P.base[r] = static_cast<unsigned char*>(r == c->peer_rank ? (void*)c->d_xchg.p : c->peer_base[r]);
  P.rank = c->peer_rank; P.world = c->peer_world; P.parity_doubles = parity_doubles; P.epoch = epoch; P.n_genomes = c->N;
  P.timeout_ns = c->peer_timeout_ms * 1000000ull;
  P.partials_out = c->d_partials.p; P.results = c->d_results.p; P.error_word = c->d_peer_error.p;
  k_peer_publish<<<1, kPeerMaxRanks, 0, xs>>>(P);
  KGL_LAUNCH_CHECK(c);
  // one resident wave at most: every block of the exchange spins on the peers' flags
  const unsigned grid = std::min<unsigned>(blocks_for(c->N * 8, 256), (unsigned)c->sm_count * 4u);
  k_peer_exchange<<<grid, 256, 0, xs>>>(P);
  KGL_LAUNCH_CHECK(c);
  c->algo = KGL_B200_ALGO_SIMPLE; c->phase = 0;     // kgl_b200_inbreed_fetch copies d_results
  c->peer_results = true;
  return mark_tail(c, false);
}

// bytes of a result from src to the host and, when a peer step produced it, the verdict on that step: did a peer time out?
// (The error word is copied with the result.)
static int fetch_peer_checked(kgl_b200_ctx* c, void* dst, const void* src, size_t bytes) {
  unsigned int peer_word = 0;
  if (c->peer_results) KGL_CUDA(c, cudaMemcpyAsync(&peer_word, c->d_peer_error.p, 4, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  if (peer_word == 0) return KGL_B200_OK;
  peer_detach(c);                                 // the epochs of the ranks no longer agree: start over with export / attach
  c->peer_results = false;
  return fail(c, KGL_B200_ERR_PEER, "peer exchange timed out: a rank did not reach the step; export and attach the exchange regions again");
}

int kgl_b200_fetch_locus_counts(kgl_b200_ctx* c, uint32_t* locus_counts) {
  if (!c || !locus_counts) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (c->d_locus_counts.cap < (size_t)c->L * 4) return fail(c, KGL_B200_ERR_STATE, "no per-locus counts have been computed");
  int rc = use_device(c); if (rc) return rc;
  return fetch_peer_checked(c, locus_counts, c->d_locus_counts.p, (size_t)c->L * 16);
}

int kgl_b200_run_count_and_inbreed(kgl_b200_ctx* c, uint32_t* locus_counts, kgl_b200_locus_results* out) {
  int rc = kgl_b200_enqueue_count_and_inbreed(c); if (rc) return rc;
  rc = join_tail(c); if (rc) return rc;
  if (locus_counts)
    KGL_CUDA(c, cudaMemcpyAsync(locus_counts, c->d_locus_counts.p, (size_t)c->L * 16, cudaMemcpyDeviceToHost, c->stream));
  if (out)
    KGL_CUDA(c, cudaMemcpyAsync(out, c->d_results.p, (size_t)c->N * sizeof(kgl_b200_locus_results), cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

// ---- estimator state machine ----------------------------------------------------------------------------------------
int kgl_b200_inbreed_begin(kgl_b200_ctx* c, int algorithm, const kgl_b200_inbreed_options* options) {
  if (!c) return KGL_B200_ERR_INVALID;
  if (algorithm < KGL_B200_ALGO_SIMPLE || algorithm > KGL_B200_ALGO_LOGLIKELIHOOD) return fail(c, KGL_B200_ERR_INVALID, "unknown algorithm");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, true); if (rc) return rc;
  c->algo = algorithm; c->phase = 0; c->iteration = 0; c->peer_results = false;
  c->opt = options ? *options : kgl_b200_inbreed_options{};
  c->hall_start.clear();
  if (c->opt.hall_start) c->hall_start.assign(c->opt.hall_start, c->opt.hall_start + c->N);
  c->opt.hall_start = nullptr;
  if (c->opt.count_loci) c->prep_valid = false;               // fused step: the AF vectors are re-read every pass
  if (c->opt.hall_sweeps == 0) c->opt.hall_sweeps = 50;        // MINIMUM_ITERATIONS_ (calc.h:124), SURVEY Q1
  if (c->opt.ll_tolerance <= 0.0) c->opt.ll_tolerance = 1e-12;
  if (c->opt.ll_max_iterations <= 0) c->opt.ll_max_iterations = 200;
  KGL_CUDA(c, c->d_partials.ensure((size_t)c->Npad * PART_COUNT));
  KGL_CUDA(c, c->d_iter.ensure((size_t)c->Npad * ITER_COUNT));
  KGL_CUDA(c, cudaMemsetAsync(c->d_iter.p, 0, (size_t)c->Npad * ITER_COUNT * 8, c->stream));
  KGL_CUDA(c, c->d_f.ensure(c->Npad));
  KGL_CUDA(c, c->d_bracket.ensure((size_t)c->Npad * 4));
  KGL_CUDA(c, c->d_grid.ensure(kGridMax));
  KGL_CUDA(c, c->d_done.ensure(c->Npad));
  KGL_CUDA(c, c->d_flag.ensure(1));
  KGL_CUDA(c, c->d_results.ensure(c->Npad));
  KGL_CUDA(c, c->d_limits.ensure((size_t)c->Npad * 3));
  KGL_CUDA(c, c->d_lane_state.ensure(c->Npad));
  KGL_CUDA(c, c->d_n_slow.ensure(1));
  KGL_CUDA(c, c->d_list.ensure(c->Npad));
  KGL_CUDA(c, c->d_list_count.ensure(1));
  c->limits_valid = false; c->list_len = 0; c->table_mode = -1; c->used_moments = false;
  return KGL_B200_OK;
}

int kgl_b200_inbreed_accumulate(kgl_b200_ctx* c) {
  if (!c || c->algo < 0) return fail(c, KGL_B200_ERR_STATE, "inbreed_begin first");
  int rc = use_device(c); if (rc) return rc;
  FastLaunch fl;
  if (c->phase == 0) {
    rc = enqueue_moments(c, c->opt.count_loci != 0, false, c->algo == KGL_B200_ALGO_RITLAND, c->algo != KGL_B200_ALGO_SIMPLE); if (rc) return rc;
    if (c->algo == KGL_B200_ALGO_RITLAND) {
      rc = launch_fast<FAST_RITLAND>(c, fl); if (rc) return rc;
      k_ritland_partials<<<blocks_for(c->N, 256), 256, 0, c->stream>>>(c->d_chunk_out.p, fl.n_chunks, c->Npad, 2, dense_totals(c, c->prep[c->par]),
                                                                       c->d_superpop.p, c->N, c->d_partials.p);
      KGL_LAUNCH_CHECK(c);
    }
    if (c->algo == KGL_B200_ALGO_LOGLIKELIHOOD) {   // heterozygous cells of THIS locus shard, before the partials are all-reduced
      k_stash_nhet<<<blocks_for(c->N, 256), 256, 0, c->stream>>>(c->d_partials.p, PART_COUNT, PART_NMAJHET, PART_NMINHET, c->N, c->d_limits.p);
      KGL_LAUNCH_CHECK(c);
    }
    // the multi-allelic loci last: k_ritland_partials and k_stash_nhet above work on the dense path's counts alone
    return multi_add<MULTI_MOMENTS>(c, c->d_partials.p);
  }
  const unsigned nb = blocks_for(c->N, 256);
  if (c->algo == KGL_B200_ALGO_HALLME) {
    const bool tables = moments_enabled(c);
    if (tables) { rc = ensure_moments(c, false); if (rc) return rc; }
    if (tables && c->mom_supported) {
      c->used_moments = true;
      k_mom_eval<FAST_HALL><<<(unsigned)c->N, 128, 0, c->stream>>>(reinterpret_cast<const double*>(c->d_mom_mi.p), c->mom_b_lo, c->mom_nbt, c->d_f.p,
                                                                  nullptr, 0, nullptr, c->N, nullptr, nullptr, nullptr, nullptr, c->d_iter.p);
      KGL_LAUNCH_CHECK(c);
      return multi_add<MULTI_HALL>(c, c->d_iter.p);
    }
    rc = launch_fast<FAST_HALL>(c, fl); if (rc) return rc;
    k_hall_reduce<<<blocks_for(c->N * 8, 256), 256, 0, c->stream>>>(c->d_chunk_out.p, fl.n_chunks, c->Npad, c->N, c->d_iter.p);
    KGL_LAUNCH_CHECK(c);
    return multi_add<MULTI_HALL>(c, c->d_iter.p);
  }
  if (moments_enabled(c)) {
    rc = ensure_moments(c, true); if (rc) return rc;
    if (c->mom_supported) {
      if (!c->limits_valid) { rc = copy_moment_limits(c); if (rc) return rc; }
      c->used_moments = true;
      rc = newton_sweep_moments(c); if (rc) return rc;
      return multi_add<MULTI_NEWTON>(c, c->d_iter.p);
    }
  }
  if (!c->limits_valid) {      // once per root search: the selection is fixed between inbreed_begin and inbreed_fetch
    rc = launch_fast<FAST_LIMITS>(c, fl); if (rc) return rc;
    k_limits_reduce<<<nb, 256, 0, c->stream>>>(c->d_chunk_out.p, fl.n_chunks, c->Npad, c->N, c->d_limits.p);
    KGL_LAUNCH_CHECK(c);
    c->limits_valid = true;
  }
  rc = c->unphased ? newton_sweep<FAST_NEWTON_U>(c) : newton_sweep<FAST_NEWTON>(c);
  if (rc) return rc;
  return multi_add<MULTI_NEWTON>(c, c->d_iter.p);     // evaluated cell by cell, clamps included (a clamped homozygous term moves the search right)
}

int kgl_b200_inbreed_used_moment_tables(const kgl_b200_ctx* c) { return c && c->used_moments ? (c->mom_used_mma ? 2 : 1) : 0; }

int kgl_b200_inbreed_partials_buffer(kgl_b200_ctx* c, void** device_ptr, uint64_t* n_doubles) {
  if (!c || !device_ptr || !n_doubles || c->algo < 0) return fail(c, KGL_B200_ERR_STATE, "inbreed_begin first");
  *device_ptr = (c->phase == 0) ? (void*)c->d_partials.p : (void*)c->d_iter.p;
  *n_doubles = c->N * (uint64_t)((c->phase == 0) ? PART_COUNT : ITER_COUNT);
  return KGL_B200_OK;
}

int kgl_b200_inbreed_update(kgl_b200_ctx* c, int* finished) {
  if (!c || !finished || c->algo < 0) return fail(c, KGL_B200_ERR_STATE, "inbreed_begin first");
  int rc = use_device(c); if (rc) return rc;
  const unsigned nb = blocks_for(c->N, 256);
  *finished = 0;
  if (c->phase == 0) {
    if (c->algo == KGL_B200_ALGO_SIMPLE || c->algo == KGL_B200_ALGO_RITLAND) {
      k_finalize_closed_form<<<nb, 256, 0, c->stream>>>(c->d_partials.p, c->N, c->algo, c->d_results.p, nullptr);
      KGL_LAUNCH_CHECK(c);
      *finished = 1;
      return KGL_B200_OK;
    }
    if (c->algo == KGL_B200_ALGO_HALLME) {
      if (!c->hall_start.empty()) {
        KGL_CUDA(c, cudaMemcpyAsync(c->d_f.p, c->hall_start.data(), c->N * 8, cudaMemcpyHostToDevice, c->stream));
        KGL_CUDA(c, cudaStreamSynchronize(c->stream));
      } else {
        k_fill_double<<<nb, 256, 0, c->stream>>>(c->d_f.p, c->N, 0.25);
        KGL_LAUNCH_CHECK(c);
      }
    } else {
      k_ll_init<<<nb, 256, 0, c->stream>>>(c->d_partials.p, c->N, c->d_f.p, c->d_bracket.p, c->d_done.p);
      KGL_LAUNCH_CHECK(c);
    }
    c->phase = 1; c->iteration = 0;
    return KGL_B200_OK;
  }
  // the update kernels read the (all-reduced) moments from d_partials and the (all-reduced) iteration terms from d_iter
  KGL_CUDA(c, cudaMemsetAsync(c->d_flag.p, 0, 8, c->stream));
  unsigned long long flag = 0;
  if (c->algo == KGL_B200_ALGO_HALLME) {
    ++c->iteration;
    k_hall_update<<<nb, 256, 0, c->stream>>>(c->d_partials.p, c->d_iter.p, c->N, c->d_f.p, c->d_flag.p);
    KGL_LAUNCH_CHECK(c);
    if (c->opt.hall_sweeps > 0) { *finished = (c->iteration >= c->opt.hall_sweeps) ? 1 : 0; return KGL_B200_OK; }
    KGL_CUDA(c, cudaMemcpyAsync(&flag, c->d_flag.p, 8, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    double max_delta; std::memcpy(&max_delta, &flag, 8);
    *finished = (max_delta < 1e-15 || c->iteration >= 100000) ? 1 : 0;
    return KGL_B200_OK;
  }
  ++c->iteration;
  k_ll_step<<<nb, 256, 0, c->stream>>>(c->d_iter.p, c->N, c->opt.ll_tolerance, c->d_f.p, c->d_bracket.p, c->d_done.p, c->d_flag.p);
  KGL_LAUNCH_CHECK(c);
  // Late sweeps work on a short list of genomes and cost less than a host round trip: while the list is in use the host
  // looks at the number of unfinished genomes only every fourth sweep; in between the list is re-compacted on the device and
  // its length read there (a sweep over an empty list returns at once, a finished genome ignores further steps).
  if (c->list_len && (c->iteration & 3) != 0 && c->iteration < c->opt.ll_max_iterations) {
    k_compact_active<<<1, 1024, 0, c->stream>>>(c->d_done.p, c->N, c->d_list.p, c->d_list_count.p);
    KGL_LAUNCH_CHECK(c);
    return KGL_B200_OK;
  }
  KGL_CUDA(c, cudaMemcpyAsync(&flag, c->d_flag.p, 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  *finished = (flag == 0 || c->iteration >= c->opt.ll_max_iterations) ? 1 : 0;
  // flag = genomes still searching. Once they are a minority the sweeps gather them through a list: the work of a sweep
  // follows the number of live genomes, not N (every rank sees the same done flags, so the same list).
  c->list_len = 0;
  if (!*finished && flag * 2 <= c->N) {
    k_compact_active<<<1, 1024, 0, c->stream>>>(c->d_done.p, c->N, c->d_list.p, c->d_list_count.p);
    KGL_LAUNCH_CHECK(c);
    c->list_len = flag;
  }
  return KGL_B200_OK;
}

int kgl_b200_inbreed_fetch(kgl_b200_ctx* c, kgl_b200_locus_results* out) {
  if (!c || !out || c->algo < 0) return fail(c, KGL_B200_ERR_STATE, "inbreed_begin first");
  int rc = use_device(c); if (rc) return rc;
  if (c->algo == KGL_B200_ALGO_HALLME || c->algo == KGL_B200_ALGO_LOGLIKELIHOOD) {
    k_store_coeff<<<blocks_for(c->N, 256), 256, 0, c->stream>>>(c->d_partials.p, c->d_f.p, c->N, c->d_results.p);
    KGL_LAUNCH_CHECK(c);
  }
  return fetch_peer_checked(c, out, c->d_results.p, (size_t)c->N * sizeof(kgl_b200_locus_results));
}

// HallME / the root search as ONE launch over the moment tables (k_mom_run): this context holds every locus, so nothing has to
// be all-reduced between sweeps. Leaves *finished at 0 when the tables are not available (or a genome needs the exact
// kernel): the caller then continues with the sweep-by-sweep protocol from the state the launch left behind.
static int run_whole_from_tables(kgl_b200_ctx* c, int* finished) {
  const bool hall = c->algo == KGL_B200_ALGO_HALLME;
  if (!moments_enabled(c) || c->n_multi != 0 || c->opt.sweep_by_sweep) return KGL_B200_OK;
  int rc = ensure_moments(c, !hall); if (rc) return rc;
  if (!c->mom_supported) return KGL_B200_OK;
  const size_t smem = (size_t)c->mom_nbt * (kMomJ * 8 + 16);
  if (smem > 200 * 1024) return KGL_B200_OK;
  MomRunParams P{};
  P.mom = reinterpret_cast<const double*>(c->d_mom_mi.p); P.b_lo = c->mom_b_lo; P.nbt = c->mom_nbt; P.n_genomes = c->N;
  P.partials = c->d_partials.p; P.f = c->d_f.p; P.hall_sweeps = c->opt.hall_sweeps;
  c->used_moments = true;
  if (hall) {
    KGL_CUDA(c, cudaFuncSetAttribute(k_mom_run<FAST_HALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_mom_run<FAST_HALL><<<(unsigned)c->N, kMomRunThreads, smem, c->stream>>>(P);
    KGL_LAUNCH_CHECK(c);
    c->iteration = c->opt.hall_sweeps > 0 ? c->opt.hall_sweeps : 0;
    *finished = 1;
    return KGL_B200_OK;
  }
  rc = copy_moment_limits(c); if (rc) return rc;
  P.rare = c->d_mom_list.p; P.base = c->d_mom_base.p; P.totals = c->d_mom_totals.p; P.limits = c->d_limits.p;
  P.bracket = c->d_bracket.p; P.done = c->d_done.p; P.tol = c->opt.ll_tolerance; P.max_iterations = c->opt.ll_max_iterations;
  P.remaining = c->d_flag.p;
  KGL_CUDA(c, cudaMemsetAsync(c->d_flag.p, 0, 8, c->stream));
  KGL_CUDA(c, cudaFuncSetAttribute(k_mom_run<FAST_NEWTON>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_mom_run<FAST_NEWTON><<<(unsigned)c->N, kMomRunThreads, smem, c->stream>>>(P);
  KGL_LAUNCH_CHECK(c);
  unsigned long long remaining = 0;
  KGL_CUDA(c, cudaMemcpyAsync(&remaining, c->d_flag.p, 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  *finished = remaining == 0 ? 1 : 0;
  return KGL_B200_OK;
}

int kgl_b200_run_inbreed(kgl_b200_ctx* c, int algorithm, const kgl_b200_inbreed_options* options, kgl_b200_locus_results* out) {
  if (!c || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = kgl_b200_inbreed_begin(c, algorithm, options); if (rc) return rc;
  int finished = 0;
  rc = kgl_b200_inbreed_accumulate(c); if (rc) return rc;           // the counting pass
  rc = kgl_b200_inbreed_update(c, &finished); if (rc) return rc;
  if (!finished) { rc = run_whole_from_tables(c, &finished); if (rc) return rc; }
  while (!finished) {
    rc = kgl_b200_inbreed_accumulate(c); if (rc) return rc;
    rc = kgl_b200_inbreed_update(c, &finished); if (rc) return rc;
  }
  return kgl_b200_inbreed_fetch(c, out);
}

int kgl_b200_run_loglik_grid(kgl_b200_ctx* c, const double* grid, uint64_t n_grid, double* out) {
  if (!c || !grid || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, true); if (rc) return rc;
  rc = ensure_prepared(c, false, true); if (rc) return rc;
  KGL_CUDA(c, c->d_grid.ensure(kGridMax));
  // Sums the n_chunks chunk outputs at src ([n_chunks][Npad][kGridMax]) of every genome and of grid points g0 .. g0 + ng - 1 on
  // the host, in chunk order, into out (add: onto what is there).
  std::vector<double> chunks;
  auto sum_chunks = [&](const double* src, uint64_t n_chunks, uint64_t g0, int ng, bool add) {
    chunks.resize((size_t)n_chunks * c->Npad * kGridMax);
    KGL_CUDA(c, cudaMemcpyAsync(chunks.data(), src, chunks.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    for (uint64_t g = 0; g < c->N; ++g)
      for (int j = 0; j < ng; ++j) {
        double s = 0.0;
        for (uint64_t ch = 0; ch < n_chunks; ++ch) s += chunks[(ch * c->Npad + g) * kGridMax + j];
        double& o = out[g * n_grid + g0 + j];
        o = add ? o + s : s;
      }
    return KGL_B200_OK;
  };
  for (uint64_t g0 = 0; g0 < n_grid; g0 += kGridMax) {
    const int ng = (int)std::min<uint64_t>(kGridMax, n_grid - g0);
    KGL_CUDA(c, cudaMemcpyAsync(c->d_grid.p, grid + g0, ng * 8, cudaMemcpyHostToDevice, c->stream));
    TermLaunch tl;
    rc = launch_grid_terms(c, c->d_grid.p, ng, tl); if (rc) return rc;
    rc = sum_chunks(c->d_chunk_out.p, tl.n_chunks, g0, ng, false); if (rc) return rc;
    if (c->n_multi) {          // the terms of the multi-allelic loci, cell by cell
      if (g0 == 0) { rc = multi_launch_prepare(c); if (rc) return rc; }
      uint64_t mc = 0;
      rc = multi_launch_terms<MULTI_GRID>(c, c->d_grid.p, ng, mc); if (rc) return rc;
      rc = sum_chunks(c->d_multi_out.p, mc, g0, ng, true); if (rc) return rc;
    }
  }
  return KGL_B200_OK;
}

int kgl_b200_run_ibs(kgl_b200_ctx* c, uint64_t row_begin, uint64_t row_end, uint32_t* out) {
  if (!c || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  if (row_begin >= row_end || row_end > c->N) return fail(c, KGL_B200_ERR_INVALID, "bad genome row range");
  rc = ensure_ibs_planes(c); if (rc) return rc;
  return run_pairwise(c, row_begin, row_end, 4, c->d_ibs, out, [c](const TileList& tiles, uint64_t r0, uint64_t r1, int mirror) {
    int rc = ibs_compute_tiles(c, tiles); if (rc) return rc;
    return ibs_finalize(c, (uint32_t)tiles.key.n, 1, r0, r1, mirror, c->d_ibs.p);
  });
}

int kgl_b200_run_king(kgl_b200_ctx* c, uint64_t row_begin, uint64_t row_end, double* kinship) {
  if (!c || !kinship) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = king_check(c); if (rc) return rc;
  if (row_begin >= row_end || row_end > c->N) return fail(c, KGL_B200_ERR_INVALID, "bad genome row range");
  return run_pairwise(c, row_begin, row_end, 1, c->d_king_out, kinship, [c](const TileList& tiles, uint64_t r0, uint64_t r1, int mirror) {
    KingTiles K{};
    int rc = king_compute_tiles(c, tiles, K); if (rc) return rc;
    k_king_dense<<<blocks_for((uint64_t)K.n_tiles * kIbsTileCells, 256), 256, 0, c->stream>>>(K, r0, r1, mirror, c->d_king_out.p);
    KGL_LAUNCH_CHECK(c);
    return KGL_B200_OK;
  });
}

int kgl_b200_run_king_pairs(kgl_b200_ctx* c, uint64_t n_coords, const uint32_t* coords, double min_kinship, uint64_t capacity,
                            kgl_b200_king_pair* pairs, uint64_t* n_pairs) {
  if (!c || !pairs || !n_pairs) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = king_check(c); if (rc) return rc;
  const uint64_t side = ibs_side(c), n_upper = side * (side + 1) / 2;
  const bool all = coords == nullptr || n_coords == 0;
  const uint64_t n_tiles = all ? n_upper : n_coords;
  std::vector<TileList> slabs;           // every coordinate is checked before anything runs
  for (uint64_t t0 = 0; t0 < n_tiles; t0 += kIbsMaxTilesPerLaunch) {
    const uint64_t n = std::min(n_tiles - t0, kIbsMaxTilesPerLaunch);
    if (all) {
      slabs.push_back(upper_tiles(t0, 1, n));
    } else {
      slabs.emplace_back();
      rc = listed_tiles(c, coords + 2 * t0, n, true, slabs.back()); if (rc) return rc;
    }
  }
  // device list: no more records than the tiles hold, and indices that fit the uint32 sort values
  const uint64_t dev_cap = std::min<uint64_t>(std::min<uint64_t>(capacity, n_tiles * kIbsTileCells), 0xFFFFFFFFull);
  KGL_CUDA(c, c->d_king_pairs.ensure(dev_cap));
  KGL_CUDA(c, c->d_king_keys.ensure(dev_cap));
  KGL_CUDA(c, c->d_king_index.ensure(dev_cap));
  KGL_CUDA(c, c->d_king_cursor.ensure(1));
  KGL_CUDA(c, cudaMemsetAsync(c->d_king_cursor.p, 0, 8, c->stream));
  KingTiles K{};
  for (const TileList& tiles : slabs) {
    rc = king_compute_tiles(c, tiles, K); if (rc) return rc;
    k_king_pairs<<<blocks_for((uint64_t)K.n_tiles * kIbsTileCells, 256), 256, 0, c->stream>>>(K, min_kinship, dev_cap, c->d_king_pairs.p,
                                                                                               c->d_king_keys.p, c->d_king_index.p, c->d_king_cursor.p);
    KGL_LAUNCH_CHECK(c);
  }
  unsigned long long total = 0;
  KGL_CUDA(c, cudaMemcpyAsync(&total, c->d_king_cursor.p, 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  *n_pairs = total;
  if (total > capacity || total > dev_cap) return fail(c, KGL_B200_ERR_NOMEM, "more related pairs than capacity (*n_pairs holds the total)");
  if (total == 0) return KGL_B200_OK;
  // ascending (a, b) whatever the order in which the warps appended
  const uint64_t n = total;
  int end_bit = 32;                                                // b in the low word, a < N above it
  for (uint64_t v = c->N - 1; v; v >>= 1) ++end_bit;
  KGL_CUDA(c, c->d_king_keys2.ensure(n));
  KGL_CUDA(c, c->d_king_index2.ensure(n));
  KGL_CUDA(c, c->d_king_sorted.ensure(n));
  size_t temp_bytes = 0;
  KGL_CUDA(c, cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, c->d_king_keys.p, c->d_king_keys2.p, c->d_king_index.p, c->d_king_index2.p,
                                              n, 0, end_bit, c->stream));
  KGL_CUDA(c, c->d_king_sort_temp.ensure(temp_bytes));
  KGL_CUDA(c, cub::DeviceRadixSort::SortPairs(c->d_king_sort_temp.p, temp_bytes, c->d_king_keys.p, c->d_king_keys2.p, c->d_king_index.p,
                                              c->d_king_index2.p, n, 0, end_bit, c->stream));
  k_king_gather<<<blocks_for(n, 256), 256, 0, c->stream>>>(c->d_king_pairs.p, c->d_king_index2.p, n, c->d_king_sorted.p);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaMemcpyAsync(pairs, c->d_king_sorted.p, n * sizeof(kgl_b200_king_pair), cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

int kgl_b200_set_ibs_tensor_cores(kgl_b200_ctx* c, int enable) {
  if (!c) return KGL_B200_ERR_INVALID;
  c->ibs_tensor_enabled = enable != 0;
  c->ibs_tiles_key = TileKey{}; c->ibs_n_blocks = 0;         // the cached tile list carries no block list for the other form
  return KGL_B200_OK;
}

int kgl_b200_ibs_used_tensor_cores(const kgl_b200_ctx* c) { return c && c->ibs_used_tensor ? 1 : 0; }

int kgl_b200_ibs_tile_grid(kgl_b200_ctx* c, uint64_t* tiles_per_side, uint64_t* n_upper_tiles) {
  if (!c) return KGL_B200_ERR_INVALID;
  if (!c->have_geno) return fail(c, KGL_B200_ERR_STATE, "no genotype matrix uploaded");
  const uint64_t side = ibs_side(c);
  if (tiles_per_side) *tiles_per_side = side;
  if (n_upper_tiles) *n_upper_tiles = side * (side + 1) / 2;
  return KGL_B200_OK;
}

int kgl_b200_enqueue_ibs_tiles(kgl_b200_ctx* c, uint64_t first, uint64_t stride, uint64_t count) {
  if (!c) return KGL_B200_ERR_INVALID;
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  const uint64_t side = ibs_side(c), n_upper = side * (side + 1) / 2;
  if (stride == 0 || count == 0 || count > kIbsMaxTilesPerLaunch || first + (count - 1) * stride >= n_upper)
    return fail(c, KGL_B200_ERR_INVALID, "bad tile range (count must be 1..8192 per call and stay inside the upper triangle)");
  rc = ensure_ibs_planes(c); if (rc) return rc;
  return ibs_enqueue_tiles(c, upper_tiles(first, stride, count));
}

int kgl_b200_enqueue_ibs_tile_list(kgl_b200_ctx* c, uint64_t count, const uint32_t* coords) {
  if (!c || !coords) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  if (count == 0 || count > kIbsMaxTilesPerLaunch) return fail(c, KGL_B200_ERR_INVALID, "bad tile count (1..8192 per call)");
  TileList tiles;
  rc = listed_tiles(c, coords, count, false, tiles); if (rc) return rc;
  rc = ensure_ibs_planes(c); if (rc) return rc;
  return ibs_enqueue_tiles(c, tiles);
}

int kgl_b200_run_ibs_tile_list(kgl_b200_ctx* c, uint64_t count, const uint32_t* coords, uint32_t* out) {
  if (!c || !coords || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  return ibs_run_tiles(c, count, out, [&](uint64_t done, uint64_t n) { return kgl_b200_enqueue_ibs_tile_list(c, n, coords + 2 * done); });
}

int kgl_b200_run_ibs_tiles(kgl_b200_ctx* c, uint64_t first, uint64_t stride, uint64_t count, uint32_t* out) {
  if (!c || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  return ibs_run_tiles(c, count, out, [&](uint64_t done, uint64_t n) { return kgl_b200_enqueue_ibs_tiles(c, first + done * stride, stride, n); });
}

int kgl_b200_ibs_tiles_buffer(kgl_b200_ctx* c, void** device_ptr, uint64_t* n_u32) {
  if (!c || !device_ptr || !n_u32) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (c->ibs_last_count == 0) return fail(c, KGL_B200_ERR_STATE, "enqueue_ibs_tiles first");
  *device_ptr = c->d_ibs_tiles_out.p;
  *n_u32 = c->ibs_last_count * kIbsTileCells * 4;
  return KGL_B200_OK;
}

int kgl_b200_ibs_timer_reset(kgl_b200_ctx* c) {
  if (!c) return KGL_B200_ERR_INVALID;
  c->ibs_timer.used = 0;
  return KGL_B200_OK;
}

int kgl_b200_ibs_timer_read(kgl_b200_ctx* c, float* ms, uint32_t capacity, uint32_t* n) {
  if (!c || !ms || !n) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  KGL_CUDA(c, c->ibs_timer.read(ms, capacity, n));
  return KGL_B200_OK;
}

int kgl_b200_enqueue_gram_tiles(kgl_b200_ctx* c, uint64_t first, uint64_t stride) {
  if (!c) return KGL_B200_ERR_INVALID;
  if (stride == 0 || first >= stride) return fail(c, KGL_B200_ERR_INVALID, "need first < stride");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  if (c->L >= (1ull << 29)) return fail(c, KGL_B200_ERR_INVALID, "Gram matrix: more than 2^29 loci would overflow the int32 accumulators");
  return gram_compute(c, first, stride);
}

int kgl_b200_enqueue_gram(kgl_b200_ctx* c) { return kgl_b200_enqueue_gram_tiles(c, 0, 1); }

int kgl_b200_gram_buffer(kgl_b200_ctx* c, void** device_ptr, uint64_t* n_int32, uint64_t* ld) {
  if (!c || !device_ptr || !n_int32) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->gram_valid) return fail(c, KGL_B200_ERR_STATE, "enqueue_gram first");
  *device_ptr = c->d_gram.p; *n_int32 = gram_ld(c) * gram_ld(c);
  if (ld) *ld = gram_ld(c);
  return KGL_B200_OK;
}

int kgl_b200_fetch_gram(kgl_b200_ctx* c, int32_t* out) {
  if (!c || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->gram_valid) return fail(c, KGL_B200_ERR_STATE, "enqueue_gram first");
  int rc = use_device(c); if (rc) return rc;
  const size_t n2 = (size_t)c->N * c->N;
  KGL_CUDA(c, c->d_gram_out.ensure(n2 * 4));
  k_gram_finalize<<<blocks_for(n2, 256), 256, 0, c->stream>>>(c->d_gram.p, gram_ld(c), c->N, nullptr, 0, c->d_gram_out.p);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaMemcpyAsync(out, c->d_gram_out.p, n2 * 4, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

float kgl_b200_last_gram_kernel_ms(kgl_b200_ctx* c) { return c && c->gram_e1 ? event_ms(c, c->gram_e0, c->gram_e1) : -1.0f; }

int kgl_b200_run_gram(kgl_b200_ctx* c, int32_t* out) {
  if (!c || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = kgl_b200_enqueue_gram(c); if (rc) return rc;
  return kgl_b200_fetch_gram(c, out);
}

int kgl_b200_run_grm(kgl_b200_ctx* c, uint32_t pop, double* out) {
  if (!c || !out) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  if (!c->have_loci || c->loci_len != c->L) return fail(c, KGL_B200_ERR_STATE, "the centred matrix needs the allele frequencies (kgl_b200_upload_loci)");
  if (pop >= c->n_pop) return fail(c, KGL_B200_ERR_INVALID, "population index out of range");
  int rc = kgl_b200_enqueue_gram(c); if (rc) return rc;
  const float* af_pop = c->d_af.p + (size_t)pop * c->L;
  const uint64_t rows = c->n_gblocks * 32, n_chunks = (c->n_words + kDotWords - 1) / kDotWords;
  KGL_CUDA(c, c->d_gp_chunks.ensure(n_chunks * rows));
  KGL_CUDA(c, c->d_gp.ensure(rows + 1));
  dim3 grid((unsigned)((c->n_gblocks + 7) / 8), (unsigned)n_chunks);
  k_dosage_dot<<<grid, 256, 0, c->stream>>>(c->d_sm_lo.p, c->d_sm_hi.p, c->n_gblocks, c->n_words, c->L, af_pop, c->d_gp_chunks.p);
  KGL_LAUNCH_CHECK(c);
  k_dosage_reduce<<<blocks_for(rows, 256) + 1, 256, 0, c->stream>>>(c->d_gp_chunks.p, n_chunks, rows, af_pop, c->L, c->d_gp.p);
  KGL_LAUNCH_CHECK(c);
  const size_t n2 = (size_t)c->N * c->N;
  KGL_CUDA(c, c->d_gram_out.ensure(n2 * 8));
  k_gram_finalize<<<blocks_for(n2, 256), 256, 0, c->stream>>>(c->d_gram.p, gram_ld(c), c->N, c->d_gp.p, rows, c->d_gram_out.p);
  KGL_LAUNCH_CHECK(c);
  KGL_CUDA(c, cudaMemcpyAsync(out, c->d_gram_out.p, n2 * 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

// CalcFWS::updateGenomeFWSMap (kga_PfEMP/kga_analysis_PfEMP_FWS.cpp:72-101) for all bins: per AF bin one masked pass of the
// streaming kernel (the reference filters the population and rebuilds a VariantDBVariant per bin, :27-35).
int kgl_b200_run_binned_genome_counts(kgl_b200_ctx* c, uint32_t pop, uint32_t n_bins, const double* lower, const double* upper,
                                      int present_only, uint64_t* genome_counts, uint64_t* bin_rows) {
  if (!c || !lower || !upper || !genome_counts || n_bins == 0) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  if (!c->have_loci || c->loci_len != c->L) return fail(c, KGL_B200_ERR_STATE, "AF bins need the allele frequencies (kgl_b200_upload_loci)");
  if (pop >= c->n_pop) return fail(c, KGL_B200_ERR_INVALID, "population index out of range");
  // "variants of the population" = rows carried by at least one genome: needs the per-locus counts of a raw pass
  if (present_only) { rc = launch_count(c, true, true, false); if (rc) return rc; }
  if (c->n_multi && present_only) {      // which alleles of the multi-allelic loci occur
    KGL_CUDA(c, c->d_multi_counts.ensure(c->n_multi * kMultiSlots * 3));
    k_multi_allele_count<<<(unsigned)c->n_multi, 256, 0, c->stream>>>(c->d_multi_cells.p, c->N, c->d_multi_counts.p);
    KGL_LAUNCH_CHECK(c);
  }
  if (c->bin_tables_n != c->N || c->bin_tables_units != c->units) {
    std::vector<uint32_t> pm(c->units * 2, 0);
    for (uint64_t g = 0; g < c->N; ++g) pm[g >> 5] |= 1u << (g & 31);
    std::vector<uint8_t> need(c->units * 2, 1);
    KGL_CUDA(c, c->d_bin_popmask32.ensure(pm.size()));
    KGL_CUDA(c, c->d_bin_need32.ensure(need.size()));
    KGL_CUDA(c, c->d_zero_superpop.ensure(c->Npad));
    KGL_CUDA(c, c->d_bin_state.ensure(2));
    KGL_CUDA(c, cudaMemcpyAsync(c->d_bin_popmask32.p, pm.data(), pm.size() * 4, cudaMemcpyHostToDevice, c->stream));
    KGL_CUDA(c, cudaMemcpyAsync(c->d_bin_need32.p, need.data(), need.size(), cudaMemcpyHostToDevice, c->stream));
    KGL_CUDA(c, cudaMemsetAsync(c->d_zero_superpop.p, 0, c->Npad, c->stream));
    KGL_CUDA(c, cudaStreamSynchronize(c->stream));
    c->bin_tables_n = c->N; c->bin_tables_units = c->units;
  }
  KGL_CUDA(c, c->d_bin_flags.ensure(c->padded_rows));
  KGL_CUDA(c, c->d_bin_sum64.ensure(c->padded_rows / 64));
  KGL_CUDA(c, c->d_bin_out.ensure((size_t)n_bins * c->N * 4 + n_bins));
  const MaskOverride mo{c->d_bin_flags.p, c->d_bin_sum64.p, c->d_bin_popmask32.p, c->d_bin_need32.p, c->d_zero_superpop.p};
  for (uint32_t b = 0; b < n_bins; ++b) {
    KGL_CUDA(c, cudaMemsetAsync(c->d_bin_state.p, 0, 8, c->stream));
    k_bin_flags<<<blocks_for(c->padded_rows, 256), 256, 0, c->stream>>>(c->d_af.p + (size_t)pop * c->L, present_only ? c->d_locus_counts.p : nullptr,
                                                                         c->L, c->padded_rows, lower[b], upper[b], c->keep_valid ? c->d_locus_keep.p : nullptr,
                                                                         c->d_bin_flags.p, c->d_bin_sum64.p, c->d_bin_state.p + 1);
    KGL_LAUNCH_CHECK(c);
    rc = launch_count(c, false, false, true, false, false, &mo); if (rc) return rc;
    k_genome_counts_masked<<<blocks_for(c->N, 256), 256, 0, c->stream>>>(c->d_gcounts, c->d_n3, c->N, c->d_bin_state.p + 1,
                                                                         c->d_bin_out.p + (size_t)b * c->N * 4, c->d_bin_out.p + (size_t)n_bins * c->N * 4 + b);
    KGL_LAUNCH_CHECK(c);
    if (c->n_multi) {
      k_multi_bin_counts<<<blocks_for(c->N, 128), 128, 0, c->stream>>>(c->d_multi_cells.p, c->d_multi_af.p + (size_t)pop * c->n_multi * kMultiSlots,
                                                                       present_only ? c->d_multi_counts.p : nullptr, c->d_multi_rows.p,
                                                                       c->keep_valid ? c->d_locus_keep.p : nullptr, c->n_multi, c->N, lower[b], upper[b],
                                                                       c->d_bin_out.p + (size_t)b * c->N * 4, c->d_bin_out.p + (size_t)n_bins * c->N * 4 + b);
      KGL_LAUNCH_CHECK(c);
    }
  }
  KGL_CUDA(c, cudaMemcpyAsync(genome_counts, c->d_bin_out.p, (size_t)n_bins * c->N * 32, cudaMemcpyDeviceToHost, c->stream));
  if (bin_rows) KGL_CUDA(c, cudaMemcpyAsync(bin_rows, c->d_bin_out.p + (size_t)n_bins * c->N * 4, (size_t)n_bins * 8, cudaMemcpyDeviceToHost, c->stream));
  KGL_CUDA(c, cudaStreamSynchronize(c->stream));
  return KGL_B200_OK;
}

int kgl_b200_run_grm_product(kgl_b200_ctx* c, const uint8_t* keep, uint32_t n_cols, const double* x, double* y, uint64_t* n_loci_used) {
  if (!c || !x || !y) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  if (n_cols == 0 || n_cols > (uint32_t)kPcaMaxCols) return fail(c, KGL_B200_ERR_INVALID, "n_cols must be 1..48");
  uint64_t m = 0;
  rc = pca_prepare(c, keep, m); if (rc) return rc;
  if (m == 0) return fail(c, KGL_B200_ERR_INVALID, "no used locus (keep, and 0 < p < 1)");
  rc = pca_apply(c, n_cols, x, y, nullptr); if (rc) return rc;
  if (n_loci_used) *n_loci_used = m;
  return KGL_B200_OK;
}

int kgl_b200_run_pca(kgl_b200_ctx* c, const kgl_b200_pca_options* options, double* eigenvalues, double* scores, double* loadings,
                     uint64_t* n_loci_used) {
  if (!c || !eigenvalues || !scores) return fail(c, KGL_B200_ERR_INVALID, "null argument");
  int rc = use_device(c); if (rc) return rc;
  rc = require_population(c, false); if (rc) return rc;
  const kgl_b200_pca_options opt = options ? *options : kgl_b200_pca_options{};
  const uint32_t k = opt.n_components ? opt.n_components : 10, q = opt.iterations ? opt.iterations : 10;
  const uint64_t N = c->N, L = c->L;
  if (k > 40 || k >= N) return fail(c, KGL_B200_ERR_INVALID, "n_components must be 1..40 and below n_genomes");
  uint64_t m = 0;
  rc = pca_prepare(c, opt.keep, m); if (rc) return rc;
  if (m == 0) return fail(c, KGL_B200_ERR_INVALID, "no used locus (keep, and 0 < p < 1)");
  if (k > m) return fail(c, KGL_B200_ERR_INVALID, "n_components exceeds the used loci");
  // block width 16 ceil((k + 6) / 16), at most the genomes
  const uint32_t b = (uint32_t)std::min<uint64_t>(N, (k + 6 + 15) / 16 * 16);
  std::vector<double> qb((size_t)N * b), aq((size_t)N * b);
  for (uint64_t g = 0; g < N; ++g)
    for (uint32_t j = 0; j < b; ++j) qb[g * b + j] = pca_start_entry(opt.seed, g, j);
  pca_orth(qb, N, b);
  for (uint32_t it = 0; it < q; ++it) {
    rc = pca_apply(c, b, qb.data(), aq.data(), nullptr); if (rc) return rc;
    qb.swap(aq);
    pca_orth(qb, N, b);
  }
  // Rayleigh-Ritz: T = Q^T (Z^T Z Q), symmetrised
  rc = pca_apply(c, b, qb.data(), aq.data(), nullptr); if (rc) return rc;
  std::vector<double> t((size_t)b * b, 0.0), u;
  for (uint64_t g = 0; g < N; ++g)
    for (uint32_t i = 0; i < b; ++i)
      for (uint32_t j = 0; j < b; ++j) t[(size_t)i * b + j] += qb[g * b + i] * aq[g * b + j];
  for (uint32_t i = 0; i < b; ++i)
    for (uint32_t j = i + 1; j < b; ++j) t[(size_t)i * b + j] = t[(size_t)j * b + i] = 0.5 * (t[(size_t)i * b + j] + t[(size_t)j * b + i]);
  pca_jacobi(t, b, u);
  std::vector<uint32_t> order(b);
  for (uint32_t i = 0; i < b; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return t[(size_t)x * b + x] > t[(size_t)y * b + y]; });
  std::vector<double> v((size_t)N * k, 0.0), theta(k);
  for (uint32_t i = 0; i < k; ++i) {
    const uint32_t o = order[i];
    theta[i] = t[(size_t)o * b + o];
    eigenvalues[i] = theta[i] / (double)m;
    double best = -1.0;
    uint64_t arg = 0;
    for (uint64_t g = 0; g < N; ++g) {
      double s = 0.0;
      for (uint32_t j = 0; j < b; ++j) s += qb[g * b + j] * u[(size_t)j * b + o];
      v[g * k + i] = s;
      if (std::fabs(s) > best) { best = std::fabs(s); arg = g; }     // the lowest index wins a tie
    }
    if (v[arg * k + i] < 0.0)
      for (uint64_t g = 0; g < N; ++g) v[g * k + i] = -v[g * k + i];
  }
  std::copy(v.begin(), v.end(), scores);
  if (loadings) {                                    // u_i = Z v_i / sqrt(M lambda_i)
    rc = pca_apply(c, k, v.data(), nullptr, loadings); if (rc) return rc;
    for (uint32_t i = 0; i < k; ++i) {
      const double s = theta[i] > 0.0 ? std::sqrt((double)m * eigenvalues[i]) : 0.0;
      for (uint64_t l = 0; l < L; ++l) loadings[l * k + i] = s > 0.0 ? loadings[l * k + i] / s : 0.0;
    }
  }
  if (n_loci_used) *n_loci_used = m;
  return KGL_B200_OK;
}

}  // extern "C"
