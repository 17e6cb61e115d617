// terms_plan_probe.cu -- the launch plans of the estimator sweeps (plan_fast and plan_terms, kgl_gene_b200/csrc/terms_launch.cuh)
// as a host program, so that tests can check the plans without a GPU and GPU tests can pick shapes that reach a given plan.
//
// stdin : one request per line, "mode gblocks n_words sel_row_lo sel_row_hi sm_count smem_limit" (mode: FAST_RITLAND 0,
//         FAST_HALL 1, FAST_NEWTON 2, FAST_LIMITS 3, FAST_NEWTON_U 4; sel_row_hi -1: no window, every tile)
// stdout: one JSON object with the field names and the kernels' constants, then for every request one JSON array holding the
//         request and, in the field order, the plan of k_terms_fast (ok, warps, CTAs per SM, slots, gy, tile window, tiles per
//         chunk, chunks, the tiles of the last chunk, shared memory) and the plan of k_genome_terms for the same genome blocks and
//         words (words per chunk, chunks, words of the last chunk, grid.x).
#include "terms_launch.cuh"

#include <cstdio>

using namespace kgl;

int main() {
  std::printf("{\"fields\": [\"mode\", \"gblocks\", \"n_words\", \"sel_row_lo\", \"sel_row_hi\", \"sm_count\", \"smem_limit\", \"ok\", "
              "\"warps\", \"ctas_per_sm\", \"slots\", \"gy\", \"tile_begin\", \"tile_end\", \"tiles_per_chunk\", \"n_chunks\", "
              "\"last_chunk_tiles\", \"smem\", \"term_words_per_chunk\", \"term_n_chunks\", \"term_last_chunk_words\", \"term_gx\"], "
              "\"tile_loci\": %d, \"tile_words\": %d, \"max_warps\": %d, \"max_pop\": %d, \"term_warps\": %d, \"term_tile_words\": %d}\n",
              kFastTile, kFastTileWords, kFastMaxWarps, kMaxPop, kTermWarps, kTermTileWords);
  char line[256];
  while (std::fgets(line, sizeof line, stdin)) {
    int mode = 0, sm_count = 0;
    unsigned long long gblocks = 0, n_words = 0, lo = 0, smem_limit = 0;
    long long hi = 0;
    if (std::sscanf(line, "%d %llu %llu %llu %lld %d %llu", &mode, &gblocks, &n_words, &lo, &hi, &sm_count, &smem_limit) < 7) continue;
    const FastPlan p = plan_fast(mode, gblocks, n_words, lo, hi < 0 ? ~0ull : (uint64_t)hi, sm_count, smem_limit);
    const long long last = p.ok ? (long long)(p.tile_end > p.tile_begin ? p.tile_end - p.tile_begin : 1) -
                                      (long long)((p.n_chunks - 1) * p.tiles_per_chunk) : 0;
    const TermLaunch t = plan_terms(gblocks, n_words, sm_count);
    std::printf("[%d, %llu, %llu, %llu, %lld, %d, %llu, %d, %d, %d, %u, %llu, %llu, %llu, %llu, %llu, %lld, %zu, %u, %llu, %lld, %u]\n",
                mode, gblocks, n_words, lo, hi, sm_count, smem_limit, p.ok ? 1 : 0, p.warps, p.ctas_per_sm, p.slots,
                (unsigned long long)p.gy, (unsigned long long)p.tile_begin, (unsigned long long)p.tile_end,
                (unsigned long long)p.tiles_per_chunk, (unsigned long long)p.n_chunks, last, p.smem, t.words_per_chunk,
                (unsigned long long)t.n_chunks, (long long)n_words - (long long)((t.n_chunks - 1) * t.words_per_chunk), t.grid.x);
  }
  return 0;
}
