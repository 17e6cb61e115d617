// ibs_plan_probe.cu -- the launch plan of pairwise IBS on the popcount kernel (plan_ibs, ibs_words_used and ibs_repair_segments,
// kgl_gene_b200/csrc/ibs_launch.cuh) as a host program, so that tests can check the plans without a GPU and GPU tests can pick
// shapes that reach a given plan.
//
// stdin : one request per line, "n_tiles n_loci sm_count n_dropped n_genomes [max_rows]" (max_rows: the most dropped rows of
//         one genome, 0 or absent when it does not matter)
// stdout: one JSON object with the field names and the kernels' constants, then for every request one JSON array holding the
//         request and, in the field order, what k_ibs_tiles and k_ibs_missing_fix run: words_used, the plan (words per chunk,
//         chunks, grid), the units (tile x chunk, counted in 64 bits) and the most one CTA runs, the 16-word stages of a chunk
//         and of the last chunk, the words of the last stage, the repair's segments, the most rows one repair thread walks
//         (ceil(max_rows / segs)) and the counter passes that walk takes (one more per kIbsFixRows rows).
#include "ibs_launch.cuh"

#include <cstdio>

using namespace kgl;

int main() {
  std::printf("{\"fields\": [\"n_tiles\", \"n_loci\", \"sm_count\", \"n_dropped\", \"n_genomes\", \"max_rows\", \"words_used\", "
              "\"words_per_chunk\", \"n_chunks\", \"grid\", \"units\", \"max_units_per_cta\", \"stages_per_chunk\", \"last_chunk_words\", "
              "\"last_chunk_stages\", \"last_stage_words\", \"segs\", \"walk_rows\", \"walk_passes\"], \"stage_words\": %d, \"ring\": %d, "
              "\"prefetch\": %d, \"flush_rows\": %u, \"max_tiles_per_launch\": %llu, \"tile\": %d}\n",
              kIbsKW, kIbsStages, kIbsPrefetch, kIbsFixRows, (unsigned long long)kIbsMaxTilesPerLaunch, kIbsT);
  char line[256];
  while (std::fgets(line, sizeof line, stdin)) {
    unsigned n_tiles = 0;
    int sm_count = 0;
    unsigned long long n_loci = 0, n_dropped = 0, n_genomes = 0, max_rows = 0;
    if (std::sscanf(line, "%u %llu %d %llu %llu %llu", &n_tiles, &n_loci, &sm_count, &n_dropped, &n_genomes, &max_rows) < 5) continue;
    const uint32_t words = ibs_words_used(n_loci);
    const IbsPlan p = plan_ibs(n_tiles, words, sm_count);
    const unsigned long long units = (unsigned long long)n_tiles * p.n_chunks;
    const unsigned long long per_cta = p.grid ? (units + p.grid - 1) / p.grid : 0;
    const long long last = (long long)words - (long long)(p.n_chunks - 1) * p.words_per_chunk;
    const long long last_stages = (last + kIbsKW - 1) / kIbsKW;
    const long long last_stage_words = last - (last_stages - 1) * kIbsKW;
    const uint32_t segs = ibs_repair_segments(n_dropped, n_genomes, n_tiles, sm_count);
    const unsigned long long walk = (max_rows + segs - 1) / segs;
    const unsigned long long passes = walk ? (walk + kIbsFixRows - 1) / kIbsFixRows : 1;
    std::printf("[%u, %llu, %d, %llu, %llu, %llu, %u, %u, %u, %u, %llu, %llu, %u, %lld, %lld, %lld, %u, %llu, %llu]\n", n_tiles, n_loci,
                sm_count, n_dropped, n_genomes, max_rows, words, p.words_per_chunk, p.n_chunks, p.grid, units, per_cta,
                p.words_per_chunk / kIbsKW, last, last_stages, last_stage_words, segs, walk, passes);
  }
  return 0;
}
