// gram_plan_probe.cu -- the launch planner of the tensor-core Gram kernel (plan_gram, kgl_gene_b200/csrc/gram_launch.cuh) as a
// host program, so that tests can check its plans without a GPU and GPU tests can pick loci or tile counts that reach a given plan.
//
// stdin : one request per line, "n_tiles k_stages sm_count [chunk_stages_hint]" (k_stages = ceil(K / 128), the hint 0 or absent)
// stdout: one JSON object with the field names, then for every request one JSON array holding the request and
//         plan_gram(n_tiles, k_stages, sm_count, hint) in that field order, with what follows from it for k_gram_i8: the units
//         (tile x chunk, counted in 64 bits), the stages of the last chunk and the most units one CTA runs.
#include "gram_launch.cuh"

#include <cstdio>

using namespace kgl;

int main() {
  std::printf("{\"fields\": [\"n_tiles\", \"k_stages\", \"sm_count\", \"hint\", \"stages_per_chunk\", \"n_chunks\", \"grid\", "
              "\"units\", \"last_stages\", \"max_units_per_cta\"], \"ring\": %d, \"tile\": %d, \"stage_loci\": %d}\n",
              kGramStages, kGramM, kGramK);
  char line[256];
  while (std::fgets(line, sizeof line, stdin)) {
    unsigned n_tiles = 0, k_stages = 0, hint = 0;
    int sm_count = 0;
    if (std::sscanf(line, "%u %u %d %u", &n_tiles, &k_stages, &sm_count, &hint) < 3) continue;
    const GramPlan p = plan_gram(n_tiles, k_stages, sm_count, hint);
    const unsigned long long units = (unsigned long long)n_tiles * p.n_chunks;
    const long long last = (long long)k_stages - (long long)(p.n_chunks - 1) * p.stages_per_chunk;
    const unsigned long long per_cta = p.grid ? (units + p.grid - 1) / p.grid : 0;
    std::printf("[%u, %u, %d, %u, %u, %u, %u, %llu, %lld, %llu]\n", n_tiles, k_stages, sm_count, hint, p.stages_per_chunk, p.n_chunks,
                p.grid, units, last, per_cta);
  }
  return 0;
}
