// stream_plan_probe.cu -- the launch planner of the streaming pass (kgl_gene_b200/csrc/stream_common.cuh) as a host program,
// so that tests can check its plans without a GPU and GPU tests can pick loci that reach a given plan.
//
// stdin : whitespace-separated triples "units n_loci sm_count" (units = 128-bit units of a host row, ceil(genomes / 64))
// stdout: one JSON object with the field names and the counter constants, then for every triple one JSON array holding
//         plan_stream(stream_units_padded(units), n_loci, sm_count) in that field order -- the plan the C ABI launches.
#include "stream_common.cuh"

#include <cstdio>

using namespace kgl;

int main() {
  std::printf("{\"fields\": [\"units\", \"n_loci\", \"sm_count\", \"units_padded\", \"shape\", \"slice_units\", \"slices\", "
              "\"rows_per_stage\", \"h_parts\", \"h_units\", \"v_row_lanes\", \"n_stages\", \"threads\", \"total_stages\", "
              "\"stages_per_cta\", \"n_ctas\", \"flush_stages\", \"chunks_per_cta\", \"padded_rows\", \"smem\"], "
              "\"levels\": %d, \"max_calls\": %d, \"consumer_threads\": %d, \"max_stages\": %d, \"max_slice_units\": %d}\n",
              kScLevels, kScMaxCalls, kScConsumerThreads, kScMaxStages, kScMaxSliceUnits);
  unsigned long long units = 0, n_loci = 0;
  int sm_count = 0;
  while (std::scanf("%llu %llu %d", &units, &n_loci, &sm_count) == 3) {
    const StreamPlan p = plan_stream(stream_units_padded(units), n_loci, sm_count);
    std::printf("[%llu, %llu, %d, %u, %d, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %llu, %zu]\n", units, n_loci, sm_count,
                p.units_padded, p.shape, p.slice_units, p.slices, p.rows_per_stage, p.h_parts, p.h_units, p.v_row_lanes, p.n_stages,
                p.threads, p.total_stages, p.stages_per_cta, p.n_ctas, p.flush_stages, p.chunks_per_cta,
                (unsigned long long)p.padded_rows, p.smem);
  }
  return 0;
}
