// ld_band_probe.cu -- the band tile list of the LD entry points (ld_band, kgl_gene_b200/csrc/ld.cuh) as a host program, so that
// tests can check it without a GPU.
//
// stdin : one case: "n_loci window_loci window_bp code3 budget_bytes", then n_loci ranks (kLdNotEligible = 4294967295 for an
//         ineligible locus), then n_loci offsets
// stdout: {"tiles": [[I, J], ...], "slab_begin": [...], "tile_blocks": [1 | 4 | 6 per tile], "block_bytes": 262144}
#include "ld.cuh"

#include <cstdio>
#include <vector>

using namespace kgl;

int main() {
  unsigned long long n_loci = 0, budget = 0;
  unsigned window_loci = 0, window_bp = 0, code3 = 0;
  if (std::scanf("%llu %u %u %u %llu", &n_loci, &window_loci, &window_bp, &code3, &budget) != 5) return 1;
  std::vector<uint32_t> rank(n_loci), offsets(n_loci);
  for (auto& r : rank) if (std::scanf("%u", &r) != 1) return 1;
  for (auto& o : offsets) if (std::scanf("%u", &o) != 1) return 1;
  const LdBand band = ld_band(rank.data(), offsets.data(), n_loci, window_loci, window_bp, code3 != 0, budget);
  std::printf("{\"tiles\": [");
  for (size_t t = 0; t < band.tiles.size(); ++t) std::printf("%s[%u, %u]", t ? ", " : "", band.tiles[t].x, band.tiles[t].y);
  std::printf("], \"slab_begin\": [");
  for (size_t s = 0; s < band.slab_begin.size(); ++s) std::printf("%s%u", s ? ", " : "", band.slab_begin[s]);
  std::printf("], \"tile_blocks\": [");
  for (size_t t = 0; t < band.tiles.size(); ++t)
    std::printf("%s%llu", t ? ", " : "", (unsigned long long)ld_tile_blocks(code3 != 0, band.tiles[t].x == band.tiles[t].y));
  std::printf("], \"block_bytes\": %llu}\n", (unsigned long long)kLdBlockBytes);
  return 0;
}
