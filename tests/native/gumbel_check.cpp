// TEST-ONLY host build of the Gumbel draw of csrc/rng.cuh (gumbel_draw), so that tests/test_host_gumbel.py can check its
// interval and moments without a GPU and tests/test_gpu_gumbel.py can compare the device's draws with it.
#include <stdint.h>
#include "../../caro-ai_b200/csrc/rng.cuh"
using namespace caro;

extern "C" {
double gc_gumbel(uint32_t seed_lo, uint32_t seed_hi, uint64_t uid, uint32_t search_index, uint32_t ply, uint32_t action) {
  return gumbel_draw(seed_lo, seed_hi, uid, search_index, ply, action);
}
// the uniform behind the draw, for the open-interval check
double gc_uniform(uint32_t seed_lo, uint32_t seed_hi, uint64_t uid, uint32_t search_index, uint32_t ply, uint32_t action) {
  return exp(-exp(-gumbel_draw(seed_lo, seed_hi, uid, search_index, ply, action)));
}
}
