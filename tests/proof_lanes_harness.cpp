// TEST AID for tests/test_proof_lanes.py: the lane planner of b200zk_create_proofs (proof_lanes.hpp) compiled with a host
// compiler.  Never linked into the product library.
#include "../halo2-experiments_b200/csrc/proof_lanes.hpp"

extern "C" {

uint32_t plan_lanes_c(uint32_t count, uint32_t want, const char* env, uint64_t free_bytes, uint64_t per_lane, uint32_t have) {
    return b200zk::plan_lanes(count, want, env, (size_t)free_bytes, (size_t)per_lane, have);
}
uint32_t lanes_default_cap() { return b200zk::LANES_DEFAULT_CAP; }
uint32_t lanes_max() { return b200zk::LANES_MAX; }

}  // extern "C"
