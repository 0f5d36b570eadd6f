// How many proofs of one proving key b200zk_create_proofs runs at once on the key's device.  Host code only, so that a
// CPU test can compile it (tests/proof_lanes_harness.cpp).
//
// A lane is the state one proof in flight needs: its arena and its ctx's workspaces.  Lane 0 is the proving key's own
// state and costs nothing extra; every further lane costs `per_lane` bytes of device memory.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstdlib>

namespace b200zk {

// Default number of lanes.  Small proofs are chains of dependent, latency-bound launches; a few proofs side by side fill
// the SMs between them, and more lanes than that only queue behind each other (DESIGN.md, "Several proofs of one key").
constexpr uint32_t LANES_DEFAULT_CAP = 4;
constexpr uint32_t LANES_MAX = 64;
// extra lanes may take at most this share of the device memory that is free when they are planned
constexpr size_t LANES_FREE_NUM = 1, LANES_FREE_DEN = 2;

// B200ZK_PROOF_LANES: a positive number replaces the caller's request and the default cap; anything else is ignored
inline uint32_t lanes_env(const char* v) {
    if (!v || !*v) return 0;
    char* end = nullptr;
    long x = strtol(v, &end, 10);
    return (*end == 0 && x > 0) ? (uint32_t)(x < (long)LANES_MAX ? x : LANES_MAX) : 0;
}

// count: proofs in the batch (0 = no batch, a reservation); want: the caller's request (0 = the default cap);
// env: B200ZK_PROOF_LANES; free_bytes: free device memory now; per_lane: bytes of one more lane; have: extra lanes that
// already exist (their memory is no longer free).  Result: >= 1, <= count (when count > 0), <= the request, and no more
// extra lanes than `have` plus what fits in the free-memory share.
inline uint32_t plan_lanes(uint32_t count, uint32_t want, const char* env, size_t free_bytes, size_t per_lane, uint32_t have) {
    uint32_t n = lanes_env(env);
    if (!n) n = want ? want : LANES_DEFAULT_CAP;
    if (n > LANES_MAX) n = LANES_MAX;
    if (count && n > count) n = count;
    const size_t budget = free_bytes / LANES_FREE_DEN * LANES_FREE_NUM;
    const size_t fit = (size_t)have + (per_lane ? budget / per_lane : (size_t)LANES_MAX);
    if ((size_t)n > 1 + fit) n = (uint32_t)(1 + fit);
    return n ? n : 1;
}

}  // namespace b200zk
