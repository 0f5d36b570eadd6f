// Rank-to-rank plumbing of one create_proof sharded over several GPUs (SURVEY.md 8(e)).
//
// The sharded prover (prover.cu) is SPMD: every rank runs the same host sequence on its own
// device with identical inputs, computes only its share of each phase (its columns, its lookups,
// its quotient cosets, its point range of the dense commits), and meets the other ranks at two
// kinds of exchange:
//   share           every listed device buffer is broadcast from the rank that produced it into
//                   each rank's own copy, ordered on the caller's stream (polynomials other ranks
//                   extend / open).  The ranks' buffers need not sit at the same addresses or
//                   arena offsets;
//   allgather_host  host memory of any size, the same size on every rank (commitments, partial MSM
//                   sums, permutation totals, evaluations) — what the Blake2b transcript absorbs,
//                   identically on every rank.
// Two implementations (comm.cu):
//   NcclComm   one process per GPU; grouped ncclBroadcast / ncclAllGather over NVLink / NVSwitch
//              (libnccl.so.2 is dlopen'ed on first use, so the library loads without NCCL);
//   LocalComm  the ranks are threads of one process (b200zk_group_*): peer-to-peer
//              cudaMemcpyAsync from the owner's own buffer with event hand-offs.  The ranks may
//              share one device, which is how the single-GPU test tier checks the sharded prover.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

struct b200zk_ctx;

namespace b200zk {

struct CommPiece {
    void* ptr;          // this rank's copy; every rank lists the same pieces, in the same order and of the same sizes
    size_t bytes;
    int owner;          // rank holding the valid copy
};

struct Comm {
    int rank = 0, world = 1;
    virtual ~Comm() {}
    virtual int32_t share(b200zk_ctx* ctx, const CommPiece* pieces, size_t count, cudaStream_t st) = 0;
    // `all` receives world * bytes, rank r's at r * bytes; synchronises `st` (results of earlier kernels are needed on
    // the host anyway)
    virtual int32_t allgather_host(b200zk_ctx* ctx, const void* mine, size_t bytes, void* all, cudaStream_t st) = 0;
    // a rank that fails outside an exchange releases the ranks waiting for it
    virtual void abort() = 0;
};

}  // namespace b200zk
