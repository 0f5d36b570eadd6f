// The transcript replay of plonk::verify_proof + VerifierSHPLONK (verifier.cu), shared by b200zk_verify_proof and
// b200zk_verify_proofs (verify_batch.cu).  It returns the proof's opening as linear terms instead of group elements:
// VerifierSHPLONK's DualMSM (left, right) = (h2, u h2 + L / z_0), with every G1 operation verify_proof used to fold
// (the h pieces in x^n, the v / y weights, the [r(u)] G terms, Z_T(u) h1, the division by z_0) moved into the scalars.
// The single verifier evaluates the terms on the host; the batch evaluates them on the device.
#pragma once
#include <vector>
#include "cs_desc.hpp"
#include "host_field.hpp"

namespace b200zk {

// the verifying key and SRS points the verifier reads (host, 64-byte G1Affine Montgomery limbs)
struct VkPoints { const void* fixed; const void* sigma; const void* g1; };

// a base of the opening: a point of the proof (its index in read order), a fixed or permutation commitment, or G
struct OpenBase {
    enum Kind : uint32_t { PROOF, FIXED, SIGMA, GEN } kind;
    uint32_t idx;
};
struct OpenTerm { OpenBase base; host::HFr scalar; };
struct Opening {
    std::vector<host::HAffine> points;     // the proof's points in read order
    uint32_t h2 = 0;                       // left = points[h2]
    std::vector<OpenTerm> right;           // right = sum scalar * base
};

// the point a base stands for; proof_points = Opening::points
host::HAffine open_base_point(const VkPoints& vk, const host::HAffine* proof_points, const OpenBase& b);

// Byte offsets of a proof's points in read order (the commitments, then h1 and h2 after the evaluations) and the
// length of a complete proof.  Both are fixed by the constraint system.
size_t proof_point_offsets(const CsDesc& cs, std::vector<size_t>* offs);

// Replays one proof.  points: null = decompress the points from the proof bytes; otherwise the proof's points already
// decompressed, in read order (the caller has rejected proofs with an invalid encoding or shorter than
// proof_point_offsets' length).  B200ZK_OK with *out filled, B200ZK_EVERIFY for every stage-1 Err of upstream's verifier
// (malformed proof, instance too large, x^n = 1, z_0 = 0), B200ZK_EINVAL for an instance column that is missing or a
// constraint system whose expressions do not evaluate.  cs.k must be in 1 ..= FR_TWO_ADICITY.
int32_t replay_proof(const CsDesc& cs, const VkPoints& vk, const void* const* instance_columns, const uint32_t* instance_lens,
                     const void* transcript_repr, const uint8_t* proof, size_t proof_len, const host::HAffine* points, Opening* out);

}  // namespace b200zk
