// Many proofs of one verifying key, checked with one pairing: halo2_proofs v2023_02_02 AccumulatorStrategy
// (src/poly/kzg/strategy.rs) over VerifierSHPLONK / Blake2bRead / Challenge255 (b200zk_verify_proofs, include/b200zk.h).
//
// Stage 1, per proof: every point of every proof is decompressed on the device in one launch (g1_decompress, the body
// G1Affine::from_bytes uses in formats.cu); the transcripts are replayed on a pool of host threads (replay_proof,
// verifier.cu), each giving the proof's opening (h2, right) as linear terms over proof points, vk commitments and G.
// Stage 2: the scalars of proof i are multiplied by c_i = prod_{j > i} r_j on the host; one launch computes every term
// c_i s * B (one thread per term, xyzz_mul), one launch sums each proof's terms (one warp per segment), so every proof
// ends with its own pair c_i (left_i, right_i).  The accumulator is the host sum of the pairs; one host pairing checks it
// (a lone device check is no faster: DESIGN.md §6.5).  If it fails, one device call (pairing_checks_run, pairing.cu)
// checks every pair on its own, so each proof's status is its own verdict and the launches do not depend on how many
// proofs fail.
#include "context.hpp"
#include "g1_ntt.cuh"
#include "pairing.hpp"
#include "verify_replay.hpp"
#include <atomic>
#include <string>
#include <thread>
#include <vector>

using namespace b200zk;
using namespace b200zk::host;

namespace b200zk {

static constexpr uint32_t VB_THREADS = 128;

// thread t: point t % npts of proof slot t / npts; slot s starts at word s * stride_words, point j at word point_word[j]
__global__ void __launch_bounds__(VB_THREADS) vb_decompress_kernel(const uint32_t* words, size_t stride_words, const uint32_t* point_word,
                                                                   uint32_t npts, size_t total, affine_t* out, uint32_t* bad) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const size_t slot = t / npts;
    affine_t r;
    if (!g1_decompress(words + slot * stride_words + point_word[t % npts], &r)) bad[slot] = 1u;
    out[t] = r;
}

// out[t] = scalars[t] * bases[base_idx[t]]  (scalars canonical, non-zero; bases not the identity)
__global__ void __launch_bounds__(VB_THREADS) vb_term_kernel(const affine_t* bases, const uint32_t* base_idx, const fe_t* scalars, size_t n,
                                                             xyzz_t* out) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    out[t] = xyzz_mul(xyzz_from_affine(bases[base_idx[t]]), scalars[t]);
}

ZK_D xyzz_t xyzz_shfl_down(const xyzz_t& p, int d) {
    xyzz_t r;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        r.x.l[j] = __shfl_down_sync(0xffffffffu, p.x.l[j], d);
        r.y.l[j] = __shfl_down_sync(0xffffffffu, p.y.l[j], d);
        r.zz.l[j] = __shfl_down_sync(0xffffffffu, p.zz.l[j], d);
        r.zzz.l[j] = __shfl_down_sync(0xffffffffu, p.zzz.l[j], d);
    }
    return r;
}

// one warp per segment [seg[s], seg[s + 1]) of terms: strided sums per lane, then a shuffle tree
__global__ void __launch_bounds__(VB_THREADS) vb_segment_sum_kernel(const xyzz_t* terms, const uint32_t* seg, uint32_t nseg, xyzz_t* out) {
    const size_t s = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / 32;
    const uint32_t lane = threadIdx.x & 31;
    if (s >= nseg) return;                                       // whole warps
    xyzz_t acc = xyzz_identity();
    for (uint32_t i = seg[s] + lane; i < seg[s + 1]; i += 32) xyzz_add(acc, terms[i]);
    for (int d = 16; d > 0; d >>= 1) {
        xyzz_t o = xyzz_shfl_down(acc, d);
        xyzz_add(acc, o);
    }
    if (lane == 0) out[s] = acc;
}

}  // namespace b200zk

namespace {

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
unsigned blocks_for(size_t threads) { return (unsigned)((threads + VB_THREADS - 1) / VB_THREADS); }

struct Pair { HXyzz left, right; };

constexpr uint32_t PAIR_SKIP = 0xffffffffu;                    // PC_SKIP of pairing.cuh

// e(left_j, [s]_2) * e(-right_j, [1]_2) == 1 for every pair, on the device; an identity point contributes 1
int32_t pairs_check(b200zk_ctx* ctx, const std::vector<Pair>& pairs, const void* s_g2, const void* g2, int32_t* status) {
    const size_t n = pairs.size();
    std::vector<HAffine> aff(2 * n);
    hx_batch_to_affine(&pairs[0].left, 2 * n, aff.data());
    std::vector<uint32_t> q(2 * n);
    for (size_t j = 0; j < n; ++j) {
        aff[2 * j + 1].y = aff[2 * j + 1].y.neg();
        for (int h = 0; h < 2; ++h) q[2 * j + h] = aff[2 * j + h].x.is_zero() && aff[2 * j + h].y.is_zero() ? PAIR_SKIP : h;
    }
    uint8_t qs[256];
    memcpy(qs, s_g2, 128);
    memcpy(qs + 128, g2, 128);
    return pairing_checks_run(ctx, aff.data(), q.data(), qs, 2, 2, (uint32_t)n, status);
}

void store_affine(const HAffine& a, void* out) { a.x.store(out); a.y.store((uint8_t*)out + 32); }

}  // namespace

extern "C" int32_t b200zk_verify_proofs(b200zk_ctx* ctx, const uint32_t* cs_blob, size_t blob_words, const void* fixed_commitments,
                                        const void* sigma_commitments, const void* g1_generator, const void* g2, const void* s_g2,
                                        uint32_t count, const void* const* instance_columns, const uint32_t* instance_lens,
                                        const void* transcript_repr, const uint8_t* const* proofs, const size_t* proof_lens,
                                        const void* rng_wide, int32_t* status, void* accumulator_out) {
    if (!ctx) return B200ZK_EINVAL;
    auto bad_arg = [&](const std::string& why) { return fail(ctx, B200ZK_EINVAL, "verify_proofs", why.c_str()); };
    CsDesc cs;
    if (!cs_blob || !parse_cs(cs_blob, blob_words, cs)) return bad_arg("the constraint-system blob does not parse");
    if (!g1_generator || !g2 || !s_g2 || !transcript_repr || !proofs || !proof_lens || !rng_wide || !status) return bad_arg("null argument");
    if (count == 0) return bad_arg("count == 0");
    if ((cs.F && !fixed_commitments) || (!cs.perm.empty() && !sigma_commitments)) return bad_arg("missing verifying-key commitments");
    if (cs.I && (!instance_columns || !instance_lens)) return bad_arg("missing instance columns");
    if (cs.k < 1 || cs.k > FR_TWO_ADICITY) return bad_arg("k out of range");
    for (uint32_t i = 0; i < count; ++i) {
        if (!proofs[i] && proof_lens[i]) return bad_arg("proof " + std::to_string(i) + " is NULL with a nonzero length");
        for (uint32_t c = 0; c < cs.I; ++c)
            if (instance_lens[(size_t)i * cs.I + c] && !instance_columns[(size_t)i * cs.I + c])
                return bad_arg("instance column " + std::to_string(c) + " of proof " + std::to_string(i) + " is NULL");
    }
    const G2A qs[2] = {g2_from_limbs(s_g2), g2_from_limbs(g2)};
    if (!g2_on_curve(qs[0]) || !g2_on_curve(qs[1]) || g2_is_identity(qs[0]) || g2_is_identity(qs[1])) return bad_arg("bad G2 point");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));

    // ---- stage 1a: every complete proof gets a slot, and its points are decompressed on the device
    const VkPoints vk = {fixed_commitments, sigma_commitments, g1_generator};
    std::vector<size_t> offs;
    const size_t plen = proof_point_offsets(cs, &offs);
    const uint32_t npts = (uint32_t)offs.size();
    const size_t F = cs.F, P = cs.perm.size(), nvk = F + P + 1;
    std::vector<uint32_t> proof_of;                                   // slot -> proof
    for (uint32_t i = 0; i < count; ++i) {
        status[i] = proof_lens[i] < plen ? B200ZK_EVERIFY : B200ZK_OK;
        if (status[i] == B200ZK_OK) proof_of.push_back(i);
    }
    const size_t nslot = proof_of.size();
    // the device's base table: F fixed commitments, P permutation commitments, G, then npts points per slot; a mirror here
    std::vector<HAffine> bases(nvk + nslot * npts);
    for (size_t j = 0; j < F; ++j) bases[j] = open_base_point(vk, nullptr, {OpenBase::FIXED, (uint32_t)j});
    for (size_t j = 0; j < P; ++j) bases[F + j] = open_base_point(vk, nullptr, {OpenBase::SIGMA, (uint32_t)j});
    bases[F + P] = open_base_point(vk, nullptr, {OpenBase::GEN, 0});
    std::vector<uint32_t> bad(nslot, 0);
    ZK_TRY(ws_reserve(ctx, ctx->io_b, bases.size() * sizeof(affine_t)));
    affine_t* d_bases = (affine_t*)ctx->io_b.p;
    ZK_CUDA(ctx, cudaMemcpyAsync(d_bases, bases.data(), nvk * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream));
    std::vector<uint8_t> bytes(nslot * plen);
    if (nslot) {
        std::vector<uint32_t> point_word(npts);
        for (uint32_t j = 0; j < npts; ++j) point_word[j] = (uint32_t)(offs[j] / 4);
        for (size_t s = 0; s < nslot; ++s) memcpy(&bytes[s * plen], proofs[proof_of[s]], plen);
        const size_t o_words = align256(bytes.size()), o_bad = o_words + align256(npts * 4);
        ZK_TRY(ws_reserve(ctx, ctx->io_a, o_bad + nslot * 4));
        char* a = (char*)ctx->io_a.p;
        ZK_CUDA(ctx, cudaMemcpyAsync(a, bytes.data(), bytes.size(), cudaMemcpyHostToDevice, ctx->stream));
        ZK_CUDA(ctx, cudaMemcpyAsync(a + o_words, point_word.data(), npts * 4, cudaMemcpyHostToDevice, ctx->stream));
        ZK_CUDA(ctx, cudaMemsetAsync(a + o_bad, 0, nslot * 4, ctx->stream));
        vb_decompress_kernel<<<blocks_for(nslot * npts), VB_THREADS, 0, ctx->stream>>>(
            (const uint32_t*)a, plen / 4, (const uint32_t*)(a + o_words), npts, nslot * npts, d_bases + nvk, (uint32_t*)(a + o_bad));
        ctx->launches++;
        ZK_CUDA(ctx, cudaGetLastError());
        ZK_CUDA(ctx, cudaMemcpyAsync(&bases[nvk], d_bases + nvk, nslot * npts * sizeof(affine_t), cudaMemcpyDeviceToHost, ctx->stream));
        ZK_CUDA(ctx, cudaMemcpyAsync(bad.data(), a + o_bad, nslot * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));

    // ---- stage 1b: transcript replays, one proof per task on a pool of host threads
    std::vector<Opening> ops(nslot);
    std::vector<int32_t> rcs(nslot, B200ZK_OK);
    std::atomic<size_t> next{0};
    auto work = [&]() {
        for (size_t s; (s = next++) < nslot;) {
            const size_t i = proof_of[s];
            if (bad[s]) { rcs[s] = B200ZK_EVERIFY; continue; }
            rcs[s] = replay_proof(cs, vk, cs.I ? instance_columns + i * cs.I : nullptr, cs.I ? instance_lens + i * cs.I : nullptr,
                                  transcript_repr, proofs[i], proof_lens[i], &bases[nvk + s * npts], &ops[s]);
        }
    };
    {
        const size_t want = std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), nslot);
        std::vector<std::thread> pool;
        for (size_t t = 1; t < want; ++t) {
            try { pool.emplace_back(work); } catch (...) { break; }       // fewer threads is not an error
        }
        work();
        for (auto& th : pool) th.join();
    }
    for (size_t s = 0; s < nslot; ++s) {
        if (rcs[s] == B200ZK_EINVAL) return fail(ctx, B200ZK_EINVAL, "verify_proofs", "the constraint system's expressions do not evaluate");
        if (rcs[s] != B200ZK_OK) status[proof_of[s]] = B200ZK_EVERIFY;
    }

    // ---- stage 2a: c_i = prod_{j > i} r_j folded into the scalars; one segment per half of each surviving proof's pair
    std::vector<HFr> c(count);
    c[count - 1] = HFr::one();
    for (uint32_t i = count - 1; i > 0; --i) {
        uint64_t w[8];
        memcpy(w, (const uint8_t*)rng_wide + 64 * (size_t)i, 64);
        c[i - 1] = c[i] * HFr::from_u512(w);
    }
    std::vector<uint32_t> base_idx, seg, surv;
    std::vector<fe_t> scalars;
    for (size_t s = 0; s < nslot; ++s) {
        if (rcs[s] != B200ZK_OK) continue;
        const HFr& ci = c[proof_of[s]];
        const size_t first = nvk + s * npts;
        auto index = [&](const OpenBase& b) -> uint32_t {
            return b.kind == OpenBase::PROOF ? (uint32_t)(first + b.idx) : b.kind == OpenBase::FIXED ? b.idx : b.kind == OpenBase::SIGMA ? (uint32_t)(F + b.idx) : (uint32_t)(F + P);
        };
        auto emit = [&](uint32_t b, const HFr& sc) {
            if (sc.is_zero() || (bases[b].x.is_zero() && bases[b].y.is_zero())) return;
            fe_t f;
            uint64_t canon[4];
            sc.to_canonical(canon);
            memcpy(f.l, canon, 32);
            base_idx.push_back(b);
            scalars.push_back(f);
        };
        surv.push_back(proof_of[s]);
        seg.push_back((uint32_t)base_idx.size());
        emit((uint32_t)(first + ops[s].h2), ci);
        seg.push_back((uint32_t)base_idx.size());
        for (const OpenTerm& t : ops[s].right) emit(index(t.base), ci * t.scalar);
    }
    seg.push_back((uint32_t)base_idx.size());
    const size_t nterms = base_idx.size(), nseg = 2 * surv.size();

    // ---- stage 2b: every term on the device, one pair per proof
    std::vector<Pair> pairs(surv.size(), Pair{hx_identity(), hx_identity()});
    if (nterms) {
        const size_t o_sc = align256(nterms * 4), o_seg = o_sc + align256(nterms * sizeof(fe_t));
        ZK_TRY(ws_reserve(ctx, ctx->io_a, o_seg + (nseg + 1) * 4));
        ZK_TRY(ws_reserve(ctx, ctx->setup_ws, (nterms + nseg) * sizeof(xyzz_t)));
        char* a = (char*)ctx->io_a.p;
        xyzz_t* d_terms = (xyzz_t*)ctx->setup_ws.p;
        ZK_CUDA(ctx, cudaMemcpyAsync(a, base_idx.data(), nterms * 4, cudaMemcpyHostToDevice, ctx->stream));
        ZK_CUDA(ctx, cudaMemcpyAsync(a + o_sc, scalars.data(), nterms * sizeof(fe_t), cudaMemcpyHostToDevice, ctx->stream));
        ZK_CUDA(ctx, cudaMemcpyAsync(a + o_seg, seg.data(), (nseg + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
        vb_term_kernel<<<blocks_for(nterms), VB_THREADS, 0, ctx->stream>>>(d_bases, (const uint32_t*)a, (const fe_t*)(a + o_sc), nterms, d_terms);
        ctx->launches++;
        ZK_CUDA(ctx, cudaGetLastError());
        vb_segment_sum_kernel<<<blocks_for(nseg * 32), VB_THREADS, 0, ctx->stream>>>(d_terms, (const uint32_t*)(a + o_seg), (uint32_t)nseg,
                                                                                      d_terms + nterms);
        ctx->launches++;
        ZK_CUDA(ctx, cudaGetLastError());
        static_assert(sizeof(Pair) == 2 * sizeof(xyzz_t), "a pair is two device XYZZ points");
        ZK_CUDA(ctx, cudaMemcpyAsync(pairs.data(), d_terms + nterms, nseg * sizeof(xyzz_t), cudaMemcpyDeviceToHost, ctx->stream));
        ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }

    // ---- stage 2c: the accumulator and its pairing check; when it fails, every pair's own check on the device
    HXyzz l = hx_identity(), r = hx_identity();
    for (const Pair& p : pairs) { l = hx_add(l, p.left); r = hx_add(r, p.right); }
    const HAffine la = hx_to_affine(l), ra = hx_to_affine(r);
    if (accumulator_out) {
        store_affine(la, accumulator_out);
        store_affine(ra, (uint8_t*)accumulator_out + 64);
    }
    const HAffine acc[2] = {la, {ra.x, ra.y.neg()}};
    if (!pairs.empty() && !pairing_product_is_one(acc, qs, 2)) {
        std::vector<int32_t> own(pairs.size());
        ZK_TRY(pairs_check(ctx, pairs, s_g2, g2, own.data()));
        for (size_t j = 0; j < pairs.size(); ++j) if (own[j] != B200ZK_OK) status[surv[j]] = B200ZK_EVERIFY;
    }
    for (uint32_t i = 0; i < count; ++i) if (status[i] != B200ZK_OK) return B200ZK_EVERIFY;
    return B200ZK_OK;
}
