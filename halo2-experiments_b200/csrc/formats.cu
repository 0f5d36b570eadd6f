// On-disk / on-wire formats of the objects around the hot path (SURVEY.md 8(f3)):
//   ParamsKZG::write / read      halo2_proofs v2023_02_02 src/poly/kzg/commitment.rs — what a caller of
//                                `ParamsKZG::setup` (/root/reference/src/circuits/utils.rs:28) stores to reuse an SRS
//   VerifyingKey commitments     src/plonk.rs VerifyingKey::write / read (the commitments part)
//   G1Affine / G2Affine::to_bytes / from_bytes   halo2curves 0.3.1 src/derive/curve.rs
//   vk.transcript_repr           src/plonk.rs VerifyingKey::from_parts (see b200zk_vk_transcript_repr)
// The O(n) parts — compressing and decompressing the 2n SRS points (one Fq exponentiation per point to recover y) —
// run on the device; everything else is host code.
#include "context.hpp"
#include "cs_desc.hpp"
#include "pairing.hpp"
#include "transcript.hpp"
#include <new>
#include <vector>

using namespace b200zk;
using host::F2;
using host::HAffine;
using host::HFq;
using host::HFr;

namespace b200zk {

static constexpr uint32_t FMT_THREADS = 128;

// G1Affine::to_bytes: x (canonical, little-endian) with the parity of y in bit 7 of byte 31; identity = 32 zero bytes
__global__ void __launch_bounds__(FMT_THREADS) g1_compress_kernel(const affine_t* in, size_t n, uint32_t* out8) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    affine_t p = in[i];
    fe_t x = Fq::from_mont(p.x), y = Fq::from_mont(p.y);
    if (!(Fq::is_zero(p.x) && Fq::is_zero(p.y))) x.l[7] |= (y.l[0] & 1u) << 31;
#pragma unroll
    for (int j = 0; j < 8; ++j) out8[8 * i + j] = x.l[j];
}
// G1Affine::from_bytes (g1_decompress, curve.cuh); *bad is set for any invalid encoding
__global__ void __launch_bounds__(FMT_THREADS) g1_decompress_kernel(const uint32_t* in8, size_t n, affine_t* out, uint32_t* bad) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    affine_t r;
    if (!g1_decompress(in8 + 8 * i, &r)) atomicOr(bad, 1u);
    out[i] = r;
}

static unsigned fmt_blocks(size_t n) { return (unsigned)((n + FMT_THREADS - 1) / FMT_THREADS); }

static int32_t compress_points(b200zk_ctx* ctx, const affine_t* d_pts, size_t n, uint8_t* host_out) {
    ZK_TRY(ws_reserve(ctx, ctx->io_a, n * 32));
    g1_compress_kernel<<<fmt_blocks(n), FMT_THREADS, 0, ctx->stream>>>(d_pts, n, (uint32_t*)ctx->io_a.p);
    ctx->launches++;
    ZK_CUDA(ctx, cudaGetLastError());
    ZK_CUDA(ctx, cudaMemcpyAsync(host_out, ctx->io_a.p, n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}
static int32_t decompress_points(b200zk_ctx* ctx, const uint8_t* host_in, size_t n, affine_t* d_out) {
    ZK_TRY(ws_reserve(ctx, ctx->io_a, n * 32 + 256));
    uint32_t* d_bad = (uint32_t*)((char*)ctx->io_a.p + n * 32);
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_a.p, host_in, n * 32, cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(ctx, cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
    g1_decompress_kernel<<<fmt_blocks(n), FMT_THREADS, 0, ctx->stream>>>((const uint32_t*)ctx->io_a.p, n, d_out, d_bad);
    ctx->launches++;
    ZK_CUDA(ctx, cudaGetLastError());
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (*(const uint32_t*)ctx->pinned) return fail(ctx, B200ZK_EINVAL, "params_deserialize", "a point is not a canonical encoding of a curve point");
    return B200ZK_OK;
}

// ---- G2Affine::to_bytes / from_bytes (64 bytes: x.c0 || x.c1 little-endian, parity of y — of y.c0, or of y.c1 when
// y.c0 = 0 — in bit 7 of byte 63; identity = 64 zero bytes).  [M]: the flag convention is restated from memory of
// halo2curves 0.3.1 (rust-shim/README.md lists it among the first things to diff against real files).
static unsigned f2_parity(const F2& y) {
    uint64_t c[4];
    y.a.to_canonical(c);
    if ((c[0] | c[1] | c[2] | c[3]) == 0) y.b.to_canonical(c);
    return (unsigned)(c[0] & 1);
}
static void g2_compress(const host::G2A& p, uint8_t out[64]) {
    memset(out, 0, 64);
    if (host::g2_is_identity(p)) return;
    uint64_t c[4];
    p.x.a.to_canonical(c); memcpy(out, c, 32);
    p.x.b.to_canonical(c); memcpy(out + 32, c, 32);
    out[63] |= (uint8_t)(f2_parity(p.y) << 7);
}
// sqrt in Fq2 = Fq[u]/(u^2 + 1), q = 3 mod 4 (Adj & Rodriguez-Henriquez, algorithm 9)
static bool f2_sqrt(const F2& a, F2* out) {
    if (host::f2_is_zero(a)) { *out = a; return true; }
    static const uint64_t E1[4] = {0x4f082305b61f3f51ULL, 0x65e05aa45a1c72a3ULL, 0x6e14116da0605617ULL, 0x0c19139cb84c680aULL};   // (q - 3) / 4
    static const uint64_t E2[4] = {0x9e10460b6c3e7ea3ULL, 0xcbc0b548b438e546ULL, 0xdc2822db40c0ac2eULL, 0x183227397098d014ULL};   // (q - 1) / 2
    auto f2_pow = [](F2 b, const uint64_t e[4]) {
        F2 acc = host::f2_one();
        for (int i = 255; i >= 0; --i) { acc = host::f2_sqr(acc); if ((e[i >> 6] >> (i & 63)) & 1) acc = host::f2_mul(acc, b); }
        return acc;
    };
    F2 a1 = f2_pow(a, E1);
    F2 alpha = host::f2_mul(a1, host::f2_mul(a1, a));
    F2 a0 = host::f2_mul(F2{alpha.a, alpha.b.neg()}, alpha);       // alpha^q * alpha (the norm)
    F2 minus_one = host::f2_neg(host::f2_one());
    if (host::f2_eq(a0, minus_one)) return false;
    F2 x0 = host::f2_mul(a1, a);
    F2 x;
    if (host::f2_eq(alpha, minus_one)) x = F2{x0.b.neg(), x0.a};   // u * x0
    else x = host::f2_mul(f2_pow(host::f2_add(host::f2_one(), alpha), E2), x0);
    if (!host::f2_eq(host::f2_sqr(x), a)) return false;
    *out = x;
    return true;
}
static bool g2_decompress(const uint8_t in[64], host::G2A* out) {
    uint8_t t[64]; memcpy(t, in, 64);
    unsigned sign = t[63] >> 7;
    t[63] &= 0x7f;
    uint64_t c0[4], c1[4]; memcpy(c0, t, 32); memcpy(c1, t + 32, 32);
    if (HFq::ge_p(c0) || HFq::ge_p(c1)) return false;
    bool zero = true;
    for (int i = 0; i < 4; ++i) zero &= (c0[i] | c1[i]) == 0;
    if (zero) { if (sign) return false; *out = {host::f2_zero(), host::f2_zero()}; return true; }
    F2 x{HFq::from_canonical(c0), HFq::from_canonical(c1)};
    // twist: y^2 = x^3 + 3 / (9 + u)
    F2 b = host::f2_scale(host::f2_inv(F2{HFq::from_u64(9), HFq::one()}), HFq::from_u64(3));
    F2 rhs = host::f2_add(host::f2_mul(host::f2_sqr(x), x), b);
    F2 y;
    if (!f2_sqrt(rhs, &y)) return false;
    if (f2_parity(y) != sign) y = host::f2_neg(y);
    *out = {x, y};
    return true;
}

}  // namespace b200zk

extern "C" {

size_t b200zk_params_serialized_size(uint32_t k, int32_t with_lagrange) { return 4 + ((size_t)(with_lagrange ? 2 : 1) << k) * 32 + 128; }

// ParamsKZG::write: k (u32 LE) | n x G1 compressed (g) | n x G1 compressed (g_lagrange) | g2 | s_g2 (64 B compressed each)
int32_t b200zk_params_serialize(b200zk_params* p, const void* g2, const void* s_g2, uint8_t* out, size_t cap, size_t* len) {
    if (!p || !g2 || !s_g2 || !out) return B200ZK_EINVAL;
    b200zk_ctx* ctx = p->ctx;
    if (!p->d_g_lagrange) return fail(ctx, B200ZK_EINVAL, "params_serialize", "ParamsKZG::write needs g_lagrange");
    const size_t n = (size_t)1 << p->k, need = b200zk_params_serialized_size(p->k, 1);
    if (len) *len = need;
    if (cap < need) return fail(ctx, B200ZK_EINVAL, "params_serialize", "buffer too small");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    uint32_t k = p->k;
    memcpy(out, &k, 4);
    ZK_TRY(compress_points(ctx, p->d_g, n, out + 4));
    ZK_TRY(compress_points(ctx, p->d_g_lagrange, n, out + 4 + n * 32));
    g2_compress(host::g2_from_limbs(g2), out + 4 + 2 * n * 32);
    g2_compress(host::g2_from_limbs(s_g2), out + 4 + 2 * n * 32 + 64);
    return B200ZK_OK;
}

// ParamsKZG::read: the inverse; g2_out / s_g2_out receive the G2 elements (128-byte G2Affine, Montgomery limbs)
int32_t b200zk_params_deserialize(b200zk_ctx* ctx, const uint8_t* in, size_t len, b200zk_params** out, void* g2_out, void* s_g2_out) {
    if (!ctx || !in || !out || len < 4) return B200ZK_EINVAL;
    uint32_t k; memcpy(&k, in, 4);
    if (k > host::FR_TWO_ADICITY) return fail(ctx, B200ZK_EINVAL, "params_deserialize", "k out of range");
    const size_t n = (size_t)1 << k;
    if (len < b200zk_params_serialized_size(k, 1)) return fail(ctx, B200ZK_EINVAL, "params_deserialize", "truncated");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    host::G2A g2, s_g2;
    if (!g2_decompress(in + 4 + 2 * n * 32, &g2) || !g2_decompress(in + 4 + 2 * n * 32 + 64, &s_g2))
        return fail(ctx, B200ZK_EINVAL, "params_deserialize", "bad G2 element");
    b200zk_params* p = new (std::nothrow) b200zk_params();
    if (!p) return B200ZK_ENOMEM;
    p->ctx = ctx; p->k = k; p->d_g = nullptr; p->d_g_lagrange = nullptr; p->d_g_pre = nullptr; p->d_gl_pre = nullptr;
    int32_t rc = B200ZK_OK;
    if (cudaMalloc(&p->d_g, n * sizeof(affine_t)) != cudaSuccess || cudaMalloc(&p->d_g_lagrange, n * sizeof(affine_t)) != cudaSuccess) rc = fail(ctx, B200ZK_ENOMEM, "params_deserialize", "cudaMalloc");
    if (rc == B200ZK_OK) rc = decompress_points(ctx, in + 4, n, p->d_g);
    if (rc == B200ZK_OK) rc = decompress_points(ctx, in + 4 + n * 32, n, p->d_g_lagrange);
    if (rc == B200ZK_OK) rc = params_build_tables(p);
    if (rc != B200ZK_OK) { b200zk_params_destroy(p); return rc; }
    if (g2_out) host::g2_store(g2, g2_out);
    if (s_g2_out) host::g2_store(s_g2, s_g2_out);
    *out = p;
    return B200ZK_OK;
}

// G1Affine::to_bytes / from_bytes for a handful of points on the host (verifying-key commitments)
int32_t b200zk_g1_to_bytes(const void* affine_points, size_t count, uint8_t* out32) {
    if ((!affine_points || !out32) && count) return B200ZK_EINVAL;
    for (size_t i = 0; i < count; ++i) {
        const uint64_t* p = (const uint64_t*)affine_points + 8 * i;
        HFq x = HFq::from_limbs(p), y = HFq::from_limbs(p + 4);
        uint8_t* o = out32 + 32 * i;
        if (x.is_zero() && y.is_zero()) { memset(o, 0, 32); continue; }
        uint64_t xc[4], yc[4]; x.to_canonical(xc); y.to_canonical(yc);
        memcpy(o, xc, 32);
        o[31] |= (uint8_t)((yc[0] & 1) << 7);
    }
    return B200ZK_OK;
}
int32_t b200zk_g1_from_bytes(const uint8_t* in32, size_t count, void* affine_out) {
    if ((!in32 || !affine_out) && count) return B200ZK_EINVAL;
    for (size_t i = 0; i < count; ++i) {
        uint8_t t[32]; memcpy(t, in32 + 32 * i, 32);
        unsigned sign = t[31] >> 7;
        t[31] &= 0x7f;
        uint64_t xc[4]; memcpy(xc, t, 32);
        uint64_t* o = (uint64_t*)affine_out + 8 * i;
        if (HFq::ge_p(xc)) return B200ZK_EVERIFY;
        if ((xc[0] | xc[1] | xc[2] | xc[3]) == 0) { if (sign) return B200ZK_EVERIFY; memset(o, 0, 64); continue; }
        HFq x = HFq::from_canonical(xc), rhs = x.sqr() * x + HFq::from_u64(3);
        static const uint64_t E[4] = {0x4f082305b61f3f52ULL, 0x65e05aa45a1c72a3ULL, 0x6e14116da0605617ULL, 0x0c19139cb84c680aULL};   // (q + 1) / 4
        HFq y = rhs.pow(E);
        if (y.sqr() != rhs) return B200ZK_EVERIFY;
        uint64_t yc[4]; y.to_canonical(yc);
        if ((yc[0] & 1) != sign) y = y.neg();
        x.store(o); y.store(o + 4);
    }
    return B200ZK_OK;
}

// VerifyingKey::write (commitments part): fixed count (u32 BE) | fixed commitments | permutation commitments, 32 bytes each
size_t b200zk_vk_serialized_size(uint32_t num_fixed, uint32_t num_sigma) { return 4 + 32 * ((size_t)num_fixed + num_sigma); }
int32_t b200zk_vk_serialize(const void* fixed_commitments, uint32_t num_fixed, const void* sigma_commitments, uint32_t num_sigma, uint8_t* out, size_t cap) {
    if (!out || cap < b200zk_vk_serialized_size(num_fixed, num_sigma)) return B200ZK_EINVAL;
    out[0] = (uint8_t)(num_fixed >> 24); out[1] = (uint8_t)(num_fixed >> 16); out[2] = (uint8_t)(num_fixed >> 8); out[3] = (uint8_t)num_fixed;
    int32_t rc = b200zk_g1_to_bytes(fixed_commitments, num_fixed, out + 4);
    if (rc == B200ZK_OK) rc = b200zk_g1_to_bytes(sigma_commitments, num_sigma, out + 4 + 32 * (size_t)num_fixed);
    return rc;
}
int32_t b200zk_vk_deserialize(const uint8_t* in, size_t len, uint32_t num_sigma, void* fixed_out, uint32_t fixed_cap, uint32_t* num_fixed, void* sigma_out) {
    if (!in || len < 4 || !num_fixed) return B200ZK_EINVAL;
    uint32_t f = ((uint32_t)in[0] << 24) | ((uint32_t)in[1] << 16) | ((uint32_t)in[2] << 8) | in[3];
    *num_fixed = f;
    if (f > fixed_cap || len < b200zk_vk_serialized_size(f, num_sigma)) return B200ZK_EINVAL;
    int32_t rc = b200zk_g1_from_bytes(in + 4, f, fixed_out);
    if (rc == B200ZK_OK) rc = b200zk_g1_from_bytes(in + 4 + 32 * (size_t)f, num_sigma, sigma_out);
    return rc;
}

// vk.transcript_repr.  Upstream (VerifyingKey::from_parts) hashes Rust's `{:?}` rendering of the pinned verifying key:
//   Blake2b-512(personal "Halo2-Verify-Key") over (len as u64 LE) || format!("{:?}", vk.pinned()),  then from_bytes_wide.
// A Debug string cannot be restated outside Rust, so create_proof / verify_proof take the value as an input (the shim
// passes upstream's).  For hosts without Rust this derives a value with the same role from the same content in a
// canonical binary form: the same hash and personalisation over (len as u64 LE) || cs blob words (LE; they carry k, the
// column counts, the query lists, the gates, the lookups and the permutation columns) || fixed commitments || permutation
// commitments (x, y canonical LE, 64 bytes each).  Binding the key into the transcript is what matters for soundness;
// the value differs from upstream's, so such proofs verify with this library's verifier, not with stock halo2.
int32_t b200zk_vk_transcript_repr(const uint32_t* cs_blob, size_t blob_words, const void* fixed_commitments,
                                  const void* sigma_commitments, void* out_fr) {
    CsDesc cs;
    if (!cs_blob || !out_fr || !parse_cs(cs_blob, blob_words, cs)) return B200ZK_EINVAL;
    const size_t F = cs.F, P = cs.perm.size();
    if ((F && !fixed_commitments) || (P && !sigma_commitments)) return B200ZK_EINVAL;
    host::Blake2b h("Halo2-Verify-Key");
    const uint64_t len = 4 * (uint64_t)blob_words + 64 * (uint64_t)(F + P);
    h.update(&len, 8);
    h.update(cs_blob, 4 * blob_words);
    auto absorb = [&](const void* pts, size_t count) {
        for (size_t i = 0; i < count; ++i) {
            const uint64_t* p = (const uint64_t*)pts + 8 * i;
            uint64_t c[4];
            HFq::from_limbs(p).to_canonical(c); h.update(c, 32);
            HFq::from_limbs(p + 4).to_canonical(c); h.update(c, 32);
        }
    };
    absorb(fixed_commitments, F);
    absorb(sigma_commitments, P);
    uint8_t d[64];
    h.finalize_clone(d);
    uint64_t w[8]; memcpy(w, d, 64);
    HFr::from_u512(w).store(out_fr);
    return B200ZK_OK;
}

}  // extern "C"
