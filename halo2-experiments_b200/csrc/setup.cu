// ParamsKZG::<Bn256>::setup on the device (halo2_proofs v2023_02_02
// src/poly/kzg/commitment.rs; called at /root/reference/src/circuits/utils.rs:28):
//   g[i]          = [s^i] G
//   g_lagrange[i] = [ (s^n - 1)/n * w^i / (s - w^i) ] G
// 2n fixed-base scalar multiplications.  The generator table holds d * 256^w * G for
// w < 32, d < 256 (8160 affine points, 510 KiB, L1/L2 resident), so each point costs at most
// 32 mixed additions; results are normalised to affine with one batched Fq inversion.
// The same normalisation finishes arithmetic::g_to_lagrange (ParamsKZG::downsize), a G1 NTT (g1_ntt.cuh).
#include "context.hpp"
#include "poly.cuh"
#include "g1_ntt.cuh"

namespace b200zk {

static constexpr uint32_t SETUP_THREADS = 128;

// scalar i of the coefficient basis: s^i = lo[i & mask] * hi[i >> bits]
__global__ void __launch_bounds__(SETUP_THREADS) setup_powers_kernel(fe_t* out, size_t n, const fe_t* lo, const fe_t* hi, uint32_t bits) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe_t a = lo[i & ((1u << bits) - 1)], b = hi[i >> bits];
    out[i] = Fr::mul(a, b);
}
// den[i] = s - w^i   (w^i in `pw`)
__global__ void __launch_bounds__(SETUP_THREADS) setup_lagrange_den_kernel(fe_t* den, const fe_t* pw, size_t n, const fe_t s) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe_t w = pw[i];
    den[i] = Fr::sub(s, w);
}
// sc[i] = multiplier * w^i * den_inv[i]   (in place over pw)
__global__ void __launch_bounds__(SETUP_THREADS) setup_lagrange_scalar_kernel(fe_t* pw, const fe_t* den_inv, size_t n, const fe_t multiplier) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe_t w = pw[i], d = den_inv[i];
    pw[i] = Fr::mul(Fr::mul(multiplier, w), d);
}
__global__ void __launch_bounds__(SETUP_THREADS) setup_pow_table_kernel(fe_t* out, const fe_t base, uint32_t count, uint32_t shift) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = Fr::pow_u64(base, (unsigned long long)i << shift);
}

// out[i] = [sc[i]] G as XYZZ; zzz copied to a dense array for the batched inversion
__global__ void __launch_bounds__(SETUP_THREADS) setup_fixed_base_kernel(const fe_t* sc, size_t n, const affine_t* table, xyzz_t* out, fe_t* zzz) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe_t s = sc[i];
    s = Fr::from_mont(s);
    xyzz_t acc = xyzz_identity();
    for (uint32_t w = 0; w < 32; ++w) {
        uint32_t d = (s.l[w >> 2] >> ((w & 3) * 8)) & 0xff;
        if (d) { affine_t p = table[w * 255 + d - 1]; xyzz_madd(acc, p, false); }
    }
    out[i] = acc;
    zzz[i] = acc.zzz;
}
// x = X * ZZ^2 * iz^2, y = Y * iz  with iz = 1/ZZZ  (ZZ^3 = ZZZ^2); identity -> (0,0)
__global__ void __launch_bounds__(SETUP_THREADS) setup_normalize_kernel(const xyzz_t* in, const fe_t* zzz_inv, size_t n, affine_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    xyzz_t p = in[i];
    fe_t iz = zzz_inv[i];
    affine_t r;
    if (Fq::is_zero(p.zz)) { r.x = Fq::zero(); r.y = Fq::zero(); }
    else {
        fe_t t = Fq::mul(p.zz, iz);                     // 1/Z
        r.x = Fq::mul(p.x, Fq::sqr(t));
        r.y = Fq::mul(p.y, iz);
    }
    out[i] = r;
}

static fe_t to_dev(const host::HFr& x) { fe_t r; memcpy(r.l, x.v, 32); return r; }
static unsigned nblocks(size_t work, unsigned threads) { return (unsigned)((work + threads - 1) / threads); }

static int32_t ensure_gen_table(b200zk_ctx* ctx) {
    if (ctx->d_gen_table) return B200ZK_OK;
    using namespace host;
    // host: 32 chains of 255 additions, then one batched normalisation
    std::vector<HXyzz> pts(32 * 255);
    HXyzz base = hx_from_affine({HFq::from_u64(1), HFq::from_u64(2)});
    for (int w = 0; w < 32; ++w) {
        HXyzz cur = base;
        for (int d = 1; d <= 255; ++d) { pts[w * 255 + d - 1] = cur; cur = hx_add(cur, base); }
        base = cur;
    }
    // batch-invert zzz
    std::vector<HFq> pre(pts.size());
    HFq acc = HFq::one();
    for (size_t i = 0; i < pts.size(); ++i) { pre[i] = acc; acc = acc * pts[i].zzz; }
    acc = acc.inv();
    std::vector<HAffine> aff(pts.size());
    for (size_t i = pts.size(); i-- > 0;) {
        HFq iz = acc * pre[i];
        acc = acc * pts[i].zzz;
        HFq t = pts[i].zz * iz;
        aff[i] = {pts[i].x * t.sqr(), pts[i].y * iz};
    }
    ZK_CUDA(ctx, cudaMalloc(&ctx->d_gen_table, aff.size() * sizeof(affine_t)));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->d_gen_table, aff.data(), aff.size() * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

static int32_t fixed_base(b200zk_ctx* ctx, const fe_t* d_sc, size_t n, xyzz_t* d_xyzz, fe_t* d_zzz, affine_t* d_out) {
    setup_fixed_base_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, ctx->stream>>>(d_sc, n, ctx->d_gen_table, d_xyzz, d_zzz);
    ctx->launches++;
    ZK_TRY(batch_invert_run(ctx, d_zzz, n, 1));
    setup_normalize_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, ctx->stream>>>(d_xyzz, d_zzz, n, d_out);
    ctx->launches++;
    ZK_CUDA(ctx, cudaGetLastError());
    return B200ZK_OK;
}

int32_t params_setup_run(b200zk_ctx* ctx, uint32_t k, const host::HFr& s, affine_t* d_g, affine_t* d_g_lagrange) {
    using host::HFr;
    ZK_TRY(ensure_gen_table(ctx));
    size_t n = (size_t)1 << k;
    uint32_t bits = (k + 1) / 2;
    size_t n_lo = (size_t)1 << bits, n_hi = n >> bits ? n >> bits : 1;
    // workspace: scalars[n] | aux[n] | xyzz[n] | lo | hi
    size_t bytes = n * sizeof(fe_t) * 2 + n * sizeof(xyzz_t) + (n_lo + n_hi) * sizeof(fe_t);
    ZK_TRY(ws_reserve(ctx, ctx->setup_ws, bytes));
    fe_t* sc = (fe_t*)ctx->setup_ws.p;
    fe_t* aux = sc + n;
    xyzz_t* xyzz = (xyzz_t*)(aux + n);
    fe_t* lo = (fe_t*)(xyzz + n);
    fe_t* hi = lo + n_lo;
    cudaStream_t st = ctx->stream;
    auto powers = [&](const HFr& base) {
        setup_pow_table_kernel<<<nblocks(n_lo, SETUP_THREADS), SETUP_THREADS, 0, st>>>(lo, to_dev(base), (uint32_t)n_lo, 0);
        setup_pow_table_kernel<<<nblocks(n_hi, SETUP_THREADS), SETUP_THREADS, 0, st>>>(hi, to_dev(base), (uint32_t)n_hi, bits);
        setup_powers_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, st>>>(sc, n, lo, hi, bits);
        ctx->launches += 3;
    };
    powers(s);
    ZK_TRY(fixed_base(ctx, sc, n, xyzz, aux, d_g));
    if (d_g_lagrange) {
        HFr root = host::fr_root_of_unity();
        for (uint32_t i = k; i < host::FR_TWO_ADICITY; ++i) root = root.sqr();
        HFr multiplier = (s.pow_u64(n) - HFr::one()) * HFr::from_u64(n).inv();
        powers(root);
        setup_lagrange_den_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, st>>>(aux, sc, n, to_dev(s));
        ctx->launches++;
        ZK_TRY(batch_invert_run(ctx, aux, n, 0));
        setup_lagrange_scalar_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, st>>>(sc, aux, n, to_dev(multiplier));
        ctx->launches++;
        ZK_TRY(fixed_base(ctx, sc, n, xyzz, aux, d_g_lagrange));
    }
    ZK_CUDA(ctx, cudaGetLastError());
    return B200ZK_OK;
}

// ---- arithmetic::g_to_lagrange: G1 NTT with w^-1, then n^-1 (g1_ntt.cuh) -----------------------
__global__ void __launch_bounds__(SETUP_THREADS) g1_ntt_load_kernel(const affine_t* g, size_t n, uint32_t k, xyzz_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    size_t r = k ? __brevll((unsigned long long)i) >> (64 - k) : 0;
    out[i] = xyzz_from_affine(g[r]);
}
// one butterfly per thread (g1_ntt_stage_body)
__global__ void __launch_bounds__(SETUP_THREADS) g1_ntt_stage_kernel(xyzz_t* a, const fe_t* tw, uint32_t s, uint32_t k) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ((size_t)1 << (k - 1))) g1_ntt_stage_body(a, tw, t, s, k);
}
// p *= n^-1 (canonical); zzz copied to a dense array for the batched inversion
__global__ void __launch_bounds__(SETUP_THREADS) g1_ntt_scale_kernel(xyzz_t* a, size_t n, const fe_t n_inv, fe_t* zzz) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    xyzz_t p = xyzz_mul(a[i], n_inv);
    a[i] = p;
    zzz[i] = p.zzz;
}

int32_t g_to_lagrange_run(b200zk_ctx* ctx, const affine_t* d_g, uint32_t k, affine_t* d_out) {
    using host::HFr;
    if (k > host::FR_TWO_ADICITY) return fail(ctx, B200ZK_EINVAL, "g_to_lagrange", "k exceeds Fr two-adicity");
    const size_t n = (size_t)1 << k, half = n / 2;
    // workspace: xyzz[n] | zzz[n] | tw[n/2]
    ZK_TRY(ws_reserve(ctx, ctx->setup_ws, n * (sizeof(xyzz_t) + sizeof(fe_t)) + half * sizeof(fe_t)));
    xyzz_t* xyzz = (xyzz_t*)ctx->setup_ws.p;
    fe_t* zzz = (fe_t*)(xyzz + n);
    fe_t* tw = zzz + n;
    cudaStream_t st = ctx->stream;
    HFr omega_inv = host::fr_root_of_unity();
    for (uint32_t i = k; i < host::FR_TWO_ADICITY; ++i) omega_inv = omega_inv.sqr();
    omega_inv = omega_inv.inv();
    ZK_TRY(powers_run(ctx, omega_inv, half, tw));
    g1_ntt_load_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, st>>>(d_g, n, k, xyzz);
    ctx->launches++;
    for (uint32_t s = 0; s < k; ++s) {
        g1_ntt_stage_kernel<<<nblocks(half, SETUP_THREADS), SETUP_THREADS, 0, st>>>(xyzz, tw, s, k);
        ctx->launches++;
    }
    uint64_t n_inv[4];
    HFr::from_u64(n).inv().to_canonical(n_inv);
    fe_t n_inv_d; memcpy(n_inv_d.l, n_inv, 32);
    g1_ntt_scale_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, st>>>(xyzz, n, n_inv_d, zzz);
    ctx->launches++;
    ZK_TRY(batch_invert_run(ctx, zzz, n, 1));
    setup_normalize_kernel<<<nblocks(n, SETUP_THREADS), SETUP_THREADS, 0, st>>>(xyzz, zzz, n, d_out);
    ctx->launches++;
    ZK_CUDA(ctx, cudaGetLastError());
    return B200ZK_OK;
}

}  // namespace b200zk
