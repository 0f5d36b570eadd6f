// Many pairing-product checks in one call (b200zk_pairing_checks, include/b200zk.h): halo2curves'
// `multi_miller_loop(..).final_exponentiation() == Gt::identity()`, batched, with the pairing of csrc/pairing.hpp.
// Three launches on the ctx stream:
//   pc_prepare_kernel    one thread per distinct G2 point: its 195 Miller-loop lines (g2_prepare, pairing.cuh)
//   pc_miller_kernel     one thread per check: the multi-Miller product of its m pairs, Fq12 accumulator per thread
//   pc_final_exp_kernel  one thread per check: the final exponentiation and the verdict
// One check is one dependent chain of about 3 * 10^4 Fq multiplications (m = 2), so a batch fills the device and a
// single check runs on one thread.
#include "context.hpp"
#include "pairing.cuh"
#include "pairing.hpp"
#include <map>
#include <vector>

using namespace b200zk;

namespace b200zk {

static constexpr uint32_t PC_THREADS = 128;

__global__ void __launch_bounds__(PC_THREADS) pc_prepare_kernel(const fq2_t* g2, uint32_t nq, pc_line_t* tables) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nq) return;
    g2_prepare(g2[2 * t], g2[2 * t + 1], tables + (size_t)t * PC_LINES);
}

__global__ void __launch_bounds__(PC_THREADS) pc_miller_kernel(const affine_t* g1, const uint32_t* q, const pc_line_t* tables, uint32_t m,
                                                               uint32_t count, fq12_t* f) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    f[t] = pc_miller_product(g1 + (size_t)t * m, q + (size_t)t * m, tables, m);
}

__global__ void __launch_bounds__(PC_THREADS) pc_final_exp_kernel(const fq12_t* f, uint32_t count, int32_t* status) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    status[t] = fq12_is_one(fq12_final_exp(f[t])) ? B200ZK_OK : B200ZK_EVERIFY;
}

namespace {
size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
unsigned blocks_for(size_t threads) { return (unsigned)((threads + PC_THREADS - 1) / PC_THREADS); }
}  // namespace

int32_t pairing_checks_run(b200zk_ctx* ctx, const void* g1, const uint32_t* q, const void* g2, uint32_t nq, uint32_t m, uint32_t count,
                           int32_t* status) {
    const size_t npairs = (size_t)count * m;
    const size_t o_q = align256(npairs * sizeof(affine_t)), o_g2 = o_q + align256(npairs * 4);
    const size_t o_f = align256((size_t)nq * PC_LINES * sizeof(pc_line_t)), o_st = o_f + align256((size_t)count * sizeof(fq12_t));
    ZK_TRY(ws_reserve(ctx, ctx->io_a, o_g2 + (size_t)nq * 128));
    ZK_TRY(ws_reserve(ctx, ctx->setup_ws, o_st + (size_t)count * 4));
    char* a = (char*)ctx->io_a.p;
    char* w = (char*)ctx->setup_ws.p;
    ZK_CUDA(ctx, cudaMemcpyAsync(a, g1, npairs * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(ctx, cudaMemcpyAsync(a + o_q, q, npairs * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (nq) {
        ZK_CUDA(ctx, cudaMemcpyAsync(a + o_g2, g2, (size_t)nq * 128, cudaMemcpyHostToDevice, ctx->stream));
        pc_prepare_kernel<<<blocks_for(nq), PC_THREADS, 0, ctx->stream>>>((const fq2_t*)(a + o_g2), nq, (pc_line_t*)w);
        ctx->launches++;
        ZK_CUDA(ctx, cudaGetLastError());
    }
    pc_miller_kernel<<<blocks_for(count), PC_THREADS, 0, ctx->stream>>>((const affine_t*)a, (const uint32_t*)(a + o_q), (const pc_line_t*)w,
                                                                       m, count, (fq12_t*)(w + o_f));
    ctx->launches++;
    ZK_CUDA(ctx, cudaGetLastError());
    pc_final_exp_kernel<<<blocks_for(count), PC_THREADS, 0, ctx->stream>>>((const fq12_t*)(w + o_f), count, (int32_t*)(w + o_st));
    ctx->launches++;
    ZK_CUDA(ctx, cudaGetLastError());
    ZK_CUDA(ctx, cudaMemcpyAsync(status, w + o_st, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

}  // namespace b200zk

extern "C" int32_t b200zk_pairing_checks(b200zk_ctx* ctx, const void* g1_points, const void* g2_points, uint32_t m, uint32_t count,
                                         int32_t* status) {
    using namespace b200zk::host;
    if (!ctx) return B200ZK_EINVAL;
    if (!g1_points || !g2_points || !status) return fail(ctx, B200ZK_EINVAL, "pairing_checks", "null argument");
    if (count == 0 || m == 0) return fail(ctx, B200ZK_EINVAL, "pairing_checks", "count == 0 or m == 0");
    const size_t npairs = (size_t)count * m;
    // G2 points by their bytes: one line table per distinct point, one curve check per distinct point
    auto less = [](const uint8_t* x, const uint8_t* y) { return memcmp(x, y, 128) < 0; };
    std::map<const uint8_t*, uint32_t, decltype(less)> seen(less);
    std::vector<const uint8_t*> distinct;
    std::vector<uint32_t> q(npairs);
    const HFq b = HFq::from_u64(3);
    for (size_t i = 0; i < npairs; ++i) {
        const uint64_t* p = (const uint64_t*)g1_points + 8 * i;
        const HFq x = HFq::from_limbs(p), y = HFq::from_limbs(p + 4);
        const bool p_id = x.is_zero() && y.is_zero();
        if (!p_id && y.sqr() != x.sqr() * x + b) return fail(ctx, B200ZK_EINVAL, "pairing_checks", "a G1 point is not on the curve");
        const uint8_t* g2 = (const uint8_t*)g2_points + 128 * i;
        auto it = seen.find(g2);
        if (it == seen.end()) {
            const G2A qa = g2_from_limbs(g2);
            if (!g2_on_curve(qa)) return fail(ctx, B200ZK_EINVAL, "pairing_checks", "a G2 point is not on the twist");
            uint32_t idx = PC_SKIP;
            if (!g2_is_identity(qa)) { idx = (uint32_t)distinct.size(); distinct.push_back(g2); }
            it = seen.emplace(g2, idx).first;
        }
        q[i] = p_id ? PC_SKIP : it->second;
    }
    std::vector<uint8_t> g2s(distinct.size() * 128);
    for (size_t k = 0; k < distinct.size(); ++k) memcpy(&g2s[k * 128], distinct[k], 128);
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(pairing_checks_run(ctx, g1_points, q.data(), g2s.data(), (uint32_t)distinct.size(), m, count, status));
    for (uint32_t j = 0; j < count; ++j) if (status[j] != B200ZK_OK) return B200ZK_EVERIFY;
    return B200ZK_OK;
}
