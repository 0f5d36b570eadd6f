// C ABI of libb200zk.so (declarations and reference mapping: include/b200zk.h).
#include "context.hpp"
#include "comm.hpp"
#include <algorithm>
#include <vector>
#include <new>
#include <cuda_profiler_api.h>

using namespace b200zk;
using host::HFr;
using host::HFq;

namespace b200zk {

int32_t fail(b200zk_ctx* ctx, int32_t code, const char* what, const char* detail) {
    if (ctx) {
        ctx->err = std::string(what) + ": " + (detail ? detail : "");
    }
    return code;
}

int32_t ws_reserve(b200zk_ctx* ctx, Workspace& w, size_t bytes) {
    w.used = std::max(w.used, bytes);
    if (bytes <= w.cap) return B200ZK_OK;
    if (w.p) { ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); ZK_CUDA(ctx, cudaFree(w.p)); w.p = nullptr; w.cap = 0; }
    size_t cap = bytes + bytes / 8;
    cudaError_t e = cudaMalloc(&w.p, cap);
    if (e != cudaSuccess) { cap = bytes; e = cudaMalloc(&w.p, cap); }
    if (e != cudaSuccess) { w.p = nullptr; return fail(ctx, B200ZK_ENOMEM, "cudaMalloc(workspace)", cudaGetErrorString(e)); }
    w.cap = cap;
    return B200ZK_OK;
}

// Fixed-base tables for ParamsKZG commits: every MSM of create_proof is over `g` or `g_lagrange`,
// so 2^(c j) * base_i is precomputed once per params object (W * n * 64 B per basis; 0.9 GiB at
// k = 20) when it fits comfortably in HBM.  B200ZK_MSM_PRECOMPUTE=0 disables it.
int32_t params_build_tables(b200zk_params* p) {
    b200zk_ctx* ctx = p->ctx;
    const char* e = getenv("B200ZK_MSM_PRECOMPUTE");
    if (e && e[0] == '0') return B200ZK_OK;
    const size_t n = (size_t)1 << p->k;
    if (p->k < 6) return B200ZK_OK;                               // tiny params: not worth it
    MsmPre pre{msm_pre_shape(n), (uint32_t)n};
    if ((size_t)pre.shape.nwin * n >= ((size_t)1 << 31)) return B200ZK_OK;
    const size_t per_basis = (size_t)pre.shape.nwin * n * sizeof(affine_t);
    const size_t nbases = p->d_g_lagrange ? 2 : 1;
    size_t free_b = 0, total_b = 0;
    ZK_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
    if (per_basis * nbases > free_b / 5 * 2 || per_basis * nbases > ((size_t)48 << 30)) return B200ZK_OK;
    if (cudaMalloc(&p->d_g_pre, per_basis) != cudaSuccess) { p->d_g_pre = nullptr; cudaGetLastError(); return B200ZK_OK; }
    if (p->d_g_lagrange && cudaMalloc(&p->d_gl_pre, per_basis) != cudaSuccess) {
        cudaFree(p->d_g_pre); p->d_g_pre = nullptr; p->d_gl_pre = nullptr; cudaGetLastError(); return B200ZK_OK;
    }
    p->pre = pre;
    ZK_TRY(msm_precompute_run(ctx, p->d_g, n, pre.shape.c, pre.shape.nwin, p->d_g_pre));
    if (p->d_g_lagrange) ZK_TRY(msm_precompute_run(ctx, p->d_g_lagrange, n, pre.shape.c, pre.shape.nwin, p->d_gl_pre));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

// c * (sum of the basis) from the 8-bit window table
static host::HXyzz sum_table_mul(const std::vector<host::HXyzz>& tab, const host::HFr& c_mont) {
    uint64_t limbs[4];
    c_mont.to_canonical(limbs);
    host::HXyzz acc = host::hx_identity();
    for (uint32_t j = 0; j < 32; ++j) {
        uint32_t d = (uint32_t)(limbs[j / 8] >> (8 * (j % 8))) & 0xff;
        if (d) acc = host::hx_add(acc, tab[(size_t)j * 255 + d - 1]);
    }
    return acc;
}

static int32_t build_sum_table(b200zk_params* p, int which, const affine_t* bases, const affine_t* table) {
    b200zk_ctx* ctx = p->ctx;
    const size_t n = (size_t)1 << p->k;
    fe_t* ones = nullptr;
    ZK_CUDA(ctx, cudaMalloc(&ones, n * sizeof(fe_t)));
    fe_t one;
    memcpy(one.l, host::HFr::one().v, 32);
    std::vector<fe_t> h(n, one);
    // on the ctx stream: a plain cudaMemcpy from pageable memory may return before its DMA has landed, and the
    // non-blocking ctx stream does not order itself after the legacy stream (a 64 KB column of ones was read stale)
    cudaError_t e = cudaMemcpyAsync(ones, h.data(), n * sizeof(fe_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    host::HAffine sum;
    int32_t rc = e != cudaSuccess ? fail(ctx, B200ZK_ECUDA, "sum_table", cudaGetErrorString(e))
                                  : (table ? msm_run_ex(ctx, ones, table, n, &p->pre, &sum) : msm_run(ctx, ones, bases, n, &sum));
    cudaFree(ones);
    if (rc != B200ZK_OK) return rc;
    std::vector<host::HXyzz>& tab = p->sum_table[which];
    tab.assign((size_t)32 * 255, host::hx_identity());
    host::HXyzz base = sum.x.is_zero() && sum.y.is_zero() ? host::hx_identity() : host::hx_from_affine(sum);
    for (uint32_t j = 0; j < 32; ++j) {
        host::HXyzz acc = base;
        for (uint32_t d = 1; d <= 255; ++d) { tab[(size_t)j * 255 + d - 1] = acc; acc = host::hx_add(acc, base); }
        base = acc;                                                  // 256 * base
    }
    return B200ZK_OK;
}

// ParamsKZG::commit / commit_lagrange.  Columns of a padded circuit are constant on most rows:
// advice columns are 0 there (the digit pass skips them), but a grand-product column z holds one
// full-width value c on every unused row, which would put 2^k points into each of the W window
// buckets.  When three probes of a full-length column agree on a non-zero c the commitment is
// computed as  MSM(poly - c) + c * sum(basis):  the subtraction happens inside the digit pass and
// turns the column sparse, sum(basis) is computed once per params.  Exact for any column (if the
// probes mislead, MSM(poly - c) is simply dense again).  Several columns of the same length are
// committed in one batched launch sequence (msm_run_multi).
int32_t params_commit_multi(b200zk_params* p, const fe_t* const* d_polys, uint32_t ncols, size_t len, bool lagrange, host::HAffine* outs) {
    b200zk_ctx* ctx = p->ctx;
    const affine_t* bases = lagrange ? p->d_g_lagrange : p->d_g;
    if (!bases) return fail(ctx, B200ZK_EINVAL, "commit", "basis not loaded");
    const size_t n = (size_t)1 << p->k;
    if (len > n) return fail(ctx, B200ZK_EINVAL, "commit", "polynomial longer than the SRS");
    if (ncols == 0) return B200ZK_OK;
    const affine_t* table = lagrange ? p->d_gl_pre : p->d_g_pre;
    const int which = lagrange ? 1 : 0;
    std::vector<fe_t> sub(ncols);
    std::vector<const fe_t*> subp(ncols, nullptr);
    static const bool const_run = !(getenv("B200ZK_MSM_CONST_RUN") && getenv("B200ZK_MSM_CONST_RUN")[0] == '0');
    bool any = false;
    if (const_run && len == n && n >= 1024 && (size_t)ncols * 3 * sizeof(fe_t) <= ((size_t)60 << 10)) {
        fe_t* probe = (fe_t*)ctx->pinned;
        const size_t at[3] = {n / 2, n / 2 + 1, n / 4 * 3};
        for (uint32_t b = 0; b < ncols; ++b)
            for (int i = 0; i < 3; ++i)
                ZK_CUDA(ctx, cudaMemcpyAsync(probe + 3 * b + i, d_polys[b] + at[i], sizeof(fe_t), cudaMemcpyDeviceToHost, ctx->stream));
        ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const fe_t zero{};
        for (uint32_t b = 0; b < ncols; ++b) {
            const fe_t* q = probe + 3 * b;
            if (!memcmp(q, q + 1, 32) && !memcmp(q, q + 2, 32) && memcmp(q, &zero, 32)) { sub[b] = q[0]; subp[b] = &sub[b]; any = true; }
        }
    }
    if (any && p->sum_table[which].empty()) ZK_TRY(build_sum_table(p, which, bases, table));
    ZK_TRY(msm_run_multi(ctx, d_polys, ncols, table ? table : bases, len, table ? &p->pre : nullptr, outs, any ? subp.data() : nullptr));
    for (uint32_t b = 0; b < ncols; ++b) {
        if (!subp[b]) continue;
        host::HFr c;
        memcpy(c.v, sub[b].l, 32);
        host::HXyzz acc = sum_table_mul(p->sum_table[which], c);
        if (!(outs[b].x.is_zero() && outs[b].y.is_zero())) acc = host::hx_add(acc, host::hx_from_affine(outs[b]));
        outs[b] = host::hx_to_affine(acc);
    }
    return B200ZK_OK;
}

int32_t params_commit_range(b200zk_params* p, const fe_t* const* d_polys, uint32_t ncols, size_t lo, size_t hi, bool lagrange, host::HAffine* outs) {
    b200zk_ctx* ctx = p->ctx;
    const affine_t* bases = lagrange ? p->d_g_lagrange : p->d_g;
    if (!bases) return fail(ctx, B200ZK_EINVAL, "commit", "basis not loaded");
    const size_t n = (size_t)1 << p->k;
    if (lo > hi || hi > n) return fail(ctx, B200ZK_EINVAL, "commit", "point range outside the SRS");
    if (ncols == 0) return B200ZK_OK;
    const affine_t* table = lagrange ? p->d_gl_pre : p->d_g_pre;
    std::vector<const fe_t*> cols(ncols);
    for (uint32_t b = 0; b < ncols; ++b) cols[b] = d_polys[b] + lo;
    // table row j of point i sits at table[j * n + i]: offsetting the base pointer by lo keeps that stride
    return msm_run_multi(ctx, cols.data(), ncols, (table ? table : bases) + lo, hi - lo, table ? &p->pre : nullptr, outs, nullptr);
}

int32_t params_sum_tables(b200zk_params* p) {
    if (p->sum_table[0].empty()) ZK_TRY(build_sum_table(p, 0, p->d_g, p->d_g_pre));
    if (p->d_g_lagrange && p->sum_table[1].empty()) ZK_TRY(build_sum_table(p, 1, p->d_g_lagrange, p->d_gl_pre));
    return B200ZK_OK;
}

int32_t params_commit_run(b200zk_params* p, const fe_t* d_poly, size_t len, bool lagrange, host::HAffine* out) {
    return params_commit_multi(p, &d_poly, 1, len, lagrange, out);
}

}  // namespace b200zk

static void write_g1(const host::HAffine& a, void* out_g1) {
    uint64_t* o = (uint64_t*)out_g1;
    if (a.x.is_zero() && a.y.is_zero()) {           // G1::identity() = (0, 1, 0)
        memset(o, 0, 96);
        HFq::one().store(o + 4);
        return;
    }
    a.x.store(o); a.y.store(o + 4); HFq::one().store(o + 8);
}

extern "C" {

int32_t b200zk_ctx_create(int32_t device, b200zk_ctx** out) {
    if (!out) return B200ZK_EINVAL;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return B200ZK_ENODEV;
    if (cudaSetDevice(device) != cudaSuccess) return B200ZK_ENODEV;
    b200zk_ctx* ctx = new (std::nothrow) b200zk_ctx();
    if (!ctx) return B200ZK_ENOMEM;
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return B200ZK_ENODEV; }
    ctx->sm_count = prop.multiProcessorCount;
    if (prop.major < 10) { delete ctx; return B200ZK_ENODEV; }     // sm_100a code only
    // the main stream outranks the side stream: its (often small, latency-bound) kernels take the
    // block slots that free up before the side stream's big NTT grids refill them
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) { delete ctx; return B200ZK_ECUDA; }
    if (cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_lo) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess) { cudaStreamDestroy(ctx->stream); delete ctx; return B200ZK_ECUDA; }
    for (auto& e : ctx->events) if (cudaEventCreate(&e) != cudaSuccess) { delete ctx; return B200ZK_ECUDA; }
    if (cudaHostAlloc(&ctx->pinned, 1 << 16, cudaHostAllocDefault) != cudaSuccess) { delete ctx; return B200ZK_ECUDA; }
    *out = ctx;
    return B200ZK_OK;
}

void b200zk_ctx_destroy(b200zk_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->comm && ctx->comm_owned) delete ctx->comm;
    ctx->comm = nullptr;
    for (auto& kv : ctx->ntt_plans) if (!kv.second.borrowed) { cudaFree(kv.second.roots); cudaFree(kv.second.tw_lo); cudaFree(kv.second.tw_hi); cudaFree(kv.second.tw_full); cudaFree(kv.second.roots_s); cudaFree(kv.second.tw_full_s); }
    for (Workspace* w : {&ctx->ntt_scratch, &ctx->ntt_scratch2, &ctx->msm_ws, &ctx->msm_ws2, &ctx->lookup_ws, &ctx->io_a, &ctx->io_b, &ctx->poly_ws, &ctx->poly_heads, &ctx->poly_batch, &ctx->setup_ws}) if (w->p) cudaFree(w->p);
    if (ctx->d_gen_table) cudaFree(ctx->d_gen_table);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    for (auto& e : ctx->events) if (e) cudaEventDestroy(e);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* b200zk_last_error(const b200zk_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }

int32_t b200zk_sync(b200zk_ctx* ctx) {
    if (!ctx) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

uint64_t b200zk_launch_count(const b200zk_ctx* ctx) { return ctx ? ctx->launches : 0; }

int32_t b200zk_profiler_range(b200zk_ctx* ctx, int32_t start) {
    if (!ctx) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (start) ZK_CUDA(ctx, cudaProfilerStart()); else ZK_CUDA(ctx, cudaProfilerStop());
    return B200ZK_OK;
}

int32_t b200zk_event_record(b200zk_ctx* ctx, uint32_t slot) {
    if (!ctx || slot >= 64) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaEventRecord(ctx->events[slot], ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_event_elapsed_ms(b200zk_ctx* ctx, uint32_t from_slot, uint32_t to_slot, float* ms) {
    if (!ctx || from_slot >= 64 || to_slot >= 64 || !ms) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaEventSynchronize(ctx->events[to_slot]));
    ZK_CUDA(ctx, cudaEventElapsedTime(ms, ctx->events[from_slot], ctx->events[to_slot]));
    return B200ZK_OK;
}

// ---- memory ------------------------------------------------------------------
int32_t b200zk_malloc(b200zk_ctx* ctx, size_t bytes, void** dptr) {
    if (!ctx || !dptr) return B200ZK_EINVAL;
    cudaError_t e = cudaMalloc(dptr, bytes ? bytes : 1);
    if (e != cudaSuccess) return fail(ctx, B200ZK_ENOMEM, "cudaMalloc", cudaGetErrorString(e));
    return B200ZK_OK;
}
int32_t b200zk_free(b200zk_ctx* ctx, void* dptr) {
    if (!ctx) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ZK_CUDA(ctx, cudaFree(dptr));
    return B200ZK_OK;
}
int32_t b200zk_upload(b200zk_ctx* ctx, void* dptr, const void* hostp, size_t bytes) {
    if (!ctx) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaMemcpyAsync(dptr, hostp, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}
int32_t b200zk_download(b200zk_ctx* ctx, void* hostp, const void* dptr, size_t bytes) {
    if (!ctx) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaMemcpyAsync(hostp, dptr, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}
int32_t b200zk_memset_zero(b200zk_ctx* ctx, void* dptr, size_t bytes) {
    if (!ctx) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaMemsetAsync(dptr, 0, bytes, ctx->stream));
    return B200ZK_OK;
}
int32_t b200zk_host_alloc(b200zk_ctx* ctx, size_t bytes, void** hptr) {
    if (!ctx || !hptr) return B200ZK_EINVAL;
    cudaError_t e = cudaHostAlloc(hptr, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(ctx, B200ZK_ENOMEM, "cudaHostAlloc", cudaGetErrorString(e));
    return B200ZK_OK;
}
int32_t b200zk_host_free(b200zk_ctx* ctx, void* hptr) {
    if (!ctx) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaFreeHost(hptr));
    return B200ZK_OK;
}

// ---- best_multiexp --------------------------------------------------------------
int32_t b200zk_msm_set_window(b200zk_ctx* ctx, int32_t c) {
    if (!ctx || c < 0 || c > 20 || c == 1) return B200ZK_EINVAL;
    ctx->msm_force_c = c;
    return B200ZK_OK;
}

int32_t b200zk_msm_dev(b200zk_ctx* ctx, const void* d_coeffs, const void* d_bases, size_t len, void* out_g1_host) {
    if (!ctx || !out_g1_host || (len && (!d_coeffs || !d_bases))) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    host::HAffine r;
    ZK_TRY(msm_run(ctx, (const fe_t*)d_coeffs, (const affine_t*)d_bases, len, &r));
    write_g1(r, out_g1_host);
    return B200ZK_OK;
}

int32_t b200zk_msm(b200zk_ctx* ctx, const void* coeffs, const void* bases, size_t len, void* out_g1) {
    if (!ctx || !out_g1 || (len && (!coeffs || !bases))) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(ws_reserve(ctx, ctx->io_a, len * sizeof(fe_t)));
    ZK_TRY(ws_reserve(ctx, ctx->io_b, len * sizeof(affine_t)));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_a.p, coeffs, len * sizeof(fe_t), cudaMemcpyHostToDevice, ctx->stream));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_b.p, bases, len * sizeof(affine_t), cudaMemcpyHostToDevice, ctx->stream));
    return b200zk_msm_dev(ctx, ctx->io_a.p, ctx->io_b.p, len, out_g1);
}

// Sum of `count` G1 points (Jacobian {x,y,z}, any z) on the host: the combine step of a
// point-range sharded MSM after the partial sums have been all-gathered (O(#GPUs) additions).
int32_t b200zk_g1_sum(const void* points_g1, size_t count, void* out_g1) {
    if (!out_g1 || (count && !points_g1)) return B200ZK_EINVAL;
    using namespace host;
    HXyzz acc = hx_identity();
    const uint64_t* p = (const uint64_t*)points_g1;
    for (size_t i = 0; i < count; ++i, p += 12) {
        HFq x = HFq::from_limbs(p), y = HFq::from_limbs(p + 4), z = HFq::from_limbs(p + 8);
        if (z.is_zero()) continue;
        HFq zz = z.sqr();
        acc = hx_add(acc, HXyzz{x, y, zz, zz * z});
    }
    write_g1(hx_to_affine(acc), out_g1);
    return B200ZK_OK;
}

// ---- best_fft ---------------------------------------------------------------------
int32_t b200zk_fft_dev(b200zk_ctx* ctx, void* d_a, const void* omega_host, uint32_t log_n) {
    if (!ctx || !d_a || !omega_host || log_n > 30) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    HFr omega = HFr::from_limbs(omega_host);
    return ntt_run(ctx, (const fe_t*)d_a, 1u << log_n, (fe_t*)d_a, log_n, omega, nullptr, nullptr);
}

int32_t b200zk_fft_colstep_dev(b200zk_ctx* ctx, void* d_block, uint32_t log_r, uint32_t log_cg, uint32_t col0,
                               const void* omega_n, uint32_t log_n) {
    if (!ctx || !d_block || !omega_n || log_n > 30 || log_r + log_cg > log_n) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    return ntt_colstep_run(ctx, (fe_t*)d_block, log_r, log_cg, col0, HFr::from_limbs(omega_n), log_n);
}

int32_t b200zk_fft_colstep_scatter_dev(b200zk_ctx* ctx, void* d_block, uint32_t log_r, uint32_t log_cg, uint32_t col0,
                                       const void* omega_n, uint32_t log_n, void* const* peer_rows, uint32_t world) {
    if (!ctx || !d_block || !omega_n || !peer_rows || log_n > 30 || log_r + log_cg > log_n) return B200ZK_EINVAL;
    for (uint32_t j = 0; j < world && j < 8; ++j) if (!peer_rows[j]) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    return ntt_colstep_run(ctx, (fe_t*)d_block, log_r, log_cg, col0, HFr::from_limbs(omega_n), log_n, (fe_t* const*)peer_rows, world);
}

// CUDA IPC: let another process on the node (one process per GPU) address a b200zk_malloc'ed buffer
int32_t b200zk_ipc_get_handle(b200zk_ctx* ctx, const void* d_ptr, void* handle64) {
    if (!ctx || !d_ptr || !handle64) return B200ZK_EINVAL;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_CUDA(ctx, cudaIpcGetMemHandle((cudaIpcMemHandle_t*)handle64, const_cast<void*>(d_ptr)));
    return B200ZK_OK;
}
int32_t b200zk_ipc_open(b200zk_ctx* ctx, const void* handle64, void** d_ptr) {
    if (!ctx || !handle64 || !d_ptr) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    ZK_CUDA(ctx, cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return B200ZK_OK;
}
int32_t b200zk_ipc_close(b200zk_ctx* ctx, void* d_ptr) {
    if (!ctx || !d_ptr) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_CUDA(ctx, cudaIpcCloseMemHandle(d_ptr));
    return B200ZK_OK;
}

int32_t b200zk_fft_rows_dev(b200zk_ctx* ctx, void* d_rows, uint32_t nrows, const void* omega_c, uint32_t log_c) {
    if (!ctx || !d_rows || !omega_c || log_c > 30) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    return ntt_rows_run(ctx, (fe_t*)d_rows, nrows, HFr::from_limbs(omega_c), log_c);
}

int32_t b200zk_fft(b200zk_ctx* ctx, void* a, const void* omega, uint32_t log_n) {
    if (!ctx || !a || !omega || log_n > 30) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    size_t bytes = sizeof(fe_t) << log_n;
    ZK_TRY(ws_reserve(ctx, ctx->io_a, bytes));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_a.p, a, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_TRY(b200zk_fft_dev(ctx, ctx->io_a.p, omega, log_n));
    ZK_CUDA(ctx, cudaMemcpyAsync(a, ctx->io_a.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

// ---- EvaluationDomain ---------------------------------------------------------------
int32_t b200zk_domain_create(b200zk_ctx* ctx, uint32_t j, uint32_t k, b200zk_domain** out) {
    if (!ctx || !out || j < 2 || k > host::FR_TWO_ADICITY) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    b200zk_domain* d = new (std::nothrow) b200zk_domain();
    if (!d) return B200ZK_ENOMEM;
    d->ctx = ctx; d->k = k;
    d->quotient_poly_degree = j - 1;
    uint64_t n = 1ull << k;
    d->extended_k = k;
    while ((1ull << d->extended_k) < n * d->quotient_poly_degree) d->extended_k++;
    if (d->extended_k > host::FR_TWO_ADICITY) { delete d; return fail(ctx, B200ZK_EINVAL, "domain_create", "extended_k exceeds Fr two-adicity"); }
    d->extended_omega = host::fr_root_of_unity();
    for (uint32_t i = d->extended_k; i < host::FR_TWO_ADICITY; ++i) d->extended_omega = d->extended_omega.sqr();
    d->omega = d->extended_omega;
    for (uint32_t i = k; i < d->extended_k; ++i) d->omega = d->omega.sqr();
    d->omega_inv = d->omega.inv();
    d->extended_omega_inv = d->extended_omega.inv();
    d->g_coset = host::fr_zeta();
    d->g_coset_inv = d->g_coset.sqr();
    d->ifft_divisor = HFr::from_u64(n).inv();
    d->extended_ifft_divisor = HFr::from_u64(1ull << d->extended_k).inv();
    d->barycentric_weight = d->ifft_divisor;
    // t_evaluations[i] = 1 / (zeta^n * (extended_omega^n)^i - 1)
    size_t m = (size_t)1 << (d->extended_k - k);
    std::vector<HFr> t(m);
    HFr cur = d->g_coset.pow_u64(n), step = d->extended_omega.pow_u64(n);
    for (size_t i = 0; i < m; ++i) { t[i] = (cur - HFr::one()).inv(); cur = cur * step; }
    cudaError_t e = cudaMalloc(&d->d_t_evaluations, m * sizeof(fe_t));
    if (e != cudaSuccess) { delete d; return fail(ctx, B200ZK_ENOMEM, "cudaMalloc", cudaGetErrorString(e)); }
    e = cudaMemcpyAsync(d->d_t_evaluations, t.data(), m * sizeof(fe_t), cudaMemcpyHostToDevice, ctx->stream);   // ordered before this ctx's kernels
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { cudaFree(d->d_t_evaluations); delete d; return fail(ctx, B200ZK_ECUDA, "cudaMemcpy", cudaGetErrorString(e)); }
    *out = d;
    return B200ZK_OK;
}

void b200zk_domain_destroy(b200zk_domain* d) {
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    cudaStreamSynchronize(d->ctx->stream);
    cudaFree(d->d_t_evaluations);
    delete d;
}

uint32_t b200zk_domain_k(const b200zk_domain* d) { return d ? d->k : 0; }
uint32_t b200zk_domain_extended_k(const b200zk_domain* d) { return d ? d->extended_k : 0; }
uint32_t b200zk_domain_quotient_poly_degree(const b200zk_domain* d) { return d ? d->quotient_poly_degree : 0; }

int32_t b200zk_domain_constant(const b200zk_domain* d, uint32_t which, void* out_fr) {
    if (!d || !out_fr || which > 8) return B200ZK_EINVAL;
    const HFr* f[] = {&d->omega, &d->omega_inv, &d->extended_omega, &d->extended_omega_inv, &d->g_coset, &d->g_coset_inv,
                      &d->ifft_divisor, &d->extended_ifft_divisor, &d->barycentric_weight};
    f[which]->store(out_fr);
    return B200ZK_OK;
}

// EvaluationDomain::rotate_omega(value, rotation) = value * omega^rotation
int32_t b200zk_domain_rotate_omega(const b200zk_domain* d, const void* value_fr, int32_t rotation, void* out_fr) {
    if (!d || !value_fr || !out_fr) return B200ZK_EINVAL;
    HFr v = HFr::from_limbs(value_fr);
    HFr r = rotation >= 0 ? v * d->omega.pow_u64((uint64_t)rotation) : v * d->omega_inv.pow_u64((uint64_t)(-(int64_t)rotation));
    r.store(out_fr);
    return B200ZK_OK;
}

// EvaluationDomain::l_i_range(x, x^n, rot_lo..=rot_hi): l_i(x) = (x^n - 1) / n * omega^i / (x - omega^i) for every
// rotation i of the range (the verifier's l_0, l_last, l_blind and instance evaluations).  Like upstream, an x
// inside the domain has no defined value here (upstream divides by zero silently): EINVAL.
int32_t b200zk_domain_l_i_range(const b200zk_domain* d, const void* x_fr, int32_t rot_lo, int32_t rot_hi, void* out_fr) {
    if (!d || !x_fr || !out_fr || rot_hi < rot_lo) return B200ZK_EINVAL;
    HFr x = HFr::from_limbs(x_fr), xn = x;
    for (uint32_t i = 0; i < d->k; ++i) xn = xn.sqr();
    HFr common = (xn - HFr::one()) * d->barycentric_weight;
    size_t count = (size_t)((int64_t)rot_hi - rot_lo + 1);
    std::vector<HFr> root(count), den(count), pref(count);
    HFr w = rot_lo >= 0 ? d->omega.pow_u64((uint64_t)rot_lo) : d->omega_inv.pow_u64((uint64_t)(-(int64_t)rot_lo));
    HFr acc = HFr::one();
    for (size_t i = 0; i < count; ++i) {
        root[i] = w; den[i] = x - w;
        if (den[i].is_zero()) return B200ZK_EINVAL;
        pref[i] = acc; acc = acc * den[i];
        w = w * d->omega;
    }
    HFr inv = acc.inv();                                       // one inversion for the range (BatchInvert)
    for (size_t i = count; i-- > 0;) {
        HFr di = inv * pref[i];
        inv = inv * den[i];
        (di * root[i] * common).store((uint8_t*)out_fr + 32 * i);
    }
    return B200ZK_OK;
}

// EvaluationDomain::rotate_extended(poly, rotation): out[i] = in[(i + rotation * 2^(extended_k - k)) mod 2^extended_k]
int32_t b200zk_rotate_extended_dev(b200zk_domain* d, const void* d_in, int32_t rotation, void* d_out) {
    if (!d || !d_in || !d_out || d_in == d_out) return B200ZK_EINVAL;
    ZK_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    const size_t ext = (size_t)1 << d->extended_k;
    const int64_t step = (int64_t)rotation * (int64_t)(1u << (d->extended_k - d->k));
    const size_t sh = (size_t)(((step % (int64_t)ext) + (int64_t)ext) % (int64_t)ext);
    const fe_t* in = (const fe_t*)d_in;
    fe_t* out = (fe_t*)d_out;
    ZK_CUDA(d->ctx, cudaMemcpyAsync(out, in + sh, (ext - sh) * sizeof(fe_t), cudaMemcpyDeviceToDevice, d->ctx->stream));
    if (sh) ZK_CUDA(d->ctx, cudaMemcpyAsync(out + (ext - sh), in, sh * sizeof(fe_t), cudaMemcpyDeviceToDevice, d->ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_lagrange_to_coeff_dev(b200zk_domain* d, void* d_a) {
    if (!d || !d_a) return B200ZK_EINVAL;
    ZK_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    HFr post[3] = {d->ifft_divisor, d->ifft_divisor, d->ifft_divisor};
    d->ctx->ntt_sparse_hint = true;
    int32_t rc = ntt_run(d->ctx, (const fe_t*)d_a, 1u << d->k, (fe_t*)d_a, d->k, d->omega_inv, nullptr, post);
    d->ctx->ntt_sparse_hint = false;
    return rc;
}

int32_t b200zk_coeff_to_extended_dev(b200zk_domain* d, const void* d_coeffs, void* d_out_ext) {
    if (!d || !d_coeffs || !d_out_ext) return B200ZK_EINVAL;
    ZK_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    HFr pre[3] = {HFr::one(), d->g_coset, d->g_coset_inv};
    return ntt_run(d->ctx, (const fe_t*)d_coeffs, 1u << d->k, (fe_t*)d_out_ext, d->extended_k, d->extended_omega, pre, nullptr);
}

int32_t b200zk_extended_to_coeff_dev(b200zk_domain* d, void* d_ext, void* d_out_coeffs) {
    if (!d || !d_ext || !d_out_coeffs) return B200ZK_EINVAL;
    b200zk_ctx* ctx = d->ctx;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    HFr dv = d->extended_ifft_divisor;
    HFr post[3] = {dv, dv * d->g_coset_inv, dv * d->g_coset};
    ZK_TRY(ntt_run(ctx, (const fe_t*)d_ext, 1u << d->extended_k, (fe_t*)d_ext, d->extended_k, d->extended_omega_inv, nullptr, post));
    size_t bytes = (sizeof(fe_t) << d->k) * d->quotient_poly_degree;
    if (d_out_coeffs != d_ext) ZK_CUDA(ctx, cudaMemcpyAsync(d_out_coeffs, d_ext, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_divide_by_vanishing_poly_dev(b200zk_domain* d, void* d_ext) {
    if (!d || !d_ext) return B200ZK_EINVAL;
    ZK_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    return fr_scale_periodic(d->ctx, (fe_t*)d_ext, (size_t)1 << d->extended_k, d->d_t_evaluations, 1u << (d->extended_k - d->k));
}

int32_t b200zk_lagrange_to_coeff(b200zk_domain* d, void* a) {
    if (!d || !a) return B200ZK_EINVAL;
    b200zk_ctx* ctx = d->ctx;
    size_t bytes = sizeof(fe_t) << d->k;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(ws_reserve(ctx, ctx->io_a, bytes));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_a.p, a, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_TRY(b200zk_lagrange_to_coeff_dev(d, ctx->io_a.p));
    ZK_CUDA(ctx, cudaMemcpyAsync(a, ctx->io_a.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_coeff_to_extended(b200zk_domain* d, const void* coeffs, void* out_ext) {
    if (!d || !coeffs || !out_ext) return B200ZK_EINVAL;
    b200zk_ctx* ctx = d->ctx;
    size_t in_bytes = sizeof(fe_t) << d->k, out_bytes = sizeof(fe_t) << d->extended_k;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(ws_reserve(ctx, ctx->io_a, in_bytes));
    ZK_TRY(ws_reserve(ctx, ctx->io_b, out_bytes));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_a.p, coeffs, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_TRY(b200zk_coeff_to_extended_dev(d, ctx->io_a.p, ctx->io_b.p));
    ZK_CUDA(ctx, cudaMemcpyAsync(out_ext, ctx->io_b.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_extended_to_coeff(b200zk_domain* d, const void* ext, void* out_coeffs) {
    if (!d || !ext || !out_coeffs) return B200ZK_EINVAL;
    b200zk_ctx* ctx = d->ctx;
    size_t in_bytes = sizeof(fe_t) << d->extended_k, out_bytes = (sizeof(fe_t) << d->k) * d->quotient_poly_degree;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(ws_reserve(ctx, ctx->io_b, in_bytes));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_b.p, ext, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_TRY(b200zk_extended_to_coeff_dev(d, ctx->io_b.p, ctx->io_b.p));
    ZK_CUDA(ctx, cudaMemcpyAsync(out_coeffs, ctx->io_b.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_divide_by_vanishing_poly(b200zk_domain* d, void* ext) {
    if (!d || !ext) return B200ZK_EINVAL;
    b200zk_ctx* ctx = d->ctx;
    size_t bytes = sizeof(fe_t) << d->extended_k;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(ws_reserve(ctx, ctx->io_b, bytes));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_b.p, ext, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_TRY(b200zk_divide_by_vanishing_poly_dev(d, ctx->io_b.p));
    ZK_CUDA(ctx, cudaMemcpyAsync(ext, ctx->io_b.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

// ---- ParamsKZG ------------------------------------------------------------------------
int32_t b200zk_params_load(b200zk_ctx* ctx, uint32_t k, const void* g, const void* g_lagrange, b200zk_params** out) {
    if (!ctx || !out || !g || k > host::FR_TWO_ADICITY) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    b200zk_params* p = new (std::nothrow) b200zk_params();
    if (!p) return B200ZK_ENOMEM;
    p->ctx = ctx; p->k = k; p->d_g = nullptr; p->d_g_lagrange = nullptr;
    size_t bytes = sizeof(affine_t) << k;
    cudaError_t e = cudaMalloc(&p->d_g, bytes);
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_g, g, bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess && g_lagrange) {
        e = cudaMalloc(&p->d_g_lagrange, bytes);
        if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_g_lagrange, g_lagrange, bytes, cudaMemcpyHostToDevice, ctx->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);             // the caller's buffers are borrowed for the call only
    if (e != cudaSuccess) {
        cudaFree(p->d_g); cudaFree(p->d_g_lagrange); delete p;
        return fail(ctx, B200ZK_ECUDA, "params_load", cudaGetErrorString(e));
    }
    int32_t rc = params_build_tables(p);
    if (rc != B200ZK_OK) { b200zk_params_destroy(p); return rc; }
    *out = p;
    return B200ZK_OK;
}

void b200zk_params_destroy(b200zk_params* p) {
    if (!p) return;
    cudaSetDevice(p->ctx->device);
    cudaStreamSynchronize(p->ctx->stream);
    cudaFree(p->d_g); cudaFree(p->d_g_lagrange); cudaFree(p->d_g_pre); cudaFree(p->d_gl_pre);
    delete p;
}

int32_t b200zk_params_read(b200zk_params* p, void* g_out, void* g_lagrange_out) {
    if (!p) return B200ZK_EINVAL;
    b200zk_ctx* ctx = p->ctx;
    size_t bytes = sizeof(affine_t) << p->k;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (g_out) ZK_CUDA(ctx, cudaMemcpyAsync(g_out, p->d_g, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (g_lagrange_out) {
        if (!p->d_g_lagrange) return fail(ctx, B200ZK_EINVAL, "params_read", "no lagrange basis loaded");
        ZK_CUDA(ctx, cudaMemcpyAsync(g_lagrange_out, p->d_g_lagrange, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_commit_dev(b200zk_params* p, const void* d_poly, size_t len, int32_t lagrange, void* out_g1_host) {
    if (!p || !out_g1_host || (len && !d_poly) || len > ((size_t)1 << p->k)) return B200ZK_EINVAL;
    ZK_CUDA(p->ctx, cudaSetDevice(p->ctx->device));
    host::HAffine r;
    ZK_TRY(params_commit_run(p, (const fe_t*)d_poly, len, lagrange != 0, &r));
    write_g1(r, out_g1_host);
    return B200ZK_OK;
}

int32_t b200zk_commit_many_dev(b200zk_params* p, const void* const* d_polys, uint32_t count, size_t len, int32_t lagrange,
                               void* out_g1_host) {
    if (!p || (count && (!d_polys || !out_g1_host)) || len > ((size_t)1 << p->k)) return B200ZK_EINVAL;
    for (uint32_t i = 0; i < count; ++i) if (len && !d_polys[i]) return B200ZK_EINVAL;
    ZK_CUDA(p->ctx, cudaSetDevice(p->ctx->device));
    std::vector<host::HAffine> r(count);
    for (uint32_t b = 0; b < count; b += 24) {
        uint32_t m = std::min<uint32_t>(24, count - b);
        ZK_TRY(params_commit_multi(p, (const fe_t* const*)d_polys + b, m, len, lagrange != 0, r.data() + b));
    }
    for (uint32_t i = 0; i < count; ++i) write_g1(r[i], (char*)out_g1_host + (size_t)i * 96);
    return B200ZK_OK;
}

static int32_t commit_host(b200zk_params* p, const void* poly, size_t len, int32_t lagrange, void* out_g1) {
    if (!p || !out_g1 || (len && !poly) || len > ((size_t)1 << p->k)) return B200ZK_EINVAL;
    b200zk_ctx* ctx = p->ctx;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(ws_reserve(ctx, ctx->io_a, len * sizeof(fe_t)));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_a.p, poly, len * sizeof(fe_t), cudaMemcpyHostToDevice, ctx->stream));
    return b200zk_commit_dev(p, ctx->io_a.p, len, lagrange, out_g1);
}

int32_t b200zk_commit(b200zk_params* p, const void* poly, size_t len, void* out_g1) { return commit_host(p, poly, len, 0, out_g1); }
int32_t b200zk_commit_lagrange(b200zk_params* p, const void* poly, size_t len, void* out_g1) { return commit_host(p, poly, len, 1, out_g1); }

int32_t b200zk_params_setup(b200zk_ctx* ctx, uint32_t k, const void* s_fr, b200zk_params** out) {
    if (!ctx || !out || !s_fr || k > host::FR_TWO_ADICITY) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    b200zk_params* p = new (std::nothrow) b200zk_params();
    if (!p) return B200ZK_ENOMEM;
    p->ctx = ctx; p->k = k; p->d_g = nullptr; p->d_g_lagrange = nullptr;
    size_t bytes = sizeof(affine_t) << k;
    cudaError_t e = cudaMalloc(&p->d_g, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_g_lagrange, bytes);
    int32_t rc = e == cudaSuccess ? params_setup_run(ctx, k, HFr::from_limbs(s_fr), p->d_g, p->d_g_lagrange)
                                  : fail(ctx, B200ZK_ENOMEM, "params_setup", cudaGetErrorString(e));
    if (rc == B200ZK_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, B200ZK_ECUDA, "params_setup", "sync failed");
    if (rc == B200ZK_OK) rc = params_build_tables(p);
    if (rc != B200ZK_OK) { b200zk_params_destroy(p); return rc; }
    *out = p;
    return B200ZK_OK;
}

int32_t b200zk_g_to_lagrange_dev(b200zk_ctx* ctx, const void* d_g, uint32_t k, void* d_out) {
    if (!ctx) return B200ZK_EINVAL;
    if (!d_g || !d_out) return fail(ctx, B200ZK_EINVAL, "g_to_lagrange", "null pointer");
    if (k > host::FR_TWO_ADICITY) return fail(ctx, B200ZK_EINVAL, "g_to_lagrange", "k exceeds Fr two-adicity");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(g_to_lagrange_run(ctx, (const affine_t*)d_g, k, (affine_t*)d_out));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_g_to_lagrange(b200zk_ctx* ctx, const void* g, uint32_t k, void* out) {
    if (!ctx) return B200ZK_EINVAL;
    if (!g || !out) return fail(ctx, B200ZK_EINVAL, "g_to_lagrange", "null pointer");
    if (k > host::FR_TWO_ADICITY) return fail(ctx, B200ZK_EINVAL, "g_to_lagrange", "k exceeds Fr two-adicity");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    size_t bytes = sizeof(affine_t) << k;
    ZK_TRY(ws_reserve(ctx, ctx->io_b, bytes));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_b.p, g, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZK_TRY(b200zk_g_to_lagrange_dev(ctx, ctx->io_b.p, k, ctx->io_b.p));
    ZK_CUDA(ctx, cudaMemcpyAsync(out, ctx->io_b.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZK_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B200ZK_OK;
}

int32_t b200zk_params_downsize(const b200zk_params* src, uint32_t k, b200zk_params** out) {
    if (!src) return B200ZK_EINVAL;
    b200zk_ctx* ctx = src->ctx;
    if (!out) return fail(ctx, B200ZK_EINVAL, "params_downsize", "null pointer");
    if (k > src->k) return fail(ctx, B200ZK_EINVAL, "params_downsize", "k exceeds the source params' k");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    b200zk_params* p = new (std::nothrow) b200zk_params();
    if (!p) return B200ZK_ENOMEM;
    p->ctx = ctx; p->k = k; p->d_g = nullptr; p->d_g_lagrange = nullptr;
    size_t bytes = sizeof(affine_t) << k;
    int32_t rc = B200ZK_OK;
    cudaError_t e = cudaMalloc(&p->d_g, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_g_lagrange, bytes);
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_g, src->d_g, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e != cudaSuccess) rc = fail(ctx, B200ZK_ENOMEM, "params_downsize", cudaGetErrorString(e));
    if (rc == B200ZK_OK) rc = g_to_lagrange_run(ctx, p->d_g, k, p->d_g_lagrange);
    if (rc == B200ZK_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = fail(ctx, B200ZK_ECUDA, "params_downsize", "sync failed");
    if (rc == B200ZK_OK) rc = params_build_tables(p);
    if (rc != B200ZK_OK) { b200zk_params_destroy(p); return rc; }
    *out = p;
    return B200ZK_OK;
}

// ---- eval_polynomial / kate_division / BatchInvert / grand-product scan ---------------------
int32_t b200zk_eval_polynomial_dev(b200zk_ctx* ctx, const void* d_poly, size_t len, const void* x_fr, void* out_fr_host) {
    if (!ctx || !x_fr || !out_fr_host || (len && !d_poly)) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    HFr head;
    ZK_TRY(recurrence_run(ctx, (const fe_t*)d_poly, nullptr, len, HFr::from_limbs(x_fr), &head));
    head.store(out_fr_host);
    return B200ZK_OK;
}

int32_t b200zk_eval_polynomial(b200zk_ctx* ctx, const void* poly, size_t len, const void* x_fr, void* out_fr) {
    if (!ctx || !x_fr || !out_fr || (len && !poly)) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    ZK_TRY(ws_reserve(ctx, ctx->io_a, len * sizeof(fe_t)));
    ZK_CUDA(ctx, cudaMemcpyAsync(ctx->io_a.p, poly, len * sizeof(fe_t), cudaMemcpyHostToDevice, ctx->stream));
    return b200zk_eval_polynomial_dev(ctx, ctx->io_a.p, len, x_fr, out_fr);
}

int32_t b200zk_kate_division_dev(b200zk_ctx* ctx, const void* d_a, size_t len, const void* b_fr, void* d_q) {
    if (!ctx || !d_a || !b_fr || !d_q || len < 1) return B200ZK_EINVAL;
    if (len == 1) return B200ZK_OK;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    // q[i] = a[i+1] + b q[i+1]: the Horner recurrence on a[1..]
    return recurrence_run(ctx, (const fe_t*)d_a + 1, (fe_t*)d_q, len - 1, HFr::from_limbs(b_fr), nullptr);
}

int32_t b200zk_batch_invert_dev(b200zk_ctx* ctx, void* d_a, size_t len, int32_t field) {
    if (!ctx || (len && !d_a) || field < 0 || field > 1) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    return batch_invert_run(ctx, (fe_t*)d_a, len, field);
}

int32_t b200zk_prefix_product_dev(b200zk_ctx* ctx, const void* d_p, void* d_z, size_t len, const void* z0_fr) {
    if (!ctx || !z0_fr || (len && (!d_p || !d_z))) return B200ZK_EINVAL;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    return prefix_product_run(ctx, (const fe_t*)d_p, (fe_t*)d_z, len, HFr::from_limbs(z0_fr));
}

}  // extern "C"
