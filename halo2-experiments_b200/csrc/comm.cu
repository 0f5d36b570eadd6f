// Comm implementations (comm.hpp) and their C ABI: b200zk_comm_* (one process per GPU, NCCL) and
// b200zk_group_* (one process driving several GPUs, the ranks are threads).
#include "context.hpp"
#include "comm.hpp"
#include <nccl.h>
#include <dlfcn.h>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <algorithm>
#include <new>
#include <thread>
#include <vector>

namespace b200zk {

// ------------------------------------------------------------------ ranks = threads of one process
struct LocalState {
    int world = 0;
    std::mutex mu;
    std::condition_variable cv;
    int count = 0;
    uint64_t gen = 0;
    bool aborted = false;
    std::vector<std::vector<CommPiece>> published;       // per rank: the pieces of its current `share`, its own pointers
    std::vector<cudaEvent_t> ev_ready, ev_done;          // per rank, on that rank's device
    std::vector<std::vector<uint8_t>> host;              // per rank allgather_host slot
    // false when a rank aborted (now or earlier): the caller gives up instead of waiting for ever
    bool barrier() {
        std::unique_lock<std::mutex> lk(mu);
        if (aborted) return false;
        const uint64_t g = gen;
        if (++count == world) { count = 0; ++gen; cv.notify_all(); return true; }
        cv.wait(lk, [&] { return gen != g || aborted; });
        return gen != g;
    }
    void abort_all() {
        std::lock_guard<std::mutex> lk(mu);
        aborted = true;
        cv.notify_all();
    }
    void reset() {
        std::lock_guard<std::mutex> lk(mu);
        aborted = false; count = 0;
    }
};

struct LocalComm : Comm {
    std::shared_ptr<LocalState> s;
    // piece i is copied from the owner's own piece i: the ranks' arenas may be laid out differently (lk_early is decided
    // per proving key)
    int32_t share(b200zk_ctx* ctx, const CommPiece* pieces, size_t count, cudaStream_t st) override {
        if (world == 1) return B200ZK_OK;
        s->published[rank].assign(pieces, pieces + count);
        ZK_CUDA(ctx, cudaEventRecord(s->ev_ready[rank], st));
        if (!s->barrier()) return fail(ctx, B200ZK_ECUDA, "comm", "a peer rank failed");
        std::vector<char> waited(world, 0);
        for (size_t i = 0; i < count; ++i) {
            const CommPiece& p = pieces[i];
            if (p.owner == rank || p.bytes == 0) continue;
            const std::vector<CommPiece>& theirs = s->published[p.owner];
            if (theirs.size() != count || theirs[i].bytes != p.bytes) return fail(ctx, B200ZK_EINVAL, "comm", "ranks disagree on the exchange");
            if (!waited[p.owner]) { ZK_CUDA(ctx, cudaStreamWaitEvent(st, s->ev_ready[p.owner], 0)); waited[p.owner] = 1; }
            ZK_CUDA(ctx, cudaMemcpyAsync(p.ptr, theirs[i].ptr, p.bytes, cudaMemcpyDefault, st));
        }
        // nobody overwrites what it shared before every reader's copy has run
        ZK_CUDA(ctx, cudaEventRecord(s->ev_done[rank], st));
        if (!s->barrier()) return fail(ctx, B200ZK_ECUDA, "comm", "a peer rank failed");
        for (int r = 0; r < world; ++r) if (r != rank) ZK_CUDA(ctx, cudaStreamWaitEvent(st, s->ev_done[r], 0));
        return B200ZK_OK;
    }
    int32_t allgather_host(b200zk_ctx* ctx, const void* mine, size_t bytes, void* all, cudaStream_t st) override {
        ZK_CUDA(ctx, cudaStreamSynchronize(st));
        if (world == 1) { memcpy(all, mine, bytes); return B200ZK_OK; }
        s->host[rank].assign((const uint8_t*)mine, (const uint8_t*)mine + bytes);
        if (!s->barrier()) return fail(ctx, B200ZK_ECUDA, "comm", "a peer rank failed");
        for (int r = 0; r < world; ++r) {
            if (s->host[r].size() != bytes) return fail(ctx, B200ZK_EINVAL, "comm", "ranks disagree on the exchange");
            memcpy((char*)all + (size_t)r * bytes, s->host[r].data(), bytes);
        }
        if (!s->barrier()) return fail(ctx, B200ZK_ECUDA, "comm", "a peer rank failed");
        return B200ZK_OK;
    }
    void abort() override { s->abort_all(); }
};

// ------------------------------------------------------------------ one process per GPU: NCCL
struct NcclApi {
    void* handle = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclCommAbort) CommAbort = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
};

// The NCCL already in the process (torch's bundled copy has the same soname) or the system one.
static NcclApi* nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return;
        api.handle = h;
#define ZK_SYM(name) api.name = (decltype(api.name))dlsym(h, "nccl" #name)
        ZK_SYM(GetUniqueId); ZK_SYM(CommInitRank); ZK_SYM(CommDestroy); ZK_SYM(CommAbort); ZK_SYM(Broadcast); ZK_SYM(AllGather);
        ZK_SYM(GroupStart); ZK_SYM(GroupEnd); ZK_SYM(GetErrorString); ZK_SYM(GetVersion);
#undef ZK_SYM
        if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.Broadcast || !api.AllGather || !api.GroupStart || !api.GroupEnd)
            api.handle = nullptr;
    });
    return api.handle ? &api : nullptr;
}

#define ZK_NCCL(ctx, expr)                                                                          \
    do {                                                                                            \
        ncclResult_t _r = (expr);                                                                   \
        if (_r != ncclSuccess) return fail((ctx), B200ZK_ECUDA, #expr, api->GetErrorString ? api->GetErrorString(_r) : "nccl error"); \
    } while (0)

struct NcclComm : Comm {
    NcclApi* api = nullptr;
    ncclComm_t comm = nullptr;
    static constexpr size_t HOST_MAX = 16 << 10;      // bytes per rank in one all-gather: larger payloads go in pieces
    char* d_stage = nullptr;            // world * HOST_MAX
    char* h_stage = nullptr;            // pinned, same size
    ~NcclComm() override {
        if (comm && api) api->CommDestroy(comm);
        if (d_stage) cudaFree(d_stage);
        if (h_stage) cudaFreeHost(h_stage);
    }
    int32_t share(b200zk_ctx* ctx, const CommPiece* pieces, size_t count, cudaStream_t st) override {
        if (world == 1 || count == 0) return B200ZK_OK;
        ZK_NCCL(ctx, api->GroupStart());
        for (size_t i = 0; i < count; ++i) {
            if (pieces[i].bytes == 0) continue;
            ncclResult_t r = api->Broadcast(pieces[i].ptr, pieces[i].ptr, pieces[i].bytes, ncclUint8, pieces[i].owner, comm, st);
            if (r != ncclSuccess) { api->GroupEnd(); return fail(ctx, B200ZK_ECUDA, "ncclBroadcast", api->GetErrorString ? api->GetErrorString(r) : ""); }
        }
        ZK_NCCL(ctx, api->GroupEnd());
        return B200ZK_OK;
    }
    int32_t allgather_host(b200zk_ctx* ctx, const void* mine, size_t bytes, void* all, cudaStream_t st) override {
        if (world == 1 || bytes == 0) { ZK_CUDA(ctx, cudaStreamSynchronize(st)); memcpy(all, mine, bytes); return B200ZK_OK; }
        for (size_t b0 = 0; b0 < bytes; b0 += HOST_MAX) {
            const size_t m = std::min(bytes - b0, HOST_MAX), slot = (m + 15) / 16 * 16;
            memcpy(h_stage + (size_t)rank * slot, (const char*)mine + b0, m);
            ZK_CUDA(ctx, cudaMemcpyAsync(d_stage + (size_t)rank * slot, h_stage + (size_t)rank * slot, slot, cudaMemcpyHostToDevice, st));
            ZK_NCCL(ctx, api->AllGather(d_stage + (size_t)rank * slot, d_stage, slot, ncclUint8, comm, st));
            ZK_CUDA(ctx, cudaMemcpyAsync(h_stage, d_stage, slot * world, cudaMemcpyDeviceToHost, st));
            ZK_CUDA(ctx, cudaStreamSynchronize(st));
            for (int r = 0; r < world; ++r) memcpy((char*)all + (size_t)r * bytes + b0, h_stage + (size_t)r * slot, m);
        }
        return B200ZK_OK;
    }
    void abort() override {
        if (comm && api && api->CommAbort) { api->CommAbort(comm); comm = nullptr; }
    }
};

}  // namespace b200zk

using namespace b200zk;

struct b200zk_group {
    std::vector<b200zk_ctx*> ctxs;
    std::shared_ptr<LocalState> state;
};

extern "C" {

// ---- one process per GPU ---------------------------------------------------------------------
int32_t b200zk_comm_unique_id(void* id_out128) {
    if (!id_out128) return B200ZK_EINVAL;
    NcclApi* api = nccl_api();
    if (!api) return B200ZK_ENODEV;
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    if (api->GetUniqueId(&id) != ncclSuccess) return B200ZK_ECUDA;
    memcpy(id_out128, &id, 128);
    return B200ZK_OK;
}

int32_t b200zk_ctx_comm_init(b200zk_ctx* ctx, uint32_t world, uint32_t rank, const void* id128) {
    if (!ctx || !id128 || world == 0 || rank >= world) return B200ZK_EINVAL;
    if (ctx->comm) return fail(ctx, B200ZK_EINVAL, "comm_init", "this ctx already has a communicator");
    NcclApi* api = nccl_api();
    if (!api) return fail(ctx, B200ZK_ENODEV, "comm_init", "libnccl.so.2 not found");
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    NcclComm* c = new (std::nothrow) NcclComm();
    if (!c) return B200ZK_ENOMEM;
    c->api = api; c->rank = (int)rank; c->world = (int)world;
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    ncclResult_t r = api->CommInitRank(&c->comm, (int)world, id, (int)rank);
    if (r != ncclSuccess) { c->comm = nullptr; delete c; return fail(ctx, B200ZK_ECUDA, "ncclCommInitRank", api->GetErrorString ? api->GetErrorString(r) : ""); }
    if (cudaMalloc(&c->d_stage, (size_t)world * c->HOST_MAX) != cudaSuccess || cudaHostAlloc(&c->h_stage, (size_t)world * c->HOST_MAX, cudaHostAllocDefault) != cudaSuccess) {
        delete c;
        return fail(ctx, B200ZK_ENOMEM, "comm_init", "staging buffers");
    }
    ctx->comm = c;
    ctx->comm_owned = true;
    return B200ZK_OK;
}

int32_t b200zk_ctx_comm_destroy(b200zk_ctx* ctx) {
    if (!ctx) return B200ZK_EINVAL;
    if (ctx->comm && ctx->comm_owned) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); delete ctx->comm; }
    ctx->comm = nullptr; ctx->comm_owned = false;
    return B200ZK_OK;
}

uint32_t b200zk_ctx_comm_world(const b200zk_ctx* ctx) { return ctx && ctx->comm ? (uint32_t)ctx->comm->world : 1u; }
uint32_t b200zk_ctx_comm_rank(const b200zk_ctx* ctx) { return ctx && ctx->comm ? (uint32_t)ctx->comm->rank : 0u; }

// ---- one process, several GPUs -----------------------------------------------------------------
void b200zk_group_destroy(b200zk_group* g) {
    if (!g) return;
    for (size_t r = 0; r < g->ctxs.size(); ++r) {
        b200zk_ctx* ctx = g->ctxs[r];
        if (!ctx) continue;
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        delete ctx->comm; ctx->comm = nullptr;
        if (g->state) {
            if (g->state->ev_ready[r]) cudaEventDestroy(g->state->ev_ready[r]);
            if (g->state->ev_done[r]) cudaEventDestroy(g->state->ev_done[r]);
        }
        b200zk_ctx_destroy(ctx);
    }
    delete g;
}

int32_t b200zk_group_create(const int32_t* devices, uint32_t n, b200zk_group** out) {
    if (!devices || !out || n == 0 || n > 64) return B200ZK_EINVAL;
    *out = nullptr;
    b200zk_group* g = new (std::nothrow) b200zk_group();
    if (!g) return B200ZK_ENOMEM;
    g->state = std::make_shared<LocalState>();
    LocalState& s = *g->state;
    s.world = (int)n;
    s.published.resize(n);
    s.ev_ready.assign(n, nullptr); s.ev_done.assign(n, nullptr);
    s.host.resize(n);
    g->ctxs.assign(n, nullptr);
    for (uint32_t r = 0; r < n; ++r) {
        int32_t rc = b200zk_ctx_create(devices[r], &g->ctxs[r]);
        if (rc != B200ZK_OK) { b200zk_group_destroy(g); return rc; }
        if (cudaEventCreateWithFlags(&s.ev_ready[r], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&s.ev_done[r], cudaEventDisableTiming) != cudaSuccess) { b200zk_group_destroy(g); return B200ZK_ECUDA; }
        LocalComm* c = new (std::nothrow) LocalComm();
        if (!c) { b200zk_group_destroy(g); return B200ZK_ENOMEM; }
        c->rank = (int)r; c->world = (int)n; c->s = g->state;
        g->ctxs[r]->comm = c;
    }
    // direct NVLink copies between the devices of the group
    for (uint32_t a = 0; a < n; ++a)
        for (uint32_t b = 0; b < n; ++b) {
            if (devices[a] == devices[b]) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, devices[a], devices[b]) == cudaSuccess && can) {
                cudaSetDevice(devices[a]);
                cudaError_t e = cudaDeviceEnablePeerAccess(devices[b], 0);
                if (e != cudaSuccess) cudaGetLastError();          // already enabled: fine
            }
        }
    *out = g;
    return B200ZK_OK;
}

uint32_t b200zk_group_size(const b200zk_group* g) { return g ? (uint32_t)g->ctxs.size() : 0; }
b200zk_ctx* b200zk_group_ctx(b200zk_group* g, uint32_t rank) { return g && rank < g->ctxs.size() ? g->ctxs[rank] : nullptr; }
// after a failed collective call: clears the abort flag so that the group can be used again
int32_t b200zk_group_reset(b200zk_group* g) {
    if (!g) return B200ZK_EINVAL;
    g->state->reset();
    return B200ZK_OK;
}

// ---- arithmetic::best_multiexp / best_fft over the GPUs of a group (host buffers in and out) -----------------------
// best_multiexp: rank r multiplies the point range [len r / G, len (r + 1) / G) on its device (one thread per rank:
// upload of its slices, Pippenger, 64-byte result), the G partial sums are added on the host.
int32_t b200zk_group_msm(b200zk_group* g, const void* coeffs, const void* bases, size_t len, void* out_g1) {
    if (!g || !out_g1 || (len && (!coeffs || !bases))) return B200ZK_EINVAL;
    const uint32_t G = (uint32_t)g->ctxs.size();
    std::vector<int32_t> rcs(G, B200ZK_OK);
    std::vector<uint64_t> parts((size_t)G * 12, 0);
    auto body = [&](uint32_t r) {
        const size_t lo = len * r / G, hi = len * (r + 1) / G;
        rcs[r] = b200zk_msm(g->ctxs[r], (const char*)coeffs + lo * 32, (const char*)bases + lo * 64, hi - lo, parts.data() + (size_t)r * 12);
    };
    std::vector<std::thread> th;
    for (uint32_t r = 1; r < G; ++r) th.emplace_back(body, r);
    body(0);
    for (auto& t : th) t.join();
    for (uint32_t r = 0; r < G; ++r) if (rcs[r] != B200ZK_OK) { g->ctxs[0]->err = g->ctxs[r]->err; return rcs[r]; }
    return b200zk_g1_sum(parts.data(), G, out_g1);
}

namespace b200zk {
// rows [R/G][C] (k_c fastest) -> [C][R/G]: the transposed block is a strided slice of the natural-order output
__global__ void group_fft_transpose_kernel(const fe_t* in, fe_t* out, uint32_t rows, uint32_t cols) {
    __shared__ fe_t tile[8][9];
    const uint32_t c0 = blockIdx.x * 8, r0 = blockIdx.y * 8;
    uint32_t c = c0 + threadIdx.x, r = r0 + threadIdx.y;
    if (r < rows && c < cols) tile[threadIdx.y][threadIdx.x] = in[(size_t)r * cols + c];
    __syncthreads();
    c = c0 + threadIdx.y; r = r0 + threadIdx.x;
    if (r < rows && c < cols) out[(size_t)c * rows + r] = tile[threadIdx.x][threadIdx.y];
}
}  // namespace b200zk

// best_fft of 2^log_n elements as a four-step transform over the group's devices (G a power of two <= 8): rank r uploads
// its block of C / G columns, runs the R-point column transforms with the exchange fused into the kernel's store phase
// (every transformed row goes straight into its owner's buffer over NVLink), then the C-point row transforms of the R / G
// rows it received, and writes them to their natural-order positions X[k_r + R k_c] of the host array.  Small sizes
// (log_n < 16) and a group of one run on rank 0.
int32_t b200zk_group_fft(b200zk_group* g, void* a, const void* omega, uint32_t log_n) {
    if (!g || !a || !omega) return B200ZK_EINVAL;
    const uint32_t G = (uint32_t)g->ctxs.size();
    if (G == 1 || log_n < 16 || (G & (G - 1)) || G > 8) return b200zk_fft(g->ctxs[0], a, omega, log_n);
    uint32_t lw = 0; while ((1u << lw) < G) ++lw;
    const uint32_t log_r = std::min<uint32_t>(10, log_n / 2), log_c = log_n - log_r;
    const size_t R = (size_t)1 << log_r, C = (size_t)1 << log_c, cg = C / G, rg = R / G;
    const host::HFr w = host::HFr::from_limbs(omega);
    const host::HFr wc = w.pow_u64(R);                                    // omega^R: root of order C for the row step
    std::vector<fe_t*> blocks(G, nullptr), rows(G, nullptr), rows_t(G, nullptr);
    std::vector<int32_t> rcs(G, B200ZK_OK);
    g->state->reset();
    // phase 0: allocate (all pointers must exist before any rank scatters into its peers)
    for (uint32_t r = 0; r < G; ++r) {
        cudaSetDevice(g->ctxs[r]->device);
        if (cudaMalloc(&blocks[r], R * cg * sizeof(fe_t)) != cudaSuccess || cudaMalloc(&rows[r], rg * C * sizeof(fe_t)) != cudaSuccess ||
            cudaMalloc(&rows_t[r], rg * C * sizeof(fe_t)) != cudaSuccess) rcs[r] = B200ZK_ENOMEM;
    }
    bool ok = true;
    for (uint32_t r = 0; r < G; ++r) ok &= rcs[r] == B200ZK_OK;
    auto body = [&](uint32_t r) {
        b200zk_ctx* ctx = g->ctxs[r];
        cudaSetDevice(ctx->device);
        cudaStream_t st = ctx->stream;
        auto step = [&](cudaError_t e) { if (e != cudaSuccess && rcs[r] == B200ZK_OK) rcs[r] = fail(ctx, B200ZK_ECUDA, "group_fft", cudaGetErrorString(e)); };
        // column block: input element (row i, column c) sits at a[i * C + c]
        step(cudaMemcpy2DAsync(blocks[r], cg * sizeof(fe_t), (const char*)a + (size_t)r * cg * sizeof(fe_t), C * sizeof(fe_t), cg * sizeof(fe_t), R,
                               cudaMemcpyHostToDevice, st));
        if (rcs[r] == B200ZK_OK) rcs[r] = ntt_colstep_run(ctx, blocks[r], log_r, log_c - lw, (uint32_t)(r * cg), w, log_n, rows.data(), G);
        step(cudaStreamSynchronize(st));
        if (!g->state->barrier()) { if (rcs[r] == B200ZK_OK) rcs[r] = B200ZK_ECUDA; return; }      // every rank's rows have arrived
        if (rcs[r] == B200ZK_OK) rcs[r] = ntt_rows_run(ctx, rows[r], (uint32_t)rg, wc, log_c);
        dim3 grid((unsigned)((C + 7) / 8), (unsigned)((rg + 7) / 8)), block(8, 8);
        group_fft_transpose_kernel<<<grid, block, 0, st>>>(rows[r], rows_t[r], (uint32_t)rg, (uint32_t)C);
        ctx->launches++;
        // rows_t[k_c][k_r local] -> a[k_r + R k_c]
        step(cudaMemcpy2DAsync((char*)a + (size_t)r * rg * sizeof(fe_t), R * sizeof(fe_t), rows_t[r], rg * sizeof(fe_t), rg * sizeof(fe_t), C,
                               cudaMemcpyDeviceToHost, st));
        step(cudaStreamSynchronize(st));
        if (rcs[r] != B200ZK_OK) g->state->abort_all();
    };
    if (ok) {
        std::vector<std::thread> th;
        for (uint32_t r = 1; r < G; ++r) th.emplace_back(body, r);
        body(0);
        for (auto& t : th) t.join();
    }
    for (uint32_t r = 0; r < G; ++r) { cudaSetDevice(g->ctxs[r]->device); cudaFree(blocks[r]); cudaFree(rows[r]); cudaFree(rows_t[r]); }
    for (uint32_t r = 0; r < G; ++r) if (rcs[r] != B200ZK_OK) { g->ctxs[0]->err = g->ctxs[r]->err; return rcs[r]; }
    return B200ZK_OK;
}

}  // extern "C"
