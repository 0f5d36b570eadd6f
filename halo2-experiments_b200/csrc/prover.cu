// keygen_pk + create_proof on the device: halo2_proofs v2023_02_02 src/plonk/keygen.rs and
// src/plonk/prover.rs (+ lookup/permutation/vanishing provers, evaluation.rs, shplonk prover),
// the calls `full_prover` makes at /root/reference/src/circuits/utils.rs:35 and :40-48.
// The host side of this file only sequences launches, runs the Blake2b transcript between phases
// and does O(#queries) scalar work; every O(n) step is a kernel.  Step numbers refer to
// SURVEY.md §3.2.
#include "context.hpp"
#include "comm.hpp"
#include "cs_desc.hpp"
#include "expr.cuh"
#include "expr_share.hpp"
#include "prover_kernels.cuh"
#include "quot_plan.hpp"
#include "transcript.hpp"
#include <algorithm>
#include <map>
#include <new>
#include <set>
#include <chrono>
#include <string>
#include <thread>

using namespace b200zk;
using host::HAffine;
using host::HFr;

namespace b200zk {

static constexpr uint32_t PK_THREADS = 128;
static unsigned nb(size_t n, unsigned t = PK_THREADS) { return (unsigned)((n + t - 1) / t); }
static fe_t to_dev(const HFr& x) { fe_t r; memcpy(r.l, x.v, 32); return r; }

// ------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(PK_THREADS) expr_kernel(const ExprArgs a) {
    uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < a.rows) expr_eval_row(a, a.row0 + idx);
}
__global__ void __launch_bounds__(PK_THREADS) from_u512_kernel(const uint32_t* wide, fe_t* out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = from_u512_row(wide + 16 * i);
}
__global__ void __launch_bounds__(PK_THREADS) perm_den_kernel(const PermLagArgs a) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.n) perm_denominator_row(a, i);
}
__global__ void __launch_bounds__(PK_THREADS) perm_num_kernel(const PermLagArgs a) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.n) perm_numerator_row(a, i);
}
__global__ void __launch_bounds__(PK_THREADS) lookup_den_kernel(const LookupProdArgs a) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.n) lookup_den_row(a, i);
}
__global__ void __launch_bounds__(PK_THREADS) lookup_num_kernel(const LookupProdArgs a) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.n) lookup_num_row(a, i);
}
__global__ void __launch_bounds__(PK_THREADS) quot_perm_a_kernel(const QuotPermAArgs a) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.rows) quot_perm_a_row(a, a.row0 + i);
}
__global__ void __launch_bounds__(PK_THREADS) quot_perm_b_kernel(const QuotPermBArgs a) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.rows) quot_perm_b_row(a, a.row0 + i);
}
__global__ void __launch_bounds__(PK_THREADS) quot_lookup_kernel(const QuotLookupArgs a) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < a.rows) quot_lookup_row(a, a.row0 + i);
}
__global__ void __launch_bounds__(PK_THREADS) coset_interpolate_kernel(const fe_t* g, const fe_t* inv_pow, const fe_t* vinv, uint32_t C, size_t n, fe_t* out, const fe_t* extra,
                                                                      const fe_t* lin) {
    size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) coset_interpolate_row(g, inv_pow, vinv, C, n, out, r, extra, lin);
}
__global__ void __launch_bounds__(PK_THREADS) lookup_extrapolate_kernel(fe_t* g, const fe_t* inv_pow, const fe_t* lambda, const fe_t* tinv, uint32_t CL, uint32_t C, size_t n) {
    size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) lookup_extrapolate_row(g, inv_pow, lambda, tinv, CL, C, n, r);
}
__global__ void __launch_bounds__(PK_THREADS) fold_pieces_kernel(const fe_t* pieces, uint32_t npieces, size_t n, const fe_t xn, fe_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) fold_pieces_row(pieces, npieces, n, xn, out, i);
}
__global__ void __launch_bounds__(PK_THREADS) axpy_kernel(fe_t* acc, const fe_t* p, const fe_t s, size_t n, int init) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) axpy_row(acc, p, s, i, init != 0);
}
__global__ void __launch_bounds__(PK_THREADS) scale_kernel(fe_t* a, const fe_t s, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) scale_row(a, s, i);
}
// acc[i] = (init ? 0 : acc[i]) + sum_j s[j] * p[j][i] for up to 16 polynomials per launch: the linear combinations of
// SHPLONK (A_i = sum_j y^j P_ij over the ~50 polynomials opened at x alone) read every polynomial once and touch the
// accumulator once per 16 of them, instead of one axpy launch (and one accumulator round trip) per polynomial.
struct LinCombArgs { const fe_t* p[16]; fe_t s[16]; uint32_t m; };
__global__ void __launch_bounds__(PK_THREADS) lincomb_kernel(fe_t* acc, const LinCombArgs a, size_t n, int init) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe_t t = init ? Fr::zero() : acc[i];
    for (uint32_t j = 0; j < a.m; ++j) { fe_t v = a.p[j][i]; t = Fr::add(t, Fr::mul(v, a.s[j])); }
    acc[i] = t;
}
struct LowCoeffs { fe_t c[8]; uint32_t m; };
__global__ void sub_low_kernel(fe_t* a, const LowCoeffs lc) {
    uint32_t i = threadIdx.x;
    if (i < lc.m) { fe_t v = a[i]; a[i] = Fr::sub(v, lc.c[i]); }
}
__global__ void __launch_bounds__(PK_THREADS) one_minus_sum_kernel(const fe_t* a, const fe_t* b, fe_t* out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) one_minus_sum_row(a, b, out, i);
}
__global__ void __launch_bounds__(PK_THREADS) sigma_kernel(const uint32_t* mc, const uint32_t* mr, const fe_t* dp, const fe_t* op, fe_t* out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sigma_row(mc, mr, dp, op, out, i);
}


}  // namespace b200zk

// ------------------------------------------------------------------ proving key
struct b200zk_pk {
    b200zk_ctx* ctx = nullptr;
    b200zk_params* params = nullptr;
    b200zk_domain* dom = nullptr;
    CsDesc cs;
    uint32_t n = 0, ext_n = 0, S = 0, chunk = 0, q = 0, L = 0, P = 0;
    fe_t *fixed_values = nullptr, *fixed_polys = nullptr, *fixed_cosets = nullptr;
    fe_t *perm_values = nullptr, *perm_polys = nullptr, *perm_cosets = nullptr;
    fe_t *l0 = nullptr, *l_last = nullptr, *l_active = nullptr;
    fe_t* omega_pows = nullptr;
    // quotient cosets c_j = zeta * extended_omega^j, j < q (see prover_kernels.cuh): ext_n = q * n
    fe_t *coset_pow = nullptr, *coset_pow_inv = nullptr;      // c_j^r and c_j^-r, [q][n]
    fe_t *coset_fac = nullptr, *vinv = nullptr;               // extended_omega^j [q]; inverse Vandermonde of c_j^n [q*q]
    std::vector<HFr> coset_t;                                  // 1 / (c_j^n - 1): the vanishing polynomial on coset j
    // lookup terms and low-degree gates on lk_cosets_n = plan.low < q cosets (prover_kernels.cuh, lookup_extrapolate_row);
    // == q: not split (no lookups, or lookups of the full degree)
    uint32_t lk_cosets_n = 0;
    QuotPlan plan;
    // lookup cosets and table values of ALL lookups kept side by side (4 arrays of lk_cosets_n * n per lookup), so that they
    // are computed on the side stream while the transcript-bound phases run; false = one lookup at a time after y (less memory)
    bool lk_early = false;
    fe_t* lk_lambda = nullptr;                                 // extrapolation weights [(q - CL) x CL]
    // device program data
    uint32_t* d_prog = nullptr;                       // gate programs of the three classes (quot_plan.hpp) | lookup programs
    std::pair<uint32_t, uint32_t> gate_prog[3] = {};             // (off, len) into d_prog, by class
    std::vector<uint32_t> gate_exp;                   // gate i enters the accumulator of its class with weight y^gate_exp[i]
    fe_t* d_wts = nullptr;                            // those weights for the current proof (ExprArgs::wts)
    fe_t* h_wts = nullptr;                            // their pinned staging buffer
    std::vector<std::pair<uint32_t, uint32_t>> lookup_prog;     // (off, len) into d_prog
    fe_t* d_consts = nullptr;
    int32_t *d_q_adv = nullptr, *d_q_fix = nullptr, *d_q_inst = nullptr;
    const fe_t** d_ptrs = nullptr;                    // pointer tables, see PtrTab
    char* arena = nullptr;
    size_t arena_bytes = 0;
    uint32_t* d_err = nullptr;
    float phase_ms[7] = {0, 0, 0, 0, 0, 0, 0};
    struct TimerEv { cudaEvent_t e0, e1; int slot; };
    std::vector<TimerEv> timer_events;                // pool, grown on demand
    size_t timer_used = 0;
    std::vector<void*> owned;
    // upload pipeline of create_proof: the advice columns arrive on copy_stream one by one (H2D from the caller's
    // buffers, or D2D), col_events[c] marks column c complete (blinding rows included)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_rnd = nullptr;
    std::vector<cudaEvent_t> col_events;
    std::map<std::string, std::pair<const void*, size_t>> dbg;     // buffers of the last proof, for b200zk_pk_debug_buffer
    std::vector<std::pair<const char*, double>> trace;             // host time (ms since the call) at the proof's synchronisation points
};

namespace b200zk {

// pointer tables in d_ptrs: [fixed_values F][fixed_cosets F][advice_values A][advice_cosets A][inst_values I][inst_cosets I]
struct PtrTab {
    uint32_t F, A, I;
    uint32_t fixed_values() const { return 0; }
    uint32_t fixed_cosets() const { return F; }
    uint32_t advice_values() const { return 2 * F; }
    uint32_t advice_cosets() const { return 2 * F + A; }
    uint32_t inst_values() const { return 2 * F + 2 * A; }
    uint32_t inst_cosets() const { return 2 * F + 2 * A + I; }
    uint32_t total() const { return 2 * (F + A + I); }
};

template <class T> static int32_t dev_alloc(b200zk_pk* pk, T** p, size_t count) {
    cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T));
    if (e != cudaSuccess) return fail(pk->ctx, B200ZK_ENOMEM, "cudaMalloc(pk)", cudaGetErrorString(e));
    pk->owned.push_back(*p);
    return B200ZK_OK;
}

struct Arena {
    char* base; size_t cap, off = 0; bool ok = true;
    template <class T> T* take(size_t count) {
        size_t bytes = (count * sizeof(T) + 255) / 256 * 256;
        if (off + bytes > cap) { ok = false; return nullptr; }
        T* p = (T*)(base + off); off += bytes; return p;
    }
};

// Where create_proof reads the caller's rng stream: one 64-byte draw per Fr::random of upstream create_proof, in its call
// order (SURVEY.md §8(a7)).  Upstream also draws a Blind for every commitment, which KZG does not use: those draws are
// gaps, drawn by the caller and never read.
struct DrawLayout {
    size_t bf1, advice, advice_blinds, lookups, sets, lk_products, random, random_blind, h_blinds, total;
    explicit DrawLayout(const b200zk_pk* pk) : bf1(pk->cs.bf + 1) {
        advice = 0;                                        // bf + 1 blinding rows per advice column
        advice_blinds = advice + pk->cs.A * bf1;           // gap: a Blind per advice column
        lookups = advice_blinds + pk->cs.A;                // per lookup: bf + 1 rows of the permuted input, bf + 1 of the permuted table, 2 Blinds (gap)
        sets = lookups + pk->L * (2 * bf1 + 2);            // per permutation set: bf blinding rows of its product, a Blind (gap)
        lk_products = sets + pk->S * bf1;                  // per lookup: bf blinding rows of its product, a Blind (gap)
        random = lk_products + pk->L * bf1;                // the n coefficients of the vanishing argument's random polynomial
        random_blind = random + pk->n;                     // gap
        h_blinds = random_blind + 1;                       // gap: a Blind per piece of h
        total = h_blinds + pk->q;
    }
    size_t advice_rows(uint32_t c) const { return advice + c * bf1; }
    size_t lookup_input_rows(uint32_t l) const { return lookups + l * (2 * bf1 + 2); }
    size_t lookup_table_rows(uint32_t l) const { return lookup_input_rows(l) + bf1; }
    size_t set_rows(uint32_t s) const { return sets + s * bf1; }
    size_t lookup_product_rows(uint32_t l) const { return lk_products + l * bf1; }
};

static size_t arena_need(const b200zk_pk* pk) {
    size_t n = pk->n, ext = pk->ext_n, A = pk->cs.A, I = pk->cs.I, L = pk->L, S = pk->S;
    size_t draws = DrawLayout(pk).total;
    size_t elems = 2 * A * n + 2 * I * n + draws + 7 * L * n + S * n + S * ext + 3 * n   // columns, lookups, perm, tmp
                   + ext * (1 + A + I + 4 + 1)                                            // h, cosets, lookup cosets + table_value, h_L
                   + n * (1 + 8 + 4 + 8 + 1);                                                 // h_poly, shplonk set sums, hx/lx/tmp, per-set quotients, linear gates
    if (pk->lk_early) elems += 4 * L * (size_t)pk->lk_cosets_n * n + 64;
    return elems * sizeof(fe_t) + (size_t)draws * 64 + (64 << 10);
}

// Per-phase device time without extra synchronisation: event pairs from a pool owned by the pk are
// recorded around each phase and summed once at the end of the proof (phase_timers_collect).
struct PhaseTimer {
    b200zk_pk* pk; size_t idx;
    PhaseTimer(b200zk_pk* pk_, int slot) : pk(pk_) {
        idx = pk->timer_used++;
        if (idx >= pk->timer_events.size()) {
            cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
            pk->timer_events.push_back({a, b, slot});
        }
        pk->timer_events[idx].slot = slot;
        cudaEventRecord(pk->timer_events[idx].e0, pk->ctx->stream);
    }
    ~PhaseTimer() { cudaEventRecord(pk->timer_events[idx].e1, pk->ctx->stream); }
};
static void phase_timers_collect(b200zk_pk* pk) {
    cudaStreamSynchronize(pk->ctx->stream);
    for (size_t i = 0; i < pk->timer_used; ++i) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, pk->timer_events[i].e0, pk->timer_events[i].e1) == cudaSuccess) pk->phase_ms[pk->timer_events[i].slot] += ms;
    }
    pk->timer_used = 0;
}
enum { PH_MSM = 0, PH_NTT = 1, PH_QUOT = 2, PH_LOOKUP = 3, PH_PERM = 4, PH_OPEN = 5, PH_OTHER = 6 };

static int cmp_canonical(const HFr& a, const HFr& b) {
    uint64_t x[4], y[4]; a.to_canonical(x); b.to_canonical(y);
    for (int i = 3; i >= 0; --i) if (x[i] != y[i]) return x[i] < y[i] ? -1 : 1;
    return 0;
}
struct FrLess { bool operator()(const HFr& a, const HFr& b) const { return cmp_canonical(a, b) < 0; } };

// arithmetic::lagrange_interpolate (host, <= 8 points): the unique polynomial of degree < m
static std::vector<HFr> lagrange_interpolate(const std::vector<HFr>& pts, const std::vector<HFr>& evals) {
    size_t m = pts.size();
    std::vector<HFr> poly(m, HFr::zero());
    for (size_t j = 0; j < m; ++j) {
        std::vector<HFr> num(1, HFr::one());
        HFr den = HFr::one();
        for (size_t k = 0; k < m; ++k) {
            if (k == j) continue;
            std::vector<HFr> nw(num.size() + 1, HFr::zero());
            for (size_t i = 0; i < num.size(); ++i) { nw[i] = nw[i] - num[i] * pts[k]; nw[i + 1] = nw[i + 1] + num[i]; }
            num.swap(nw);
            den = den * (pts[j] - pts[k]);
        }
        HFr s = evals[j] * den.inv();
        for (size_t i = 0; i < num.size(); ++i) poly[i] = poly[i] + num[i] * s;
    }
    return poly;
}
static HFr eval_small(const std::vector<HFr>& poly, const HFr& x) {
    HFr acc = HFr::zero();
    for (size_t i = poly.size(); i-- > 0;) acc = acc * x + poly[i];
    return acc;
}
static HFr rotate_omega(const b200zk_domain* d, const HFr& x, int rot) {
    return rot >= 0 ? x * d->omega.pow_u64((uint64_t)rot) : x * d->omega_inv.pow_u64((uint64_t)(-(int64_t)rot));
}

// Side-stream section: between construction and destruction every launch that goes through
// ctx->stream (NTTs, phase timers) lands on the low-priority side stream, ordered after everything
// the main stream has enqueued so far; the main stream consumes the results after waiting for
// ctx->ev_join (re-recorded at the end of every section; the side stream is in-order, so the last
// record covers all earlier sections).
struct SideStream {
    b200zk_ctx* ctx;
    explicit SideStream(b200zk_ctx* c) : ctx(c) {
        cudaEventRecord(ctx->ev_fork, ctx->stream);
        cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0);
        std::swap(ctx->stream, ctx->stream2);
        std::swap(ctx->ntt_scratch, ctx->ntt_scratch2);
    }
    ~SideStream() {
        cudaEventRecord(ctx->ev_join, ctx->stream);
        std::swap(ctx->stream, ctx->stream2);
        std::swap(ctx->ntt_scratch, ctx->ntt_scratch2);
    }
};

// several full-length columns in one batched launch sequence (msm_run_multi), <= 24 at a time
static int32_t commit_multi_dev(b200zk_pk* pk, const std::vector<const fe_t*>& cols, size_t len, bool lagrange, std::vector<HAffine>& outs) {
    PhaseTimer t(pk, PH_MSM);
    outs.resize(cols.size());
    for (size_t b = 0; b < cols.size(); b += 24) {
        uint32_t m = (uint32_t)std::min<size_t>(24, cols.size() - b);
        ZK_TRY(params_commit_multi(pk->params, cols.data() + b, m, len, lagrange, outs.data() + b));
    }
    return B200ZK_OK;
}
// inverse NTT of `count` contiguous size-n columns in place, every output multiplied by `factor`; more than one column
// runs as one launch per pass
static int32_t intt_scaled(b200zk_pk* pk, fe_t* d_a, uint32_t count, const HFr& factor) {
    HFr post[3] = {factor, factor, factor};
    if (count == 1) return ntt_run(pk->ctx, d_a, pk->n, d_a, pk->dom->k, pk->dom->omega_inv, nullptr, post);
    return ntt_rows_run(pk->ctx, d_a, count, pk->dom->omega_inv, pk->dom->k, post);
}
// `count` contiguous Lagrange columns to coefficient form
static int32_t lagrange_to_coeff(b200zk_pk* pk, fe_t* d_a, uint32_t count = 1) {
    PhaseTimer t(pk, PH_NTT);
    pk->ctx->ntt_sparse_hint = true;
    int32_t rc = intt_scaled(pk, d_a, count, pk->dom->ifft_divisor);
    pk->ctx->ntt_sparse_hint = false;
    return rc;
}
// coeff_to_extended restricted to the q cosets the quotient needs: coset j = size-n NTT of a_r * c_j^r
static int32_t coeff_to_extended(b200zk_pk* pk, const fe_t* d_coeffs, fe_t* d_out, uint32_t cosets = 0) {
    PhaseTimer t(pk, PH_NTT);
    return ntt_run_cosets(pk->ctx, d_coeffs, d_out, pk->dom->k, pk->dom->omega, pk->coset_pow, cosets ? cosets : pk->q);
}

static ExprArgs expr_args(const b200zk_pk* pk, uint32_t prog_off, uint32_t prog_len, bool extended, uint32_t mode,
                          const HFr ch[4], fe_t* out0, fe_t* out1) {
    PtrTab pt{pk->cs.F, pk->cs.A, pk->cs.I};
    ExprArgs a{};
    a.prog = pk->d_prog + prog_off; a.prog_len = prog_len; a.consts = pk->d_consts;
    a.fixed = pk->d_ptrs + (extended ? pt.fixed_cosets() : pt.fixed_values());
    a.advice = pk->d_ptrs + (extended ? pt.advice_cosets() : pt.advice_values());
    a.instance = pk->d_ptrs + (extended ? pt.inst_cosets() : pt.inst_values());
    a.q_fixed = pk->d_q_fix; a.q_advice = pk->d_q_adv; a.q_instance = pk->d_q_inst;
    a.log_size = pk->dom->k;
    a.rows = extended ? pk->ext_n : pk->n;
    a.rot_scale = 1u;
    for (int i = 0; i < 4; ++i) a.factors[i] = to_dev(ch[i]);
    a.wts = pk->d_wts;
    a.mode = mode; a.out0 = out0; a.out1 = out1;
    return a;
}

// ------------------------------------------------------------------ one proof over several ranks
// Rank layout of a sharded create_proof (comm.hpp).  G = 1 degenerates to the single-GPU prover: every
// `mine` test is true, every range is the whole, every exchange is a no-op.
struct Shard {
    Comm* cm; int G, R; uint32_t q;
    explicit Shard(b200zk_pk* pk) : cm(pk->ctx->comm), G(cm ? cm->world : 1), R(cm ? cm->rank : 0), q(pk->q) {}
    bool on() const { return G > 1; }
    // columns / lookups / permutation sets round-robin
    int owner(uint32_t i) const { return (int)(i % (uint32_t)G); }
    bool mine(uint32_t i) const { return owner(i) == R; }
    // quotient cosets in contiguous blocks: rank r evaluates cosets [coset_lo(r), coset_lo(r + 1))
    uint32_t coset_lo(int r) const { return (uint32_t)((uint64_t)q * (uint32_t)r / (uint32_t)G); }
    int coset_owner(uint32_t j) const { for (int r = 0; r < G; ++r) if (j >= coset_lo(r) && j < coset_lo(r + 1)) return r; return 0; }
    // point range of a dense commit
    size_t pt_lo(size_t len, int r) const { return len * (size_t)r / (size_t)G; }
    // Lookup arguments and permutation sets go to the least loaded rank, the load being what a rank already carries for its
    // quotient cosets (q is rarely a multiple of G: with 8 ranks and 5 cosets three ranks own none and would otherwise idle
    // through half of the proof).  Weights are in units of one size-n transform: a coset costs its column extensions plus the
    // quotient kernels, a lookup its sort, grand product, three transforms and commitments, a permutation set its product.
    // Measured on 8 GPUs (MST k = 20): round-robin 39.2 ms; this placement — all 8 lookups and the 4 sets on the three ranks
    // without a coset — 36.5 ms; weighting only the work before the challenge y (2 + 2 + 2 lookups on those ranks, 1 + 1 and the
    // sets on coset owners) 38.0 ms: the coset owners are the busy ranks from start to end, anything added to them costs.
    std::vector<int> lk_own, set_own;
    void assign(uint32_t L, uint32_t S, uint32_t columns) {
        std::vector<uint64_t> load((size_t)G, 0);
        const uint64_t w_coset = columns + 30, w_lookup = 15, w_set = 8;
        for (int r = 0; r < G; ++r) load[r] = (uint64_t)(coset_lo(r + 1) - coset_lo(r)) * w_coset;
        auto lightest = [&]() { int b = 0; for (int r = 1; r < G; ++r) if (load[r] < load[b]) b = r; return b; };
        lk_own.resize(L); set_own.resize(S);
        for (uint32_t l = 0; l < L; ++l) { int r = lightest(); lk_own[l] = r; load[r] += w_lookup; }
        for (uint32_t t = 0; t < S; ++t) { int r = lightest(); set_own[t] = r; load[r] += w_set; }
    }
    int lk_owner(uint32_t l) const { return lk_own[l]; }
    bool lk_mine(uint32_t l) const { return lk_own[l] == R; }
    int set_owner(uint32_t t) const { return set_own[t]; }
    bool set_mine(uint32_t t) const { return set_own[t] == R; }
    // Every rank fills the entries v[i] it owns (owner_of(i) == R); on return every rank holds all of them.  One host
    // exchange (it synchronises the stream); nothing to do on one rank.
    template <class T, class OwnerOf> int32_t gather(b200zk_pk* pk, std::vector<T>& v, OwnerOf owner_of) const {
        if (G == 1) return B200ZK_OK;
        std::vector<size_t> slot(v.size()), used((size_t)G, 0);
        for (size_t i = 0; i < v.size(); ++i) slot[i] = used[owner_of(i)]++;
        const size_t per = *std::max_element(used.begin(), used.end());
        std::vector<T> mine(per), all(per * G);
        for (size_t i = 0; i < v.size(); ++i) if (owner_of(i) == R) mine[slot[i]] = v[i];
        PhaseTimer t(pk, PH_OTHER);
        ZK_TRY(cm->allgather_host(pk->ctx, mine.data(), per * sizeof(T), all.data(), pk->ctx->stream));
        for (size_t i = 0; i < v.size(); ++i) v[i] = all[(size_t)owner_of(i) * per + slot[i]];
        return B200ZK_OK;
    }
};

// Commitments to `cols`, column i computed by rank owners[i]; every rank ends up with all of them.  `flag` (optional)
// is OR-ed over the ranks in the same exchange (the lookup permutation's "input not in table" bit).
static int32_t commit_multi_split(b200zk_pk* pk, const Shard& sh, const std::vector<const fe_t*>& cols, const std::vector<int>& owners,
                                  size_t len, bool lagrange, std::vector<HAffine>& outs, uint32_t* flag = nullptr) {
    const size_t m = cols.size();
    std::vector<const fe_t*> my;
    for (size_t i = 0; i < m; ++i) if (owners[i] == sh.R) my.push_back(cols[i]);
    std::vector<HAffine> mp;
    ZK_TRY(commit_multi_dev(pk, my, len, lagrange, mp));
    outs.assign(m + sh.G, HAffine{});                                 // the points, then one entry per rank for its flag
    for (size_t i = 0, j = 0; i < m; ++i) if (owners[i] == sh.R) outs[i] = mp[j++];
    if (flag) memcpy(&outs[m + sh.R], flag, 4);
    ZK_TRY(sh.gather(pk, outs, [&](size_t i) { return i < m ? owners[i] : (int)(i - m); }));
    if (flag) for (int r = 0; r < sh.G; ++r) { uint32_t f; memcpy(&f, &outs[m + r], 4); *flag |= f; }
    outs.resize(m);
    return B200ZK_OK;
}

// Dense commitments sharded by point range (SURVEY.md 8(e)2): every rank multiplies its slice [lo, hi) of every
// column, the G partial sums per column are exchanged (64 bytes each) and added on the host.
static int32_t commit_multi_range(b200zk_pk* pk, const Shard& sh, const std::vector<const fe_t*>& cols, size_t len, bool lagrange,
                                  std::vector<HAffine>& outs) {
    const uint32_t m = (uint32_t)cols.size();
    std::vector<HAffine> part((size_t)m * sh.G);                      // entry (r, i): rank r's sum for column i
    {
        PhaseTimer t(pk, PH_MSM);
        ZK_TRY(params_commit_range(pk->params, cols.data(), m, sh.pt_lo(len, sh.R), sh.pt_lo(len, sh.R + 1), lagrange, part.data() + (size_t)sh.R * m));
    }
    ZK_TRY(sh.gather(pk, part, [&](size_t i) { return (int)(i / m); }));
    outs.resize(m);
    for (uint32_t i = 0; i < m; ++i) {
        host::HXyzz acc = host::hx_identity();
        for (int r = 0; r < sh.G; ++r) {
            const HAffine& a = part[(size_t)r * m + i];
            if (!(a.x.is_zero() && a.y.is_zero())) acc = host::hx_add(acc, host::hx_from_affine(a));
        }
        outs[i] = host::hx_to_affine(acc);
    }
    return B200ZK_OK;
}

// ------------------------------------------------------------------ create_proof
// One create_proof on this rank: the state its steps (SURVEY.md §3.2) share.  prove() calls the steps in order and squeezes
// the challenges between them.
struct Prover {
    b200zk_pk* pk;
    b200zk_ctx* ctx = pk->ctx;
    const CsDesc& cs = pk->cs;
    const b200zk_domain* dom = pk->dom;
    cudaStream_t st = ctx->stream;
    Shard sh{pk};
    const DrawLayout dl{pk};
    const bool advice_on_device;
    // Sharded proof from host buffers: the host -> device traffic is split as well — every rank uploads 1/G of the rng
    // stream and its own advice columns over its PCIe link, and the ranks exchange them over NVLink.
    const bool split_upload;
    const size_t n = pk->n, ext = pk->ext_n;
    const uint32_t A = cs.A, I = cs.I, F = cs.F, L = pk->L, S = pk->S, bf = cs.bf;
    const size_t usable = n - (bf + 1);
    const uint32_t CL = pk->lk_cosets_n;                          // == q unless the lookup terms and the low gates run on fewer cosets
    const bool lk_split = CL < pk->q;
    const uint32_t cj0 = sh.coset_lo(sh.R), cj1 = sh.coset_lo(sh.R + 1);       // quotient cosets this rank extends and evaluates
    const uint32_t lj0 = std::min(cj0, CL), lj1 = std::min(cj1, CL);           // this rank's share of the cosets the lookup terms run on
    const uint32_t lk_row0 = lj0 * (uint32_t)n, lk_rows = (lj1 - lj0) * (uint32_t)n;
    const std::chrono::steady_clock::time_point t_start = std::chrono::steady_clock::now();
    host::Transcript tr;
    HFr ch[4] = {HFr::zero(), HFr::zero(), HFr::zero(), HFr::zero()};   // theta, beta, gamma, y
    HFr x;                                                        // the opening point
    HAffine random_pt = {host::HFq::zero(), host::HFq::zero()};
    // arena buffers, see carve
    fe_t *advice_values, *advice_polys, *inst_values, *inst_polys, *rnd, *lk_bufs, *perm_polys, *perm_cosets, *tmp_n, *h;
    fe_t *advice_cosets, *inst_cosets, *lk_cosets, *h_lk, *h_lin, *lk_all, *h_poly, *set_sums, *set_quot, *hx, *lx, *t0, *t1;
    uint32_t* wide;
    // openings: every (polynomial, point) pair in multiopen order, its distinct pairs and their values
    struct Query { const fe_t* poly; HFr point; };
    std::vector<Query> queries, pairs;
    std::vector<HFr> values;
    // SHPLONK's rotation sets, the low-degree equivalent of each of their polynomials, all points
    struct RotSet { std::vector<HFr> pts; std::vector<const fe_t*> polys; };
    std::vector<RotSet> rot_sets;
    std::vector<std::vector<std::vector<HFr>>> low;
    std::set<HFr, FrLess> super_points;

    Prover(b200zk_pk* p, bool advice_dev, bool rng_dev) : pk(p), advice_on_device(advice_dev), split_upload(sh.on() && !advice_dev && !rng_dev) { sh.assign(L, S, A + I + S + 3 * L); }

    // arrays of lookup l: LK as listed at lk_bufs; LKC product z, permuted input a', permuted table s', table value
    // (all indexed by global coset row)
    fe_t* LK(uint32_t l, uint32_t which) const { return lk_bufs + ((size_t)l * 7 + which) * n; }
    fe_t* LKC(uint32_t l, uint32_t which) const {
        return pk->lk_early ? lk_all + ((size_t)l * 4 + which) * CL * n : lk_cosets + (size_t)which * ext;
    }
    // column idx of type 0 advice, 1 fixed, 2 instance: its values, its quotient cosets
    const fe_t* column_values(uint32_t type, uint32_t idx) const { return (type == 0 ? advice_values : type == 1 ? pk->fixed_values : inst_values) + (size_t)idx * n; }
    const fe_t* column_cosets(uint32_t type, uint32_t idx) const { return (type == 0 ? advice_cosets : type == 1 ? pk->fixed_cosets : inst_cosets) + (size_t)idx * ext; }
    bool lin_mine() const { return pk->gate_prog[QC_LINEAR].second && sh.coset_owner(0) == sh.R; }

    void mark(const char* label) {                  // called right after a host synchronisation: where the wall clock of the proof goes
        pk->trace.push_back({label, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count()});
    }
    cudaError_t copy_rows(fe_t* dst, const fe_t* src, size_t count) {
        return cudaMemcpyAsync(dst, src, count * sizeof(fe_t), cudaMemcpyDeviceToDevice, st);
    }
    int32_t share(const std::vector<CommPiece>& pieces) {
        if (sh.G == 1 || pieces.empty()) return B200ZK_OK;
        PhaseTimer t(pk, PH_OTHER);
        return sh.cm->share(ctx, pieces.data(), pieces.size(), ctx->stream);
    }
    int32_t my_cosets(const fe_t* d_coeffs, fe_t* d_out, uint32_t j0, uint32_t j1) {     // cosets [j0, j1) of d_out
        if (j0 >= j1) return B200ZK_OK;
        PhaseTimer t(pk, PH_NTT);
        return ntt_run_cosets(ctx, d_coeffs, d_out + (size_t)j0 * n, dom->k, dom->omega, pk->coset_pow + (size_t)j0 * n, j1 - j0);
    }
    // Lagrange commitments to `cols`, column i computed by rank owners[i], into the transcript
    int32_t commit_columns(const std::vector<const fe_t*>& cols, const std::vector<int>& owners, const char* label, uint32_t* flag = nullptr) {
        std::vector<HAffine> pts;
        ZK_TRY(commit_multi_split(pk, sh, cols, owners, n, true, pts, flag));
        for (auto& pt : pts) tr.write_point(pt);
        mark(label);
        return B200ZK_OK;
    }
    int32_t commit_random() {
        std::vector<HAffine> pts;
        ZK_TRY(commit_multi_range(pk, sh, {rnd + dl.random}, n, false, pts));
        random_pt = pts[0];
        return B200ZK_OK;
    }
    void lookup_table_value(uint32_t l) {            // (compressed input + beta)(compressed table + gamma) on this rank's lookup cosets
        PhaseTimer t(pk, PH_QUOT);
        ExprArgs ea = expr_args(pk, pk->lookup_prog[l].first, pk->lookup_prog[l].second, true, EXM_LOOKUP_PROD, ch, LKC(l, 3), nullptr);
        ea.row0 = lk_row0; ea.rows = lk_rows;
        expr_kernel<<<nb(lk_rows), PK_THREADS, 0, ctx->stream>>>(ea);
        ctx->launches++;
    }
    // one gate program per class, each on its own rows (quot_plan.hpp); a class without gates starts its accumulator at 0
    int32_t gate_class(uint32_t cls, fe_t* out, uint32_t row0, uint32_t rows) {
        if (!rows) return B200ZK_OK;
        PhaseTimer t(pk, PH_QUOT);
        if (!pk->gate_prog[cls].second) {
            ZK_CUDA(ctx, cudaMemsetAsync(out + row0, 0, (size_t)rows * sizeof(fe_t), st));
            return B200ZK_OK;
        }
        ExprArgs ea = expr_args(pk, pk->gate_prog[cls].first, pk->gate_prog[cls].second, true, EXM_ACC0, ch, out, nullptr);
        ea.row0 = row0; ea.rows = rows;
        expr_kernel<<<nb(rows), PK_THREADS, 0, st>>>(ea);
        ctx->launches++;
        return B200ZK_OK;
    }
    int32_t opened(const fe_t* poly, const HFr& pt, HFr* out) const {
        for (size_t i = 0; i < pairs.size(); ++i)
            if (pairs[i].poly == poly && pairs[i].point == pt) { *out = values[i]; return B200ZK_OK; }
        return fail(ctx, B200ZK_EINVAL, "create_proof", "internal: evaluation of a pair that is not opened");
    }
    int32_t write_eval(const fe_t* poly, const HFr& pt) {
        HFr e = HFr::zero();
        ZK_TRY(opened(poly, pt, &e));
        tr.write_scalar(e);
        return B200ZK_OK;
    }

    int32_t carve() {
        Arena ar{pk->arena, pk->arena_bytes};
        advice_values = ar.take<fe_t>(A * n);
        advice_polys = ar.take<fe_t>(A * n);
        inst_values = ar.take<fe_t>(I * n);
        inst_polys = ar.take<fe_t>(I * n);
        wide = ar.take<uint32_t>(dl.total * 16);
        rnd = ar.take<fe_t>(dl.total);                                // the rng stream as field elements, laid out as dl says
        lk_bufs = ar.take<fe_t>(7 * (size_t)L * n);                   // per lookup: cin ctab pin ptab pin_poly ptab_poly z_poly
        perm_polys = ar.take<fe_t>((size_t)S * n);
        perm_cosets = ar.take<fe_t>((size_t)S * ext);
        tmp_n = ar.take<fe_t>(3 * n);
        h = ar.take<fe_t>(ext);
        advice_cosets = ar.take<fe_t>(A * ext);
        inst_cosets = ar.take<fe_t>(I * ext);
        lk_cosets = ar.take<fe_t>(4 * ext);                           // z, a', s', table_value; after vanishing_construct the q pieces of h
        h_lk = ar.take<fe_t>(ext);                                    // lookup and low-degree gate part of the quotient when it runs on fewer cosets
        h_lin = ar.take<fe_t>(n);                                     // linear gates on coset 0
        lk_all = pk->lk_early ? ar.take<fe_t>(4 * (size_t)L * CL * n) : nullptr;    // the lookup cosets of all lookups side by side
        h_poly = ar.take<fe_t>(n);
        set_sums = ar.take<fe_t>(8 * n);
        fe_t* sh_tmp = ar.take<fe_t>(4 * n);                          // SHPLONK work space: hx lx t0 t1
        set_quot = ar.take<fe_t>(8 * n);                              // SHPLONK: Q_i of every rotation set, computed by its owner
        if (!ar.ok) return fail(ctx, B200ZK_ENOMEM, "create_proof", "arena too small");
        hx = sh_tmp; lx = sh_tmp + n; t0 = sh_tmp + 2 * n; t1 = sh_tmp + 3 * n;
        pk->dbg.clear();
        pk->dbg["advice_values"] = {advice_values, A * n}; pk->dbg["advice_polys"] = {advice_polys, A * n};
        pk->dbg["lookups"] = {lk_bufs, 7 * (size_t)L * n}; pk->dbg["perm_polys"] = {perm_polys, (size_t)S * n};
        pk->dbg["h"] = {h, ext}; pk->dbg["rnd"] = {rnd, dl.total}; pk->dbg["tmp_n"] = {tmp_n, 3 * n};
        pk->dbg["advice_cosets"] = {advice_cosets, A * ext}; pk->dbg["h_poly"] = {h_poly, n};

        // pointer tables for this proof
        PtrTab pt{F, A, I};
        std::vector<const fe_t*> tab(pt.total());
        for (uint32_t c = 0; c < F; ++c) { tab[pt.fixed_values() + c] = pk->fixed_values + (size_t)c * n; tab[pt.fixed_cosets() + c] = pk->fixed_cosets + (size_t)c * ext; }
        for (uint32_t c = 0; c < A; ++c) { tab[pt.advice_values() + c] = advice_values + (size_t)c * n; tab[pt.advice_cosets() + c] = advice_cosets + (size_t)c * ext; }
        for (uint32_t c = 0; c < I; ++c) { tab[pt.inst_values() + c] = inst_values + (size_t)c * n; tab[pt.inst_cosets() + c] = inst_cosets + (size_t)c * ext; }
        ZK_CUDA(ctx, cudaMemcpyAsync(pk->d_ptrs, tab.data(), tab.size() * sizeof(void*), cudaMemcpyHostToDevice, st));
        ZK_CUDA(ctx, cudaStreamSynchronize(st));
        return B200ZK_OK;
    }

    // step 0/1: vk.hash_into, instances
    int32_t instances(const void* const* instance_columns, const uint32_t* instance_lens, const HFr& transcript_repr) {
        tr.common_scalar(transcript_repr);
        ZK_CUDA(ctx, cudaMemsetAsync(inst_values, 0, I * n * sizeof(fe_t), st));
        for (uint32_t c = 0; c < I; ++c) {
            uint32_t len = instance_lens[c];
            if (len > usable) return fail(ctx, B200ZK_ESYNTH, "create_proof", "InstanceTooLarge");
            const uint64_t* v = (const uint64_t*)instance_columns[c];
            for (uint32_t i = 0; i < len; ++i) tr.common_scalar(HFr::from_limbs(v + 4 * i));
            if (len) ZK_CUDA(ctx, cudaMemcpyAsync(inst_values + (size_t)c * n, v, (size_t)len * sizeof(fe_t), cudaMemcpyHostToDevice, st));
        }
        ZK_CUDA(ctx, cudaMemcpyAsync(inst_polys, inst_values, I * n * sizeof(fe_t), cudaMemcpyDeviceToDevice, st));
        for (uint32_t c = 0; c < I; ++c) ZK_TRY(lagrange_to_coeff(pk, inst_polys + (size_t)c * n));
        return B200ZK_OK;
    }

    // randomness: Fr::random = from_u512 of the caller's 64-byte draws.  This rank converts the draws [d0, d1): all of
    // them, or with split_upload its 1/G of the stream, which the ranks then exchange.
    int32_t upload_rng(const void* rng_wide, bool rng_on_device) {
        const int parts = split_upload ? sh.G : 1, part = split_upload ? sh.R : 0;
        auto part_lo = [&](int r) { return dl.total * (size_t)r / parts; };
        const size_t d0 = part_lo(part), d1 = part_lo(part + 1);
        ZK_CUDA(ctx, cudaMemcpyAsync(wide + d0 * 16, (const char*)rng_wide + d0 * 64, (d1 - d0) * 64,
                                     rng_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        if (d1 > d0) { from_u512_kernel<<<nb(d1 - d0), PK_THREADS, 0, st>>>(wide + d0 * 16, rnd + d0, d1 - d0); ctx->launches++; }
        std::vector<CommPiece> pieces;
        if (split_upload) for (int r = 0; r < parts; ++r) pieces.push_back({rnd + part_lo(r), (part_lo(r + 1) - part_lo(r)) * sizeof(fe_t), r});
        return share(pieces);
    }

    // step 2: advice columns: blinding rows, blinds, commitments.
    // The columns arrive on the pk's copy stream one at a time (H2D from the caller's buffers, 32 MiB each at
    // k = 20, or D2D), each followed by its blinding rows; col_events[c] marks column c complete.  Everything that
    // does not need the transcript starts under that transfer: on the side stream the coefficient form and the
    // quotient cosets of column c as soon as it has landed (step 10, moved up), and — when the columns come from
    // the host — on the main stream the commitment to the vanishing argument's random polynomial (step 8), which
    // depends on the rng stream only.  The main stream then waits for the last column and commits all of them.
    int32_t advice(const fe_t* d_advice_in, const void* const* advice_host) {
        if (!pk->copy_stream) {
            ZK_CUDA(ctx, cudaStreamCreateWithFlags(&pk->copy_stream, cudaStreamNonBlocking));
            ZK_CUDA(ctx, cudaEventCreateWithFlags(&pk->ev_rnd, cudaEventDisableTiming));
        }
        while (pk->col_events.size() < A) {
            cudaEvent_t e;
            ZK_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            pk->col_events.push_back(e);
        }
        ZK_CUDA(ctx, cudaEventRecord(pk->ev_rnd, st));
        ZK_CUDA(ctx, cudaStreamWaitEvent(pk->copy_stream, pk->ev_rnd, 0));      // rnd (and the arena's previous users on st) first
        for (uint32_t c = 0; c < A; ++c) {
            fe_t* col = advice_values + (size_t)c * n;
            if (split_upload && !sh.mine(c)) continue;                // arrives from its owner below
            if (advice_on_device) ZK_CUDA(ctx, cudaMemcpyAsync(col, d_advice_in + (size_t)c * n, n * sizeof(fe_t), cudaMemcpyDeviceToDevice, pk->copy_stream));
            else ZK_CUDA(ctx, cudaMemcpyAsync(col, advice_host[c], n * sizeof(fe_t), cudaMemcpyHostToDevice, pk->copy_stream));
            ZK_CUDA(ctx, cudaMemcpyAsync(col + usable, rnd + dl.advice_rows(c), (bf + 1) * sizeof(fe_t), cudaMemcpyDeviceToDevice, pk->copy_stream));
            ZK_CUDA(ctx, cudaEventRecord(pk->col_events[c], pk->copy_stream));
        }
        if (split_upload) {                                           // random-polynomial commit under the upload, then the column exchange
            ZK_TRY(commit_random());
            std::vector<CommPiece> pieces;
            for (uint32_t c = 0; c < A; ++c) {
                if (sh.mine(c)) ZK_CUDA(ctx, cudaStreamWaitEvent(st, pk->col_events[c], 0));
                pieces.push_back({advice_values + (size_t)c * n, n * sizeof(fe_t), sh.owner(c)});
            }
            ZK_TRY(share(pieces));
        }
        {
            SideStream side(ctx);
            // columns that are already on the device arrive at once: all their inverse transforms as one batched launch per pass
            // (columns from the host keep the per-column pipeline under the upload)
            const bool batch_intt = advice_on_device && A > 1 && ((uint64_t)A << dom->k) <= 0xFFFFFFFFull;
            if (batch_intt) {
                ZK_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, pk->col_events[A - 1], 0));
                ZK_CUDA(ctx, cudaMemcpyAsync(advice_polys, advice_values, (size_t)A * n * sizeof(fe_t), cudaMemcpyDeviceToDevice, ctx->stream));
                ZK_TRY(lagrange_to_coeff(pk, advice_polys, A));
            }
            for (uint32_t c = 0; c < A; ++c) {
                if (!batch_intt) {
                    if (!split_upload) ZK_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, pk->col_events[c], 0));
                    ZK_CUDA(ctx, cudaMemcpyAsync(advice_polys + (size_t)c * n, advice_values + (size_t)c * n, n * sizeof(fe_t), cudaMemcpyDeviceToDevice, ctx->stream));
                    ZK_TRY(lagrange_to_coeff(pk, advice_polys + (size_t)c * n));
                }
                ZK_TRY(my_cosets(advice_polys + (size_t)c * n, advice_cosets + (size_t)c * ext, cj0, std::min(cj1, pk->plan.adv_need[c])));
            }
            // only the cosets a consumer reads (QuotPlan::adv_need / inst_need): the higher ones are never written
            for (uint32_t c = 0; c < I; ++c) ZK_TRY(my_cosets(inst_polys + (size_t)c * n, inst_cosets + (size_t)c * ext, cj0, std::min(cj1, pk->plan.inst_need[c])));
        }
        if (!advice_on_device && !split_upload) ZK_TRY(commit_random());
        if (A && !split_upload) ZK_CUDA(ctx, cudaStreamWaitEvent(st, pk->col_events[A - 1], 0));
        std::vector<const fe_t*> cols;
        std::vector<int> owners;
        for (uint32_t c = 0; c < A; ++c) { cols.push_back(advice_values + (size_t)c * n); owners.push_back(sh.owner(c)); }
        return commit_columns(cols, owners, "advice_commits");
    }

    // step 4: lookups, commit_permuted.  Lookup l lives on rank sh.lk_owner(l) from here to its grand product.
    int32_t lookup_permute() {
        for (uint32_t l = 0; l < L; ++l) {
            if (!sh.lk_mine(l)) continue;
            fe_t *cin = LK(l, 0), *ctab = LK(l, 1), *pin = LK(l, 2), *ptab = LK(l, 3), *pin_poly = LK(l, 4), *ptab_poly = LK(l, 5);
            {
                PhaseTimer t(pk, PH_LOOKUP);
                ExprArgs ea = expr_args(pk, pk->lookup_prog[l].first, pk->lookup_prog[l].second, false, EXM_ACC01, ch, cin, ctab);
                expr_kernel<<<nb(n), PK_THREADS, 0, st>>>(ea);
                ctx->launches++;
                ZK_TRY(lookup_permute_run(ctx, cin, ctab, (uint32_t)usable, pin, ptab, pk->d_err));
            }
            ZK_CUDA(ctx, copy_rows(pin + usable, rnd + dl.lookup_input_rows(l), bf + 1));
            ZK_CUDA(ctx, copy_rows(ptab + usable, rnd + dl.lookup_table_rows(l), bf + 1));
            ZK_CUDA(ctx, copy_rows(pin_poly, pin, n));
            ZK_TRY(lagrange_to_coeff(pk, pin_poly));
            ZK_CUDA(ctx, copy_rows(ptab_poly, ptab, n));
            ZK_TRY(lagrange_to_coeff(pk, ptab_poly));
        }
        ZK_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, pk->d_err, 4, cudaMemcpyDeviceToHost, st));
        ZK_CUDA(ctx, cudaStreamSynchronize(st));
        uint32_t err = *(const uint32_t*)ctx->pinned;
        if (L) {                                                      // permuted input / table commitments of all lookups, one batch
            std::vector<const fe_t*> cols;
            std::vector<int> owners;
            for (uint32_t l = 0; l < L; ++l) { cols.push_back(LK(l, 2)); cols.push_back(LK(l, 3)); owners.push_back(sh.lk_owner(l)); owners.push_back(sh.lk_owner(l)); }
            ZK_TRY(commit_columns(cols, owners, "lookup_permuted_commits", &err));
        }
        if (err) return fail(ctx, B200ZK_ESYNTH, "create_proof", "ConstraintSystemFailure: lookup input not in table");
        // the permuted polynomials in coefficient form: every rank opens them, the coset owners extend them
        std::vector<CommPiece> pieces;
        for (uint32_t l = 0; l < L; ++l) { pieces.push_back({LK(l, 4), n * sizeof(fe_t), sh.lk_owner(l)}); pieces.push_back({LK(l, 5), n * sizeof(fe_t), sh.lk_owner(l)}); }
        return share(pieces);
    }

    // side stream, once theta, beta and gamma are known: the a', s' cosets and the table values of every lookup
    int32_t lookup_cosets_early() {
        if (!pk->lk_early || !lk_rows) return B200ZK_OK;
        SideStream side(ctx);
        for (uint32_t l = 0; l < L; ++l) {
            ZK_TRY(my_cosets(LK(l, 4), LKC(l, 1), lj0, lj1));
            ZK_TRY(my_cosets(LK(l, 5), LKC(l, 2), lj0, lj1));
            lookup_table_value(l);
        }
        return B200ZK_OK;
    }

    // step 6: permutation argument.
    // Upstream chains the sets through z_s[0] = z_{s-1}[n - (bf + 1)].  Here set s runs on rank sh.set_owner(s) from
    // z[0] = 1, the S totals t_s = z'_s[n - (bf + 1)] are read back after one synchronisation (and gathered when
    // sharded), and set s is scaled by t_0 ... t_{s-1} — the same field elements, without a host round trip per set.
    int32_t permutation_products() {
        const HFr beta = ch[EXF_BETA], gamma = ch[EXF_GAMMA];
        HFr deltaomega = HFr::one();
        for (uint32_t s = 0; s < S; ++s) {
            fe_t* z = perm_polys + (size_t)s * n;
            uint32_t c0 = s * pk->chunk, c1 = std::min<uint32_t>(c0 + pk->chunk, pk->P);
            PermLagArgs pa{};
            pa.ncols = c1 - c0; pa.n = (uint32_t)n;
            for (uint32_t j = c0; j < c1; ++j) {
                pa.values[j - c0] = column_values(cs.perm[j].first, cs.perm[j].second);
                pa.sigma[j - c0] = pk->perm_values + (size_t)j * n;
                pa.coef[j - c0] = to_dev(deltaomega * beta);
                deltaomega = deltaomega * host::fr_delta();
            }
            if (!sh.set_mine(s)) continue;
            {
                PhaseTimer t(pk, PH_PERM);
                pa.beta = to_dev(beta); pa.gamma = to_dev(gamma); pa.omega_pows = pk->omega_pows; pa.out = tmp_n;
                perm_den_kernel<<<nb(n), PK_THREADS, 0, st>>>(pa);
                ctx->launches++;
                ZK_TRY(batch_invert_run(ctx, tmp_n, n, 0));
                perm_num_kernel<<<nb(n), PK_THREADS, 0, st>>>(pa);
                ctx->launches++;
                ZK_TRY(prefix_product_run(ctx, tmp_n, z, n, HFr::one()));
            }
            ZK_CUDA(ctx, cudaMemcpyAsync((fe_t*)ctx->pinned + s, z + (n - (bf + 1)), sizeof(fe_t), cudaMemcpyDeviceToHost, st));
        }
        if (S) {
            std::vector<HFr> totals(S, HFr::one());
            ZK_CUDA(ctx, cudaStreamSynchronize(st));
            for (uint32_t s = 0; s < S; ++s) if (sh.set_mine(s)) totals[s] = HFr::from_limbs((const fe_t*)ctx->pinned + s);
            ZK_TRY(sh.gather(pk, totals, [&](size_t s) { return sh.set_owner((uint32_t)s); }));
            HFr carry = HFr::one();
            for (uint32_t s = 0; s < S; ++s) {
                fe_t* z = perm_polys + (size_t)s * n;
                if (sh.set_mine(s)) {
                    if (s) { scale_kernel<<<nb(n - bf), PK_THREADS, 0, st>>>(z, to_dev(carry), n - bf); ctx->launches++; }
                    ZK_CUDA(ctx, copy_rows(z + (n - bf), rnd + dl.set_rows(s), bf));
                }
                carry = carry * totals[s];
            }
            mark("perm_products");
            // the S grand products: one batch of commitments, then coefficients and cosets
            std::vector<const fe_t*> cols;
            std::vector<int> owners;
            for (uint32_t s = 0; s < S; ++s) { cols.push_back(perm_polys + (size_t)s * n); owners.push_back(sh.set_owner(s)); }
            ZK_TRY(commit_columns(cols, owners, "permutation_commits"));
        }
        std::vector<CommPiece> pieces;
        const bool batch_intt = !sh.on() && S > 1 && ((uint64_t)S << dom->k) <= 0xFFFFFFFFull;      // one rank: all sets in one launch per pass
        if (batch_intt) ZK_TRY(lagrange_to_coeff(pk, perm_polys, S));
        for (uint32_t s = 0; s < S; ++s) {
            fe_t* z = perm_polys + (size_t)s * n;
            if (!batch_intt && sh.set_mine(s)) ZK_TRY(lagrange_to_coeff(pk, z));
            pieces.push_back({z, n * sizeof(fe_t), sh.set_owner(s)});
        }
        ZK_TRY(share(pieces));
        for (uint32_t s = 0; s < S; ++s) ZK_TRY(my_cosets(perm_polys + (size_t)s * n, perm_cosets + (size_t)s * ext, cj0, cj1));
        return B200ZK_OK;
    }

    // step 7: lookups, commit_product
    int32_t lookup_products() {
        for (uint32_t l = 0; l < L; ++l) {
            if (!sh.lk_mine(l)) continue;
            fe_t* z = LK(l, 6);
            {
                PhaseTimer t(pk, PH_LOOKUP);
                LookupProdArgs la{LK(l, 2), LK(l, 3), LK(l, 0), LK(l, 1), to_dev(ch[EXF_BETA]), to_dev(ch[EXF_GAMMA]), tmp_n, (uint32_t)n};
                lookup_den_kernel<<<nb(n), PK_THREADS, 0, st>>>(la);
                ctx->launches++;
                ZK_TRY(batch_invert_run(ctx, tmp_n, n, 0));
                lookup_num_kernel<<<nb(n), PK_THREADS, 0, st>>>(la);
                ctx->launches++;
                ZK_TRY(prefix_product_run(ctx, tmp_n, z, n, HFr::one()));
            }
            ZK_CUDA(ctx, copy_rows(z + (n - bf), rnd + dl.lookup_product_rows(l), bf));
        }
        if (!L) return B200ZK_OK;
        std::vector<const fe_t*> cols;
        std::vector<int> owners;
        std::vector<CommPiece> pieces;
        for (uint32_t l = 0; l < L; ++l) { cols.push_back(LK(l, 6)); owners.push_back(sh.lk_owner(l)); pieces.push_back({LK(l, 6), n * sizeof(fe_t), sh.lk_owner(l)}); }
        ZK_TRY(commit_columns(cols, owners, "lookup_product_commits"));
        for (uint32_t l = 0; l < L; ++l) if (sh.lk_mine(l)) ZK_TRY(lagrange_to_coeff(pk, LK(l, 6)));
        ZK_TRY(share(pieces));
        if (pk->lk_early && lk_rows) {                                // side stream: the product cosets
            SideStream side(ctx);
            for (uint32_t l = 0; l < L; ++l) ZK_TRY(my_cosets(LK(l, 6), LKC(l, 0), lj0, lj1));
        }
        return B200ZK_OK;
    }

    // step 8: vanishing argument, the random polynomial (committed under the advice upload when the columns come from the host)
    int32_t random_poly() {
        if (advice_on_device) ZK_TRY(commit_random());
        tr.write_point(random_pt);
        return B200ZK_OK;
    }

    // step 11: evaluate_h on this rank's rows of the quotient: its cosets [cj0, cj1) (all of them on a single GPU)
    int32_t evaluate_h() {
        if (!pk->gate_exp.empty()) {                                  // the gates' powers of y (ExprArgs::wts)
            std::vector<HFr> ypow(1, HFr::one());
            for (uint32_t i = 0; i < cs.gates.size(); ++i) {
                while (ypow.size() <= pk->gate_exp[i]) ypow.push_back(ypow.back() * ch[EXF_Y]);
                ((fe_t*)pk->h_wts)[i] = to_dev(ypow[pk->gate_exp[i]]);
            }
            ZK_CUDA(ctx, cudaMemcpyAsync(pk->d_wts, pk->h_wts, cs.gates.size() * sizeof(fe_t), cudaMemcpyHostToDevice, st));
        }
        // step 10: the advice / instance cosets were started on the side stream after the advice commitments
        ZK_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join, 0));
        const uint32_t rot_scale = 1u;                                // rotations stay inside a coset (prover_kernels.cuh)
        const HFr beta = ch[EXF_BETA], gamma = ch[EXF_GAMMA], y = ch[EXF_Y];
        const uint32_t my_row0 = cj0 * (uint32_t)n, my_rows = (cj1 - cj0) * (uint32_t)n;
        if (lin_mine()) ZK_TRY(gate_class(QC_LINEAR, h_lin, 0, (uint32_t)n));
        if (my_rows) {
            ZK_TRY(gate_class(QC_MAIN, h, my_row0, my_rows));
            PhaseTimer t(pk, PH_QUOT);
            if (S) {
                QuotPermAArgs qa{};
                qa.h = h; qa.y = to_dev(y); qa.l0 = pk->l0; qa.l_last = pk->l_last; qa.nsets = S;
                qa.rows = my_rows; qa.row0 = my_row0; qa.log_ext = dom->k; qa.rot_scale = rot_scale; qa.last_rot = -(int32_t)(bf + 1);
                for (uint32_t s = 0; s < S; ++s) qa.z[s] = perm_cosets + (size_t)s * ext;
                quot_perm_a_kernel<<<nb(my_rows), PK_THREADS, 0, st>>>(qa);
                ctx->launches++;
                HFr cd = beta * host::fr_zeta();                      // delta_start = beta * ZETA
                for (uint32_t s = 0; s < S; ++s) {
                    uint32_t c0 = s * pk->chunk, c1 = std::min<uint32_t>(c0 + pk->chunk, pk->P);
                    QuotPermBArgs qb{};
                    qb.h = h; qb.y = to_dev(y); qb.beta = to_dev(beta); qb.gamma = to_dev(gamma); qb.l_active = pk->l_active;
                    qb.z = perm_cosets + (size_t)s * ext; qb.ncols = c1 - c0; qb.rows = my_rows; qb.row0 = my_row0; qb.log_ext = dom->k; qb.rot_scale = rot_scale;
                    qb.omega_pows = pk->omega_pows; qb.coset_fac = pk->coset_fac;
                    for (uint32_t j = c0; j < c1; ++j) {
                        qb.values[j - c0] = column_cosets(cs.perm[j].first, cs.perm[j].second);
                        qb.sigma[j - c0] = pk->perm_cosets + (size_t)j * ext;
                        qb.cdelta[j - c0] = to_dev(cd);
                        cd = cd * host::fr_delta();
                    }
                    quot_perm_b_kernel<<<nb(my_rows), PK_THREADS, 0, st>>>(qb);
                    ctx->launches++;
                }
            }
        }
        // lookup terms: on all q cosets straight into h, or — when their degree allows — on the first CL cosets into
        // h_lk, extended to the other cosets after the per-coset iNTT (lookup_extrapolate_row)
        if (lk_split) ZK_TRY(gate_class(QC_LOW, h_lk, lk_row0, lk_rows));
        for (uint32_t l = 0; l < L && lk_rows; ++l) {
            fe_t *zc = LKC(l, 0), *ac = LKC(l, 1), *sc = LKC(l, 2), *tv = LKC(l, 3);
            if (!pk->lk_early) {
                ZK_TRY(my_cosets(LK(l, 6), zc, lj0, lj1));
                ZK_TRY(my_cosets(LK(l, 4), ac, lj0, lj1));
                ZK_TRY(my_cosets(LK(l, 5), sc, lj0, lj1));
                lookup_table_value(l);
            }
            PhaseTimer t(pk, PH_QUOT);
            QuotLookupArgs ql{};
            ql.h = lk_split ? h_lk : h; ql.y = to_dev(y); ql.beta = to_dev(beta); ql.gamma = to_dev(gamma);
            ql.l0 = pk->l0; ql.l_last = pk->l_last; ql.l_active = pk->l_active; ql.z = zc; ql.a = ac; ql.s = sc; ql.table_value = tv;
            ql.log_ext = dom->k; ql.rot_scale = rot_scale; ql.rows = lk_rows; ql.row0 = lk_row0;
            { HFr yp = y * y; for (int i = 0; i < 4; ++i) { ql.ypow[i] = to_dev(yp); yp = yp * y; } }
            quot_lookup_kernel<<<nb(lk_rows), PK_THREADS, 0, st>>>(ql);
            ctx->launches++;
        }
        ZK_CUDA(ctx, cudaGetLastError());
        return B200ZK_OK;
    }

    // step 12: vanishing construct, then the commitments to the q pieces of h
    int32_t vanishing_construct() {
        {
            // divide by the vanishing polynomial (constant c_j^n - 1 on coset j), per-coset iNTT, then
            // the q x q interpolation across cosets gives the coefficients of h piece by piece
            PhaseTimer t(pk, PH_NTT);
            HFr y_lk = HFr::one();                                    // h = h_gates_perm * y^(5 L) + h_lk
            if (lk_split) {
                for (uint32_t i = 0; i < 5 * L; ++i) y_lk = y_lk * ch[EXF_Y];  // (the low gates' weights leave this factor to the lookup kernels)
                for (uint32_t j = lj0; j < lj1; ++j)                           // divided by the vanishing polynomial before the extrapolation
                    ZK_TRY(intt_scaled(pk, h_lk + j * n, 1, dom->ifft_divisor * pk->coset_t[j]));
            }
            for (uint32_t j = cj0; j < cj1; ++j) ZK_TRY(intt_scaled(pk, h + j * n, 1, dom->ifft_divisor * pk->coset_t[j] * y_lk));
            // the linear gates' part of h, degree < n: coefficients in X / c_0
            if (lin_mine()) ZK_TRY(intt_scaled(pk, h_lin, 1, dom->ifft_divisor * pk->coset_t[0]));
        }
        std::vector<CommPiece> pieces;                                // every coset's coefficients to every rank: q (+ CL) x n elements
        for (uint32_t j = 0; j < pk->q; ++j) pieces.push_back({h + (size_t)j * n, n * sizeof(fe_t), sh.coset_owner(j)});
        if (lk_split) for (uint32_t j = 0; j < CL; ++j) pieces.push_back({h_lk + (size_t)j * n, n * sizeof(fe_t), sh.coset_owner(j)});
        if (pk->gate_prog[QC_LINEAR].second) pieces.push_back({h_lin, n * sizeof(fe_t), sh.coset_owner(0)});
        ZK_TRY(share(pieces));
        {
            PhaseTimer t(pk, PH_NTT);
            if (lk_split) {
                lookup_extrapolate_kernel<<<nb(n), PK_THREADS, 0, st>>>(h_lk, pk->coset_pow_inv, pk->lk_lambda, nullptr, CL, pk->q, n);
                ctx->launches++;
            }
            coset_interpolate_kernel<<<nb(n), PK_THREADS, 0, st>>>(h, pk->coset_pow_inv, pk->vinv, pk->q, n, lk_cosets, lk_split ? h_lk : nullptr,
                                                                     pk->gate_prog[QC_LINEAR].second ? h_lin : nullptr);
            ctx->launches++;
            ZK_CUDA(ctx, cudaGetLastError());
        }
        std::vector<const fe_t*> cols;
        std::vector<HAffine> pts;
        for (uint32_t i = 0; i < pk->q; ++i) cols.push_back(lk_cosets + (size_t)i * n);
        ZK_TRY(commit_multi_range(pk, sh, cols, n, false, pts));
        for (auto& pt : pts) tr.write_point(pt);
        mark("quotient_and_h_commits");
        return B200ZK_OK;
    }

    // step 14: evaluations
    int32_t evaluations() {
        const HFr x_next = rotate_omega(dom, x, 1), x_prev = rotate_omega(dom, x, -1), x_last = rotate_omega(dom, x, -(int)(bf + 1));
        const fe_t* random = rnd + dl.random;
        // multiopen queries in upstream order (step 15); every evaluation the transcript gets is one of them, so their
        // distinct pairs are evaluated here in ONE batched launch pair
        for (size_t i = 0; i < cs.adv_q.size(); i += 2) queries.push_back({advice_polys + (size_t)cs.adv_q[i] * n, rotate_omega(dom, x, cs.adv_q[i + 1])});
        for (uint32_t s = 0; s < S; ++s) { queries.push_back({perm_polys + (size_t)s * n, x}); queries.push_back({perm_polys + (size_t)s * n, x_next}); }
        for (uint32_t s = S; s-- > 0;) if (s + 1 < S) queries.push_back({perm_polys + (size_t)s * n, x_last});
        for (uint32_t l = 0; l < L; ++l) {
            queries.push_back({LK(l, 6), x}); queries.push_back({LK(l, 4), x}); queries.push_back({LK(l, 5), x});
            queries.push_back({LK(l, 4), x_prev}); queries.push_back({LK(l, 6), x_next});
        }
        for (size_t i = 0; i < cs.fix_q.size(); i += 2) queries.push_back({pk->fixed_polys + (size_t)cs.fix_q[i] * n, rotate_omega(dom, x, cs.fix_q[i + 1])});
        for (uint32_t j = 0; j < pk->P; ++j) queries.push_back({pk->perm_polys + (size_t)j * n, x});
        queries.push_back({h_poly, x});
        queries.push_back({random, x});
        for (auto& qy : queries)
            if (std::none_of(pairs.begin(), pairs.end(), [&](const Query& p) { return p.poly == qy.poly && p.point == qy.point; })) pairs.push_back(qy);
        std::vector<const fe_t*> bp; std::vector<HFr> bx;             // pair i on rank i mod G, 32 bytes each back to everybody
        for (size_t i = 0; i < pairs.size(); ++i) if (sh.mine((uint32_t)i)) { bp.push_back(pairs[i].poly); bx.push_back(pairs[i].point); }
        std::vector<HFr> mv(bp.size());
        {
            PhaseTimer t(pk, PH_OPEN);
            // vanishing::evaluate: h_poly = sum_i (x^n)^i h_piece_i
            fold_pieces_kernel<<<nb(n), PK_THREADS, 0, st>>>(lk_cosets, pk->q, n, to_dev(x.pow_u64(n)), h_poly);
            ctx->launches++;
            ZK_TRY(eval_batch_run(ctx, bp.data(), bx.data(), bp.size(), n, mv.data()));
        }
        values.assign(pairs.size(), HFr::zero());
        for (size_t i = 0, j = 0; i < pairs.size(); ++i) if (sh.mine((uint32_t)i)) values[i] = mv[j++];
        ZK_TRY(sh.gather(pk, values, [&](size_t i) { return sh.owner((uint32_t)i); }));
        mark("evaluations");
        // the transcript's order: advice, fixed, random, sigma, permutation sets, lookups
        for (size_t i = 0; i < cs.adv_q.size(); i += 2) ZK_TRY(write_eval(advice_polys + (size_t)cs.adv_q[i] * n, rotate_omega(dom, x, cs.adv_q[i + 1])));
        for (size_t i = 0; i < cs.fix_q.size(); i += 2) ZK_TRY(write_eval(pk->fixed_polys + (size_t)cs.fix_q[i] * n, rotate_omega(dom, x, cs.fix_q[i + 1])));
        ZK_TRY(write_eval(random, x));
        for (uint32_t j = 0; j < pk->P; ++j) ZK_TRY(write_eval(pk->perm_polys + (size_t)j * n, x));
        for (uint32_t s = 0; s < S; ++s) {
            const fe_t* zp = perm_polys + (size_t)s * n;
            ZK_TRY(write_eval(zp, x)); ZK_TRY(write_eval(zp, x_next));
            if (s + 1 < S) ZK_TRY(write_eval(zp, x_last));
        }
        for (uint32_t l = 0; l < L; ++l) {                           // product z, permuted input a', permuted table s'
            ZK_TRY(write_eval(LK(l, 6), x)); ZK_TRY(write_eval(LK(l, 6), x_next));
            ZK_TRY(write_eval(LK(l, 4), x)); ZK_TRY(write_eval(LK(l, 4), x_prev)); ZK_TRY(write_eval(LK(l, 5), x));
        }
        return B200ZK_OK;
    }

    // step 15: ProverSHPLONK::create_proof over `queries`
    int32_t shplonk() {
        HFr sy, sv, su;
        {
            PhaseTimer t(pk, PH_OPEN);
            sy = tr.squeeze_challenge();
            ZK_TRY(shplonk_sets());
            sv = tr.squeeze_challenge();
            // h1 = sum_i v^i Q_i into hx.  Rotation set i (its linear combination A_i and the Kate divisions that give Q_i, of
            // n - |points| coefficients) lives on rank i mod G; both polynomials are then broadcast — every rank needs A_i again
            // for the linearisation polynomial — and h1 is formed everywhere.
            ZK_CUDA(ctx, cudaMemsetAsync(hx, 0, n * sizeof(fe_t), st));
            std::vector<CommPiece> pieces;
            for (size_t i = 0; i < rot_sets.size(); ++i) {
                fe_t *sum = set_sums + i * n, *quot = set_quot + i * n;     // A_i = sum_j y^j P_ij, Q_i
                const std::vector<HFr>& pts = rot_sets[i].pts;
                pieces.push_back({sum, n * sizeof(fe_t), sh.owner((uint32_t)i)});
                pieces.push_back({quot, (n - pts.size()) * sizeof(fe_t), sh.owner((uint32_t)i)});
                if (!sh.mine((uint32_t)i)) continue;
                HFr y_pow = HFr::one();
                std::vector<HFr> rlow(rot_sets[i].pts.size(), HFr::zero());   // R_i = sum_j y^j r_ij
                for (size_t j0 = 0; j0 < rot_sets[i].polys.size(); j0 += 16) {
                    LinCombArgs la{};
                    la.m = (uint32_t)std::min<size_t>(16, rot_sets[i].polys.size() - j0);
                    for (uint32_t j = 0; j < la.m; ++j) {
                        la.p[j] = rot_sets[i].polys[j0 + j];
                        la.s[j] = to_dev(y_pow);
                        for (size_t c = 0; c < low[i][j0 + j].size(); ++c) rlow[c] = rlow[c] + low[i][j0 + j][c] * y_pow;
                        y_pow = y_pow * sy;
                    }
                    lincomb_kernel<<<nb(n), PK_THREADS, 0, st>>>(sum, la, n, j0 == 0 ? 1 : 0);
                    ctx->launches++;
                }
                // N_i = A_i - R_i ; Q_i = N_i / prod (X - p)
                ZK_CUDA(ctx, copy_rows(t0, sum, n));
                LowCoeffs lc{}; lc.m = (uint32_t)rlow.size();
                for (size_t c = 0; c < rlow.size(); ++c) lc.c[c] = to_dev(rlow[c]);
                sub_low_kernel<<<1, 8, 0, st>>>(t0, lc);
                ctx->launches++;
                fe_t* src = t0;                                           // kate_division by each point, the last one into Q_i
                for (size_t k = 0; k < pts.size(); ++k) {
                    fe_t* dst = k + 1 == pts.size() ? quot : src == t0 ? t1 : t0;
                    ZK_TRY(recurrence_run(ctx, src + 1, dst, n - k - 1, pts[k], nullptr));
                    src = dst;
                }
            }
            ZK_TRY(share(pieces));
            HFr v_pow = HFr::one();
            for (size_t i = 0; i < rot_sets.size(); ++i) {
                const size_t len = n - rot_sets[i].pts.size();
                axpy_kernel<<<nb(len), PK_THREADS, 0, st>>>(hx, set_quot + i * n, to_dev(v_pow), len, 0);
                ctx->launches++;
                v_pow = v_pow * sv;
            }
        }
        std::vector<HAffine> pt;
        ZK_TRY(commit_multi_range(pk, sh, {hx}, n, false, pt));
        tr.write_point(pt[0]);
        mark("shplonk_h1_commit");
        {
            // the linearisation polynomial L(X) at u, divided by (X - u) into t0
            PhaseTimer t(pk, PH_OPEN);
            su = tr.squeeze_challenge();
            auto vanish = [&](const std::vector<HFr>& roots) { HFr acc = HFr::one(); for (auto& r : roots) acc = acc * (su - r); return acc; };
            HFr v_pow = HFr::one(), const_term = HFr::zero(), z0_diff = HFr::zero();
            for (size_t i = 0; i < rot_sets.size(); ++i) {
                std::vector<HFr> diffs;
                for (auto& p : super_points)
                    if (std::find_if(rot_sets[i].pts.begin(), rot_sets[i].pts.end(), [&](const HFr& o) { return o == p; }) == rot_sets[i].pts.end()) diffs.push_back(p);
                HFr z_i = vanish(diffs);
                if (i == 0) z0_diff = z_i;
                HFr y_pow = HFr::one(), c_i = HFr::zero();
                for (size_t j = 0; j < rot_sets[i].polys.size(); ++j) { c_i = c_i + eval_small(low[i][j], su) * y_pow; y_pow = y_pow * sy; }
                HFr coef = z_i * v_pow;
                axpy_kernel<<<nb(n), PK_THREADS, 0, st>>>(lx, set_sums + i * n, to_dev(coef), n, i == 0 ? 1 : 0);
                ctx->launches++;
                const_term = const_term + coef * c_i;
                v_pow = v_pow * sv;
            }
            std::vector<HFr> sp(super_points.begin(), super_points.end());
            HFr zt = vanish(sp);
            axpy_kernel<<<nb(n), PK_THREADS, 0, st>>>(lx, hx, to_dev(zt.neg()), n, 0);
            LowCoeffs lc{}; lc.m = 1; lc.c[0] = to_dev(const_term);
            sub_low_kernel<<<1, 8, 0, st>>>(lx, lc);
            ctx->launches += 2;
            ZK_TRY(recurrence_run(ctx, lx + 1, t0, n - 1, su, nullptr));              // (L(X)) / (X - u)
            scale_kernel<<<nb(n - 1), PK_THREADS, 0, st>>>(t0, to_dev(z0_diff.inv()), n - 1);
            ctx->launches++;
            ZK_CUDA(ctx, cudaGetLastError());
        }
        ZK_TRY(commit_multi_range(pk, sh, {t0}, n - 1, false, pt));
        tr.write_point(pt[0]);
        return B200ZK_OK;
    }

    // construct_intermediate_sets, and the low-degree equivalents of the polynomials of each rotation set
    int32_t shplonk_sets() {
        struct CommSet { const fe_t* poly; std::set<HFr, FrLess> pts; };
        std::vector<CommSet> comm_sets;
        for (auto& qy : queries) {
            super_points.insert(qy.point);
            auto it = std::find_if(comm_sets.begin(), comm_sets.end(), [&](const CommSet& c) { return c.poly == qy.poly; });
            if (it == comm_sets.end()) { comm_sets.push_back({qy.poly, {}}); it = comm_sets.end() - 1; }
            it->pts.insert(qy.point);
        }
        for (auto& c : comm_sets) {
            std::vector<HFr> pts(c.pts.begin(), c.pts.end());
            auto it = std::find_if(rot_sets.begin(), rot_sets.end(), [&](const RotSet& r) {
                return r.pts.size() == pts.size() && std::equal(pts.begin(), pts.end(), r.pts.begin());
            });
            if (it == rot_sets.end()) { rot_sets.push_back({pts, {}}); it = rot_sets.end() - 1; }
            if (std::find(it->polys.begin(), it->polys.end(), c.poly) == it->polys.end()) it->polys.push_back(c.poly);
        }
        if (rot_sets.size() > 8) return fail(ctx, B200ZK_EINVAL, "create_proof", "more than 8 rotation sets");
        low.resize(rot_sets.size());
        for (size_t i = 0; i < rot_sets.size(); ++i) {
            const size_t m = rot_sets[i].pts.size();
            if (m > 8) return fail(ctx, B200ZK_EINVAL, "create_proof", "rotation set with more than 8 points");
            // the Lagrange basis of the set's points once (m field inversions), then every polynomial of the set is a
            // combination of it: the same interpolant as arithmetic::lagrange_interpolate per polynomial, without an
            // inversion per polynomial and point (they were ~2 ms of host time per proof at every size)
            std::vector<std::vector<HFr>> basis(m);
            for (size_t j = 0; j < m; ++j) { std::vector<HFr> unit(m, HFr::zero()); unit[j] = HFr::one(); basis[j] = lagrange_interpolate(rot_sets[i].pts, unit); }
            for (const fe_t* poly : rot_sets[i].polys) {
                std::vector<HFr> lowp(m, HFr::zero());
                for (size_t j = 0; j < m; ++j) {
                    HFr e = HFr::zero();
                    ZK_TRY(opened(poly, rot_sets[i].pts[j], &e));
                    for (size_t c = 0; c < m; ++c) lowp[c] = lowp[c] + basis[j][c] * e;
                }
                low[i].push_back(lowp);
            }
        }
        return B200ZK_OK;
    }
};

static int32_t prove(b200zk_pk* pk, const fe_t* d_advice_in, bool advice_on_device, const void* const* advice_host,
                     const void* const* instance_columns, const uint32_t* instance_lens, const void* rng_wide, bool rng_on_device,
                     const HFr& transcript_repr, std::vector<uint8_t>& proof_out) {
    b200zk_ctx* ctx = pk->ctx;
    for (uint32_t c = 0; c < pk->cs.I; ++c) if (instance_lens[c] && !instance_columns[c]) return fail(ctx, B200ZK_EINVAL, "create_proof", "null instance column");
    if (!advice_on_device) for (uint32_t c = 0; c < pk->cs.A; ++c) if (!advice_host[c]) return fail(ctx, B200ZK_EINVAL, "create_proof", "null advice column");
    cudaStreamSynchronize(ctx->stream2);                          // nothing of an earlier (failed) proof may still be writing the arena
    if (pk->copy_stream) cudaStreamSynchronize(pk->copy_stream);
    for (float& f : pk->phase_ms) f = 0;
    pk->timer_used = 0;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    pk->trace.clear();
    Prover p(pk, advice_on_device, rng_on_device);
    ZK_CUDA(ctx, cudaMemsetAsync(pk->d_err, 0, 4, ctx->stream));
    ZK_TRY(p.carve());
    ZK_TRY(p.instances(instance_columns, instance_lens, transcript_repr));
    ZK_TRY(p.upload_rng(rng_wide, rng_on_device));
    ZK_TRY(p.advice(d_advice_in, advice_host));
    p.ch[EXF_THETA] = p.tr.squeeze_challenge();
    ZK_TRY(p.lookup_permute());
    p.ch[EXF_BETA] = p.tr.squeeze_challenge();
    p.ch[EXF_GAMMA] = p.tr.squeeze_challenge();
    ZK_TRY(p.lookup_cosets_early());
    ZK_TRY(p.permutation_products());
    ZK_TRY(p.lookup_products());
    ZK_TRY(p.random_poly());
    p.ch[EXF_Y] = p.tr.squeeze_challenge();
    ZK_TRY(p.evaluate_h());
    ZK_TRY(p.vanishing_construct());
    p.x = p.tr.squeeze_challenge();
    ZK_TRY(p.evaluations());
    ZK_TRY(p.shplonk());
    phase_timers_collect(pk);
    p.mark("end");
    proof_out = p.tr.proof();
    return B200ZK_OK;
}

}  // namespace b200zk

// ------------------------------------------------------------------ C ABI
extern "C" {

size_t b200zk_pk_rng_draws(const b200zk_pk* pk) { return pk ? DrawLayout(pk).total : 0; }

size_t b200zk_pk_proof_size(const b200zk_pk* pk) {
    if (!pk) return 0;
    const CsDesc& cs = pk->cs;
    size_t S = pk->S, L = pk->L;
    size_t points = cs.A + 2 * L + S + L + 1 + pk->q + 2;
    size_t evals = cs.adv_q.size() / 2 + cs.fix_q.size() / 2 + 1 + pk->P + (S ? 3 * S - 1 : 0) + 5 * L;
    return 32 * (points + evals);
}

uint32_t b200zk_pk_blinding_factors(const b200zk_pk* pk) { return pk ? pk->cs.bf : 0; }
uint32_t b200zk_pk_degree(const b200zk_pk* pk) { return pk ? pk->cs.degree : 0; }

// debugging aid: copy a named device buffer of the last proof to the host (elements of 32 bytes)
int32_t b200zk_pk_debug_buffer(b200zk_pk* pk, const char* name, void* host_out, size_t max_elems, size_t* count) {
    if (!pk || !name || !host_out) return B200ZK_EINVAL;
    auto it = pk->dbg.find(name);
    if (it == pk->dbg.end()) return fail(pk->ctx, B200ZK_EINVAL, "debug_buffer", "unknown buffer");
    size_t c = std::min(max_elems, it->second.second);
    if (count) *count = it->second.second;
    ZK_CUDA(pk->ctx, cudaMemcpyAsync(host_out, it->second.first, c * sizeof(fe_t), cudaMemcpyDeviceToHost, pk->ctx->stream));
    ZK_CUDA(pk->ctx, cudaStreamSynchronize(pk->ctx->stream));
    return B200ZK_OK;
}

// Field multiplications evaluate_h executes per row, as launched: out[0] custom gates, out[1] permutation terms (one row of
// every quotient coset), out[2] all lookups together (rows of the lk_cosets_n cosets the lookup terms run on), out[3] = q,
// out[4] = lk_cosets_n.  bench.py's roofline_quotient: work = n * (q * (gates + perm) + CL * lookups).  The gates run as
// three programs on q, lk_cosets_n and 1 cosets (quot_plan.hpp), so out[0] is their coset-weighted total divided by q,
// rounded: q * out[0] is the gate work launched per row of one coset.
int32_t b200zk_pk_quotient_muls(const b200zk_pk* pk, uint32_t out5[5]) {
    if (!pk || !out5) return B200ZK_EINVAL;
    // the programs live on the device; count from a host copy
    uint32_t total = 0;
    for (auto& gp : pk->gate_prog) total = std::max(total, gp.first + gp.second);
    for (auto& lp : pk->lookup_prog) total = std::max(total, lp.first + lp.second);
    std::vector<uint32_t> prog(total);
    if (total && cudaMemcpy(prog.data(), pk->d_prog, total * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return B200ZK_ECUDA;
    uint64_t gate_work = 0;
    for (uint32_t c = 0; c < 3; ++c) gate_work += (uint64_t)pk->plan.cosets(c) * ex_program_muls(prog.data() + pk->gate_prog[c].first, pk->gate_prog[c].second);
    out5[0] = (uint32_t)((gate_work + pk->q / 2) / pk->q);
    uint32_t perm = 0;
    if (pk->S) {
        perm = 5 + 2 * (pk->S - 1);
        for (uint32_t s = 0; s < pk->S; ++s) { uint32_t c0 = s * pk->chunk, c1 = std::min<uint32_t>(c0 + pk->chunk, pk->P); perm += 3 + 4 * (c1 - c0); }
    }
    out5[1] = perm;
    uint32_t lk = 0;
    for (auto& lp : pk->lookup_prog) lk += ex_program_muls(prog.data() + lp.first, lp.second) + 1 + 13;       // table value product + quot_lookup_row
    out5[2] = lk; out5[3] = pk->q; out5[4] = pk->lk_cosets_n;
    return B200ZK_OK;
}

// host wall clock of the last create_proof at its synchronisation points: "label:ms;label:ms;..." (ms since the call)
int32_t b200zk_pk_last_trace(const b200zk_pk* pk, char* out, size_t cap) {
    if (!pk || !out || cap == 0) return B200ZK_EINVAL;
    std::string t;
    for (auto& kv : pk->trace) { char buf[96]; snprintf(buf, sizeof buf, "%s:%.3f;", kv.first, kv.second); t += buf; }
    if (t.size() + 1 > cap) return B200ZK_EINVAL;
    memcpy(out, t.c_str(), t.size() + 1);
    return B200ZK_OK;
}

int32_t b200zk_pk_last_phase_ms(const b200zk_pk* pk, float* out7) {
    if (!pk || !out7) return B200ZK_EINVAL;
    memcpy(out7, pk->phase_ms, sizeof(pk->phase_ms));
    return B200ZK_OK;
}

// keygen_vk's O(n) part (src/plonk/keygen.rs): the commitments to the fixed and the permutation
// polynomials a VerifyingKey holds, computed on the device from the pk's coefficient forms.
int32_t b200zk_pk_vk_commitments(b200zk_pk* pk, void* fixed_out, void* sigma_out) {
    if (!pk || (pk->cs.F && !fixed_out) || (pk->P && !sigma_out)) return B200ZK_EINVAL;
    cudaSetDevice(pk->ctx->device);
    size_t n = pk->n;
    auto run = [&](const fe_t* base, uint32_t count, void* out) -> int32_t {
        if (!count) return B200ZK_OK;
        std::vector<const fe_t*> cols;
        std::vector<HAffine> pts;
        for (uint32_t c = 0; c < count; ++c) cols.push_back(base + (size_t)c * n);
        ZK_TRY(commit_multi_dev(pk, cols, n, false, pts));
        for (uint32_t c = 0; c < count; ++c) { pts[c].x.store((uint8_t*)out + 64 * (size_t)c); pts[c].y.store((uint8_t*)out + 64 * (size_t)c + 32); }
        return B200ZK_OK;
    };
    ZK_TRY(run(pk->fixed_polys, pk->cs.F, fixed_out));
    ZK_TRY(run(pk->perm_polys, pk->P, sigma_out));
    pk->timer_used = 0;
    return B200ZK_OK;
}

void b200zk_pk_destroy(b200zk_pk* pk) {
    if (!pk) return;
    cudaSetDevice(pk->ctx->device);
    if (pk->copy_stream) { cudaStreamSynchronize(pk->copy_stream); cudaStreamDestroy(pk->copy_stream); }
    if (pk->ev_rnd) cudaEventDestroy(pk->ev_rnd);
    if (pk->h_wts) cudaFreeHost(pk->h_wts);
    for (cudaEvent_t e : pk->col_events) cudaEventDestroy(e);
    cudaStreamSynchronize(pk->ctx->stream);
    for (void* p : pk->owned) cudaFree(p);
    for (auto& t : pk->timer_events) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
    if (pk->dom) b200zk_domain_destroy(pk->dom);
    delete pk;
}

int32_t b200zk_pk_create(b200zk_params* params, const uint32_t* cs_blob, size_t blob_words, const void* const* fixed_columns,
                         const uint32_t* map_col, const uint32_t* map_row, b200zk_pk** out) {
    if (!params || !cs_blob || !out) return B200ZK_EINVAL;
    b200zk_ctx* ctx = params->ctx;
    ZK_CUDA(ctx, cudaSetDevice(ctx->device));
    b200zk_pk* pk = new (std::nothrow) b200zk_pk();
    if (!pk) return B200ZK_ENOMEM;
    pk->ctx = ctx; pk->params = params;
    auto bail = [&](int32_t rc) { b200zk_pk_destroy(pk); return rc; };
    if (!parse_cs(cs_blob, blob_words, pk->cs)) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "malformed constraint-system blob"));
    CsDesc& cs = pk->cs;
    if (cs.k != params->k || !params->d_g_lagrange) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "params do not match k / lagrange basis missing"));
    if (cs.F && !fixed_columns) return bail(B200ZK_EINVAL);
    int32_t rc = b200zk_domain_create(ctx, cs.degree, cs.k, &pk->dom);
    if (rc != B200ZK_OK) return bail(rc);
    const b200zk_domain* dom = pk->dom;
    pk->n = 1u << cs.k;
    pk->P = (uint32_t)cs.perm.size(); pk->L = (uint32_t)cs.lookups.size();
    pk->chunk = cs.degree - 2;
    pk->S = (pk->P + pk->chunk - 1) / pk->chunk;
    pk->q = dom->quotient_poly_degree;
    pk->ext_n = pk->q * pk->n;                                    // q cosets of size n (prover_kernels.cuh)
    if (pk->chunk > ZK_MAXC || pk->S > ZK_MAXC || pk->q > (uint32_t)ZK_MAXCOSETS || pk->q > (1u << (dom->extended_k - dom->k)) ||
        (uint64_t)pk->q * pk->n > 0xFFFFFFFFull)
        return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "permutation too wide for this build"));
    if (pk->P && (!map_col || !map_row)) return bail(B200ZK_EINVAL);
    const size_t n = pk->n, ext = pk->ext_n;
    const uint32_t F = cs.F, P = pk->P;
    cudaStream_t st = ctx->stream;
#define PK_TRY(expr) do { int32_t _r = (expr); if (_r != B200ZK_OK) return bail(_r); } while (0)
#define PK_CUDA(expr) do { cudaError_t _e = (expr); if (_e != cudaSuccess) return bail(fail(ctx, B200ZK_ECUDA, #expr, cudaGetErrorString(_e))); } while (0)
    PK_TRY(dev_alloc(pk, &pk->fixed_values, F * n)); PK_TRY(dev_alloc(pk, &pk->fixed_polys, F * n)); PK_TRY(dev_alloc(pk, &pk->fixed_cosets, F * ext));
    PK_TRY(dev_alloc(pk, &pk->perm_values, P * n)); PK_TRY(dev_alloc(pk, &pk->perm_polys, P * n)); PK_TRY(dev_alloc(pk, &pk->perm_cosets, P * ext));
    PK_TRY(dev_alloc(pk, &pk->l0, ext)); PK_TRY(dev_alloc(pk, &pk->l_last, ext)); PK_TRY(dev_alloc(pk, &pk->l_active, ext));
    PK_TRY(dev_alloc(pk, &pk->omega_pows, n));
    PK_TRY(dev_alloc(pk, &pk->d_err, 1));
    // quotient cosets: powers of c_j and 1/c_j, extended_omega^j, 1/(c_j^n - 1), inverse Vandermonde of c_j^n
    {
        const uint32_t C = pk->q;
        PK_TRY(dev_alloc(pk, &pk->coset_pow, (size_t)C * n)); PK_TRY(dev_alloc(pk, &pk->coset_pow_inv, (size_t)C * n));
        PK_TRY(dev_alloc(pk, &pk->coset_fac, C)); PK_TRY(dev_alloc(pk, &pk->vinv, (size_t)C * C));
        std::vector<HFr> y(C);
        std::vector<fe_t> fac(C);
        HFr w = HFr::one();
        for (uint32_t j = 0; j < C; ++j) {
            HFr cj = dom->g_coset * w;
            PK_TRY(powers_run(ctx, cj, n, pk->coset_pow + (size_t)j * n));
            PK_TRY(powers_run(ctx, cj.inv(), n, pk->coset_pow_inv + (size_t)j * n));
            y[j] = cj.pow_u64(n);
            pk->coset_t.push_back((y[j] - HFr::one()).inv());
            fac[j] = to_dev(w);
            w = w * dom->extended_omega;
        }
        // V[j][t] = y_j^t; vinv = V^-1 by Gauss-Jordan (C <= 32; the y_j are distinct, so V is regular)
        std::vector<std::vector<HFr>> m(C, std::vector<HFr>(2 * C, HFr::zero()));
        for (uint32_t j = 0; j < C; ++j) { HFr p = HFr::one(); for (uint32_t t = 0; t < C; ++t) { m[j][t] = p; p = p * y[j]; } m[j][C + j] = HFr::one(); }
        for (uint32_t c = 0; c < C; ++c) {
            uint32_t piv = c;
            while (piv < C && m[piv][c] == HFr::zero()) ++piv;
            if (piv == C) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "internal: singular coset Vandermonde"));
            std::swap(m[c], m[piv]);
            HFr inv = m[c][c].inv();
            for (auto& v : m[c]) v = v * inv;
            for (uint32_t r = 0; r < C; ++r) {
                if (r == c || m[r][c] == HFr::zero()) continue;
                HFr f = m[r][c];
                for (uint32_t k2 = 0; k2 < 2 * C; ++k2) m[r][k2] = m[r][k2] - f * m[c][k2];
            }
        }
        std::vector<fe_t> vin((size_t)C * C);
        for (uint32_t t = 0; t < C; ++t) for (uint32_t j = 0; j < C; ++j) vin[(size_t)t * C + j] = to_dev(m[t][C + j]);
        PK_CUDA(cudaMemcpyAsync(pk->coset_fac, fac.data(), C * sizeof(fe_t), cudaMemcpyHostToDevice, st));
        PK_CUDA(cudaMemcpyAsync(pk->vinv, vin.data(), vin.size() * sizeof(fe_t), cudaMemcpyHostToDevice, st));
        pk->plan = quot_plan(cs, C, lookup_cosets(cs, C));
        const uint32_t CL = pk->plan.low;
        pk->lk_cosets_n = CL;
        std::vector<fe_t> lam((size_t)std::max<uint32_t>(C - CL, 1) * CL);
        for (uint32_t jp = CL; jp < C; ++jp)
            for (uint32_t j = 0; j < CL; ++j) {
                HFr num = HFr::one(), den = HFr::one();
                for (uint32_t m2 = 0; m2 < CL; ++m2) { if (m2 == j) continue; num = num * (y[jp] - y[m2]); den = den * (y[j] - y[m2]); }
                lam[(size_t)(jp - CL) * CL + j] = to_dev(num * den.inv());
            }
        PK_TRY(dev_alloc(pk, &pk->lk_lambda, lam.size()));
        PK_CUDA(cudaMemcpyAsync(pk->lk_lambda, lam.data(), lam.size() * sizeof(fe_t), cudaMemcpyHostToDevice, st));
        PK_CUDA(cudaStreamSynchronize(st));
    }
    // fixed columns
    for (uint32_t c = 0; c < F; ++c) PK_CUDA(cudaMemcpyAsync(pk->fixed_values + (size_t)c * n, fixed_columns[c], n * sizeof(fe_t), cudaMemcpyHostToDevice, st));
    PK_CUDA(cudaMemcpyAsync(pk->fixed_polys, pk->fixed_values, F * n * sizeof(fe_t), cudaMemcpyDeviceToDevice, st));
    for (uint32_t c = 0; c < F; ++c) {
        PK_TRY(lagrange_to_coeff(pk, pk->fixed_polys + (size_t)c * n));
        PK_TRY(coeff_to_extended(pk, pk->fixed_polys + (size_t)c * n, pk->fixed_cosets + (size_t)c * ext));
    }
    PK_TRY(powers_run(ctx, dom->omega, n, pk->omega_pows));
    // permutation polynomials: sigma_c[r] = delta^map_col * omega^map_row
    if (P) {
        uint32_t *d_mc = nullptr, *d_mr = nullptr; fe_t* d_dp = nullptr;
        PK_TRY(dev_alloc(pk, &d_mc, P * n)); PK_TRY(dev_alloc(pk, &d_mr, P * n)); PK_TRY(dev_alloc(pk, &d_dp, P));
        for (size_t i = 0; i < (size_t)P * n; ++i) if (map_col[i] >= P || map_row[i] >= n) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "permutation mapping out of range"));
        PK_CUDA(cudaMemcpyAsync(d_mc, map_col, P * n * 4, cudaMemcpyHostToDevice, st));
        PK_CUDA(cudaMemcpyAsync(d_mr, map_row, P * n * 4, cudaMemcpyHostToDevice, st));
        PK_TRY(powers_run(ctx, host::fr_delta(), P, d_dp));
        sigma_kernel<<<nb((size_t)P * n), PK_THREADS, 0, st>>>(d_mc, d_mr, d_dp, pk->omega_pows, pk->perm_values, (size_t)P * n);
        ctx->launches++;
        PK_CUDA(cudaMemcpyAsync(pk->perm_polys, pk->perm_values, P * n * sizeof(fe_t), cudaMemcpyDeviceToDevice, st));
        for (uint32_t c = 0; c < P; ++c) {
            PK_TRY(lagrange_to_coeff(pk, pk->perm_polys + (size_t)c * n));
            PK_TRY(coeff_to_extended(pk, pk->perm_polys + (size_t)c * n, pk->perm_cosets + (size_t)c * ext));
        }
    }
    // l0, l_last, l_blind -> l_active_row
    {
        fe_t* tmp = nullptr; fe_t* lb = nullptr;
        PK_TRY(dev_alloc(pk, &tmp, n)); PK_TRY(dev_alloc(pk, &lb, ext));
        fe_t one = to_dev(HFr::one());
        auto indicator = [&](size_t lo, size_t hi, fe_t* out_ext) -> int32_t {
            ZK_CUDA(ctx, cudaMemsetAsync(tmp, 0, n * sizeof(fe_t), st));
            std::vector<fe_t> ones(hi - lo, one);
            ZK_CUDA(ctx, cudaMemcpyAsync(tmp + lo, ones.data(), ones.size() * sizeof(fe_t), cudaMemcpyHostToDevice, st));
            ZK_CUDA(ctx, cudaStreamSynchronize(st));
            ZK_TRY(lagrange_to_coeff(pk, tmp));
            return coeff_to_extended(pk, tmp, out_ext);
        };
        PK_TRY(indicator(0, 1, pk->l0));
        PK_TRY(indicator(n - cs.bf, n, lb));
        PK_TRY(indicator(n - cs.bf - 1, n - cs.bf, pk->l_last));
        one_minus_sum_kernel<<<nb(ext), PK_THREADS, 0, st>>>(pk->l_last, lb, pk->l_active, ext);
        ctx->launches++;
    }
    // programs: gates of each class with WSUM(acc0, gate); lookups with FOLD(acc0/acc1, theta)
    {
        std::vector<uint32_t> prog;
        // the gates, then the permutation terms (2 S + 1), then the lookup terms (5 L) fold in y in evaluate_h: gate i has
        // weight y^(G - 1 - i + 2 S + 1 + 5 L) in h.  The main class is multiplied by y^(2 S + 1) in the permutation kernels
        // and by y^(5 L) in the iNTT (or the lookup kernels when they share its cosets), the low class by y^(5 L) in the
        // lookup kernels; the linear class is added as it is.
        const uint32_t G = (uint32_t)cs.gates.size(), perm_terms = pk->S ? 2 * pk->S + 1 : 0;
        if (G >= EXW_INDEX) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "too many gate polynomials for this build"));
        for (uint32_t i = 0; i < G; ++i) {
            const uint32_t cls = pk->plan.gate_class[i];
            pk->gate_exp.push_back(G - 1 - i + (cls == QC_MAIN ? 0 : perm_terms) + (cls == QC_LINEAR ? 5 * pk->L : 0));
        }
        for (uint32_t cls = 0; cls < 3; ++cls) {
            std::vector<ExFold> items;
            for (uint32_t i = 0; i < G; ++i) if (pk->plan.gate_class[i] == cls) items.push_back({cs.gates[i].first, cs.gates[i].second, EX_WSUM | ((EXW_ACC0 | i) << 8)});
            const uint32_t off = (uint32_t)prog.size();
            if (!ex_share_common(cs.prog, items, prog, true)) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "malformed expression program"));
            pk->gate_prog[cls] = {off, (uint32_t)prog.size() - off};
        }
        if (G) {
            PK_TRY(dev_alloc(pk, &pk->d_wts, G));
            PK_CUDA(cudaMallocHost((void**)&pk->h_wts, G * sizeof(fe_t)));
        }
        for (auto& lk : cs.lookups) {
            uint32_t off = (uint32_t)prog.size();
            std::vector<ExFold> items;
            for (auto& e : lk.ins) items.push_back({e.first, e.second, EX_FOLD | ((0u << 4 | EXF_THETA) << 8)});
            for (auto& e : lk.tabs) items.push_back({e.first, e.second, EX_FOLD | ((1u << 4 | EXF_THETA) << 8)});
            if (!ex_share_common(cs.prog, items, prog)) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "malformed expression program"));
            pk->lookup_prog.push_back({off, (uint32_t)prog.size() - off});
        }
        // stack depth check
        int depth = 0, maxd = 0;
        for (uint32_t w : prog) {
            uint32_t op = w & 0xff;
            if (op <= EX_INSTANCE || op == EX_TMP) ++depth; else if (op == EX_ADD || op == EX_MUL || op == EX_FOLD || op == EX_WSUM || op == EX_GROUP) --depth;
            maxd = std::max(maxd, depth);
            if (depth < 0) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "malformed expression program"));
        }
        if (maxd > EX_STACK) return bail(fail(ctx, B200ZK_EINVAL, "pk_create", "expression too deep for the evaluator stack"));
        PK_TRY(dev_alloc(pk, &pk->d_prog, prog.size()));
        PK_CUDA(cudaMemcpyAsync(pk->d_prog, prog.data(), prog.size() * 4, cudaMemcpyHostToDevice, st));
        PK_TRY(dev_alloc(pk, &pk->d_consts, cs.consts.size()));
        PK_CUDA(cudaMemcpyAsync(pk->d_consts, cs.consts.data(), cs.consts.size() * sizeof(fe_t), cudaMemcpyHostToDevice, st));
        PK_TRY(dev_alloc(pk, &pk->d_q_adv, cs.adv_q.size())); PK_TRY(dev_alloc(pk, &pk->d_q_fix, cs.fix_q.size())); PK_TRY(dev_alloc(pk, &pk->d_q_inst, cs.inst_q.size()));
        PK_CUDA(cudaMemcpyAsync(pk->d_q_adv, cs.adv_q.data(), cs.adv_q.size() * 4, cudaMemcpyHostToDevice, st));
        PK_CUDA(cudaMemcpyAsync(pk->d_q_fix, cs.fix_q.data(), cs.fix_q.size() * 4, cudaMemcpyHostToDevice, st));
        PK_CUDA(cudaMemcpyAsync(pk->d_q_inst, cs.inst_q.data(), cs.inst_q.size() * 4, cudaMemcpyHostToDevice, st));
        PK_CUDA(cudaStreamSynchronize(st));
        PtrTab pt{cs.F, cs.A, cs.I};
        PK_TRY(dev_alloc(pk, &pk->d_ptrs, pt.total()));
    }
    {
        // early lookup cosets when their 4 L CL n elements are a modest share of the device (B200ZK_LOOKUP_EARLY=0/1 overrides)
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const size_t extra = 4 * (size_t)pk->L * pk->lk_cosets_n * pk->n * sizeof(fe_t);
        pk->lk_early = pk->L > 0 && extra <= free_b / 4;
        if (const char* e = getenv("B200ZK_LOOKUP_EARLY")) pk->lk_early = pk->L > 0 && e[0] != '0';
    }
    pk->arena_bytes = arena_need(pk);
    PK_TRY(dev_alloc(pk, &pk->arena, pk->arena_bytes));
    PK_CUDA(cudaStreamSynchronize(st));
    PK_CUDA(cudaGetLastError());
#undef PK_TRY
#undef PK_CUDA
    *out = pk;
    return B200ZK_OK;
}

static int32_t finish_proof(b200zk_pk* pk, int32_t rc, const std::vector<uint8_t>& proof, uint8_t* proof_out, size_t cap, size_t* proof_len) {
    // a rank that fails on its own (not the collective ConstraintSystemFailure / InstanceTooLarge) releases its peers
    if (rc != B200ZK_OK && rc != B200ZK_ESYNTH && pk->ctx->comm) pk->ctx->comm->abort();
    if (rc != B200ZK_OK) {
        // a failed proof may have left column uploads in flight: the caller's buffers are borrowed for the call only
        if (pk->copy_stream) cudaStreamSynchronize(pk->copy_stream);
        return rc;
    }
    if (proof_len) *proof_len = proof.size();
    if (proof.size() > cap) return fail(pk->ctx, B200ZK_EINVAL, "create_proof", "proof buffer too small");
    memcpy(proof_out, proof.data(), proof.size());
    return B200ZK_OK;
}

int32_t b200zk_create_proof(b200zk_pk* pk, const void* const* advice_columns, const void* const* instance_columns,
                            const uint32_t* instance_lens, const void* rng_wide, const void* transcript_repr,
                            uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
    if (!pk || !rng_wide || !transcript_repr || !proof_out || (pk->cs.A && !advice_columns) || (pk->cs.I && (!instance_columns || !instance_lens))) return B200ZK_EINVAL;
    std::vector<uint8_t> proof;
    int32_t rc = prove(pk, nullptr, false, advice_columns, instance_columns, instance_lens, rng_wide, false, HFr::from_limbs(transcript_repr), proof);
    return finish_proof(pk, rc, proof, proof_out, proof_cap, proof_len);
}

int32_t b200zk_create_proof_dev(b200zk_pk* pk, const void* d_advice, const void* const* instance_columns,
                                const uint32_t* instance_lens, const void* d_rng_wide, const void* transcript_repr,
                                uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
    if (!pk || !d_rng_wide || !transcript_repr || !proof_out || (pk->cs.A && !d_advice) || (pk->cs.I && (!instance_columns || !instance_lens))) return B200ZK_EINVAL;
    std::vector<uint8_t> proof;
    int32_t rc = prove(pk, (const fe_t*)d_advice, true, nullptr, instance_columns, instance_lens, d_rng_wide, true, HFr::from_limbs(transcript_repr), proof);
    return finish_proof(pk, rc, proof, proof_out, proof_cap, proof_len);
}

// ---- one create_proof over the GPUs of a group (b200zk_group_create): rank r = thread r on pks[r]'s device.
// Every rank gets the same inputs; the proof (identical on every rank) is rank 0's.
static int32_t group_prove(b200zk_group* g, b200zk_pk* const* pks, const void* const* d_advice_per_rank, const void* const* advice_columns,
                           const void* const* instance_columns, const uint32_t* instance_lens, const void* const* d_rng_per_rank,
                           const void* rng_wide, const void* transcript_repr, uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
    const uint32_t G = b200zk_group_size(g);
    if (!G || !pks || !transcript_repr || !proof_out) return B200ZK_EINVAL;
    for (uint32_t r = 0; r < G; ++r) {
        if (!pks[r] || pks[r]->ctx != b200zk_group_ctx(g, r)) return B200ZK_EINVAL;
        if (pks[r]->cs.I && (!instance_columns || !instance_lens)) return B200ZK_EINVAL;
        if (d_advice_per_rank ? (!d_rng_per_rank || (pks[r]->cs.A && !d_advice_per_rank[r]) || !d_rng_per_rank[r]) : (!rng_wide || (pks[r]->cs.A && !advice_columns))) return B200ZK_EINVAL;
    }
    b200zk_group_reset(g);
    std::vector<int32_t> rcs(G, B200ZK_OK);
    std::vector<std::vector<uint8_t>> proofs(G);
    const HFr repr = HFr::from_limbs(transcript_repr);
    auto body = [&](uint32_t r) {
        b200zk_pk* pk = pks[r];
        cudaSetDevice(pk->ctx->device);
        int32_t rc = d_advice_per_rank ? prove(pk, (const fe_t*)d_advice_per_rank[r], true, nullptr, instance_columns, instance_lens, d_rng_per_rank[r], true, repr, proofs[r])
                                       : prove(pk, nullptr, false, advice_columns, instance_columns, instance_lens, rng_wide, false, repr, proofs[r]);
        if (rc != B200ZK_OK && rc != B200ZK_ESYNTH) pk->ctx->comm->abort();
        if (rc != B200ZK_OK && pk->copy_stream) cudaStreamSynchronize(pk->copy_stream);
        rcs[r] = rc;
    };
    std::vector<std::thread> threads;
    for (uint32_t r = 1; r < G; ++r) threads.emplace_back(body, r);
    body(0);
    for (auto& t : threads) t.join();
    for (uint32_t r = 0; r < G; ++r) if (rcs[r] != B200ZK_OK) return rcs[r];
    for (uint32_t r = 1; r < G; ++r) if (proofs[r] != proofs[0]) return fail(pks[0]->ctx, B200ZK_ECUDA, "group_create_proof", "internal: ranks disagree on the proof");
    if (proof_len) *proof_len = proofs[0].size();
    if (proofs[0].size() > proof_cap) return fail(pks[0]->ctx, B200ZK_EINVAL, "create_proof", "proof buffer too small");
    memcpy(proof_out, proofs[0].data(), proofs[0].size());
    return B200ZK_OK;
}

int32_t b200zk_group_create_proof(b200zk_group* g, b200zk_pk* const* pks, const void* const* advice_columns, const void* const* instance_columns,
                                  const uint32_t* instance_lens, const void* rng_wide, const void* transcript_repr,
                                  uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
    return group_prove(g, pks, nullptr, advice_columns, instance_columns, instance_lens, nullptr, rng_wide, transcript_repr, proof_out, proof_cap, proof_len);
}

int32_t b200zk_group_create_proof_dev(b200zk_group* g, b200zk_pk* const* pks, const void* const* d_advice_per_rank, const void* const* instance_columns,
                                      const uint32_t* instance_lens, const void* const* d_rng_wide_per_rank, const void* transcript_repr,
                                      uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
    if (!d_advice_per_rank || !d_rng_wide_per_rank) return B200ZK_EINVAL;
    return group_prove(g, pks, d_advice_per_rank, nullptr, instance_columns, instance_lens, d_rng_wide_per_rank, nullptr, transcript_repr, proof_out, proof_cap, proof_len);
}

}  // extern "C"
