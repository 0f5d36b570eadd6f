// Internal context shared by the translation units of libb200zk.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <map>
#include <array>
#include <string>
#include <vector>
#include "../../include/b200zk.h"
#include "host_field.hpp"
#include "field.cuh"
#include "curve.cuh"
#include "ntt_plan.hpp"
#include "msm_plan.hpp"

namespace b200zk {

struct NttPlan {
    NttShape shape;
    fe_t* roots = nullptr;
    fe_t* tw_lo = nullptr;
    fe_t* tw_hi = nullptr;
    fe_t* tw_full = nullptr;    // omega^E for all E < N (multi-pass plans up to 2^24)
    bool warp = false;          // passes run on ntt_warp_pass_kernel (ntt_warp.cuh)
    struct fe2_t* roots_s = nullptr;    // {plain value, floor(value * 2^256 / r)} forms of roots / tw_full for Field::mul_shoup
    struct fe2_t* tw_full_s = nullptr;  // (warp plans only; null = CIOS multiplications against the Montgomery tables)
    bool borrowed = false;      // tables owned by another ctx on the same device (a proof lane's, prover.cu): not freed here
};

struct fe2_t;

struct Workspace {
    void* p = nullptr;
    size_t cap = 0;
    size_t used = 0;            // largest request since create_proof last reset it (the size a proof lane reserves)
};

struct Comm;                    // comm.hpp: the exchanges of a proof sharded over several GPUs

}  // namespace b200zk

struct b200zk_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;                                    // side stream: work independent of the transcript (advice cosets)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::string err;
    uint64_t launches = 0;
    cudaEvent_t events[64] = {};
    int sm_count = 148;
    int msm_force_c = 0;
    bool ntt_sparse_hint = false;                                      // next ntt_run: input is a Lagrange column (often zero outside the used rows)
    std::map<std::array<uint64_t, 5>, b200zk::NttPlan> ntt_plans;     // key: log_n + omega limbs
    b200zk::Workspace ntt_scratch, ntt_scratch2, msm_ws, msm_ws2, io_a, io_b, poly_ws, poly_heads, poly_batch, setup_ws, lookup_ws;
    b200zk::affine_t* d_gen_table = nullptr;                          // fixed-base table of the G1 generator (setup.cu)
    void* pinned = nullptr;                                            // small pinned staging (results)
    bool ntt_attr_set = false;                                         // cudaFuncSetAttribute is per device: once per ctx
    b200zk::Comm* comm = nullptr;                                      // set: create_proof on this ctx is one rank of a sharded proof
    bool comm_owned = false;                                           // comm created by b200zk_ctx_comm_init (not by a group)
};

struct b200zk_domain {
    b200zk_ctx* ctx;
    uint32_t k, extended_k, quotient_poly_degree;
    b200zk::host::HFr omega, omega_inv, extended_omega, extended_omega_inv, g_coset, g_coset_inv;
    b200zk::host::HFr ifft_divisor, extended_ifft_divisor, barycentric_weight;
    b200zk::fe_t* d_t_evaluations;           // 2^(extended_k - k), already inverted
};

namespace b200zk {
struct MsmPre {                 // fixed-base table geometry (msm.cu)
    MsmShape shape;
    uint32_t stride;            // points per window = the params' n
};
}  // namespace b200zk

struct b200zk_params {
    b200zk_ctx* ctx;
    uint32_t k;
    b200zk::affine_t* d_g;
    b200zk::affine_t* d_g_lagrange;
    // fixed-base tables T[j*n + i] = 2^(c j) * base_i (null when they would not fit in memory)
    b200zk::affine_t* d_g_pre;
    b200zk::affine_t* d_gl_pre;
    b200zk::MsmPre pre;
    // sum of all n points of each basis ([0] = g, [1] = g_lagrange) as an 8-bit fixed-window table
    // (32 x 255 multiples), built on first use by params_commit_run for constant-run columns
    std::vector<b200zk::host::HXyzz> sum_table[2];
};

namespace b200zk {

int32_t fail(b200zk_ctx* ctx, int32_t code, const char* what, const char* detail);

#define ZK_CUDA(ctx, expr)                                                          \
    do {                                                                            \
        cudaError_t _e = (expr);                                                    \
        if (_e != cudaSuccess) return fail((ctx), B200ZK_ECUDA, #expr, cudaGetErrorString(_e)); \
    } while (0)

#define ZK_TRY(expr)                      \
    do {                                  \
        int32_t _r = (expr);              \
        if (_r != B200ZK_OK) return _r;   \
    } while (0)

// grow-only device workspace
int32_t ws_reserve(b200zk_ctx* ctx, Workspace& w, size_t bytes);

// ntt.cu ---------------------------------------------------------------------
// out[i] = sum_j in[j] omega^(ij) over N = 2^log_n; in has n_in valid elements (rest
// read as zero).  pre/post: three host Fr multipliers indexed by position mod 3, or null.
// d_out may alias d_in.
int32_t ntt_run(b200zk_ctx* ctx, const fe_t* d_in, uint32_t n_in, fe_t* d_out, uint32_t log_n,
                const host::HFr& omega, const host::HFr* pre, const host::HFr* post, const fe_t* d_pre_tab = nullptr);
int32_t ntt_run_cosets(b200zk_ctx* ctx, const fe_t* d_in, fe_t* d_out, uint32_t log_n, const host::HFr& omega,
                       const fe_t* d_pre_tab, uint32_t batch);
// four-step sharded NTT building blocks (ntt.cu)
int32_t ntt_colstep_run(b200zk_ctx* ctx, fe_t* d_block, uint32_t log_r, uint32_t log_cg, uint32_t col0,
                        const host::HFr& omega_n, uint32_t log_n, fe_t* const* peer_rows = nullptr, uint32_t world = 0);
int32_t ntt_rows_run(b200zk_ctx* ctx, fe_t* d_rows, uint32_t nrows, const host::HFr& omega_c, uint32_t log_c, const host::HFr* post = nullptr);
// a[i] *= m[i mod period]  (divide_by_vanishing_poly), m on device
int32_t fr_scale_periodic(b200zk_ctx* ctx, fe_t* d_a, size_t n, const fe_t* d_m, uint32_t period);

// msm.cu ---------------------------------------------------------------------
int32_t msm_run(b200zk_ctx* ctx, const fe_t* d_scalars, const affine_t* d_bases, size_t n, host::HAffine* out);
// fixed-base variant: d_bases is a table built by msm_precompute_run (pre != null)
int32_t msm_run_multi(b200zk_ctx* ctx, const fe_t* const* d_cols, uint32_t ncols, const affine_t* d_bases, size_t n, const MsmPre* pre,
                      host::HAffine* outs, const fe_t* const* subs);
int32_t msm_run_ex(b200zk_ctx* ctx, const fe_t* d_scalars, const affine_t* d_bases, size_t n, const MsmPre* pre, host::HAffine* out,
                   const fe_t* sub = nullptr);
int32_t msm_precompute_run(b200zk_ctx* ctx, const affine_t* d_bases, size_t n, uint32_t c, uint32_t nwin, affine_t* d_table);
// commit over a params basis, through the fixed-base table when it exists
int32_t params_commit_run(b200zk_params* p, const fe_t* d_poly, size_t len, bool lagrange, host::HAffine* out);
int32_t params_commit_multi(b200zk_params* p, const fe_t* const* d_polys, uint32_t ncols, size_t len, bool lagrange, host::HAffine* outs);
// partial commitments over the point range [lo, hi): sum_{lo <= i < hi} poly[i] * basis[i] (one rank's share of a
// commit sharded by point range; the partial sums are added on the host)
int32_t params_commit_range(b200zk_params* p, const fe_t* const* d_polys, uint32_t ncols, size_t lo, size_t hi, bool lagrange, host::HAffine* outs);
// builds the fixed-base tables of a params object if memory allows (capi.cu)
int32_t params_build_tables(b200zk_params* p);
// builds the sum tables of both bases now (params_commit_multi otherwise builds them on first use), so that params views
// on other ctxs can copy them and nothing writes them while proofs run concurrently (capi.cu)
int32_t params_sum_tables(b200zk_params* p);

// poly.cu --------------------------------------------------------------------
int32_t batch_invert_run(b200zk_ctx* ctx, fe_t* d_a, size_t n, int field /* 0 Fr, 1 Fq */);
int32_t recurrence_run(b200zk_ctx* ctx, const fe_t* d_a, fe_t* d_y, size_t n, const host::HFr& b, host::HFr* head_out);
int32_t prefix_product_run(b200zk_ctx* ctx, const fe_t* d_p, fe_t* d_z, size_t n, const host::HFr& z0);
int32_t eval_batch_run(b200zk_ctx* ctx, const fe_t* const* h_polys, const host::HFr* h_points, size_t Q, size_t n, host::HFr* out);

// setup.cu -------------------------------------------------------------------
// ParamsKZG::setup bases on the device: g[i] = [s^i]G, g_lagrange[i] = [l_i(s)]G
int32_t params_setup_run(b200zk_ctx* ctx, uint32_t k, const host::HFr& s, affine_t* d_g, affine_t* d_g_lagrange);
// arithmetic::g_to_lagrange: d_out[i] = n^-1 * sum_j w^(-ij) d_g[j] over n = 2^k points (d_out may alias d_g)
int32_t g_to_lagrange_run(b200zk_ctx* ctx, const affine_t* d_g, uint32_t k, affine_t* d_out);

// out[i] = base^i, i < n (two-level tables built on the device)
int32_t powers_run(b200zk_ctx* ctx, const host::HFr& base, size_t n, fe_t* d_out);

// pairing.cu ------------------------------------------------------------------
// for j < count: status[j] = prod_{i < m} e(g1[j m + i], Q_{q[j m + i]}) == 1 ? B200ZK_OK : B200ZK_EVERIFY.  g1: host
// G1Affine on the curve; q: host indices into the nq G2Affine points g2 (128 B each, on the twist, not the identity), or
// PC_SKIP (pairing.cuh) for a pair that contributes 1.  Three launches; buffers in io_a and setup_ws.
int32_t pairing_checks_run(b200zk_ctx* ctx, const void* g1, const uint32_t* q, const void* g2, uint32_t nq, uint32_t m, uint32_t count,
                           int32_t* status);

// lookup_sort.cu --------------------------------------------------------------
int32_t lookup_permute_run(b200zk_ctx* ctx, const fe_t* d_in, const fe_t* d_tab, uint32_t u, fe_t* d_pin, fe_t* d_ptab, uint32_t* d_err);

}  // namespace b200zk
