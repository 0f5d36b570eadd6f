/* b200zk — C ABI of the B200-native halo2 (PSE fork, bn256 KZG) proving backend.
 *
 * Every entry point replaces one function of halo2_proofs v2023_02_02 /
 * halo2curves 0.3.1 (third-party crates pinned at /root/reference/Cargo.toml:10-11)
 * that the reference reaches from its only prover call site,
 * `full_prover` (/root/reference/src/circuits/utils.rs:22-70).  A patched
 * halo2_proofs binds these symbols over Rust FFI (see INTEGRATION.md); chips and
 * circuits recompile unchanged.
 *
 * Conventions
 *  - Field elements are 32-byte little-endian Montgomery limbs, exactly the
 *    in-memory layout of halo2curves `Fr([u64;4])` / `Fq([u64;4])`, so `&[Fr]`
 *    and `&[G1Affine]` are passed as plain pointers with no conversion.
 *    G1Affine = {x, y} 64 B (identity (0,0)); G1 = {x, y, z} Jacobian 96 B.
 *  - Every function returns 0 on success and a negative B200ZK_E* code on error;
 *    nothing is thrown across the boundary.  b200zk_last_error() gives the text.
 *    The Rust shim turns a non-zero code into the panic / plonk::Error the
 *    upstream function would have raised (e.g. length mismatch in best_multiexp).
 *  - A ctx owns one CUDA device, one stream and its scratch memory and is used by
 *    one caller thread at a time.  There is no CPU fallback: if no CUDA device is
 *    usable, ctx creation fails with B200ZK_ENODEV.
 *  - "_dev" variants take device pointers obtained from b200zk_malloc() and leave
 *    results on the device; the host variants copy in and out (H2D, kernel, D2H).
 */
#ifndef B200ZK_H
#define B200ZK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200ZK_OK 0
#define B200ZK_EINVAL (-1)   /* bad argument (length mismatch, log_n out of range ...) */
#define B200ZK_ENODEV (-2)   /* no usable CUDA device / extension unusable           */
#define B200ZK_ECUDA (-3)    /* CUDA runtime error, see b200zk_last_error            */
#define B200ZK_ENOMEM (-4)

typedef struct b200zk_ctx b200zk_ctx;
typedef struct b200zk_domain b200zk_domain;
typedef struct b200zk_params b200zk_params;

/* ---- context ------------------------------------------------------------ */
int32_t b200zk_ctx_create(int32_t device, b200zk_ctx** out);
void b200zk_ctx_destroy(b200zk_ctx* ctx);
const char* b200zk_last_error(const b200zk_ctx* ctx);
int32_t b200zk_sync(b200zk_ctx* ctx);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
uint64_t b200zk_launch_count(const b200zk_ctx* ctx);
/* cudaProfilerStart / cudaProfilerStop (for `ncu --profile-from-start off` captures of one step) */
int32_t b200zk_profiler_range(b200zk_ctx* ctx, int32_t start);
/* CUDA events on the ctx stream, for device-side timing of the calls in between */
int32_t b200zk_event_record(b200zk_ctx* ctx, uint32_t slot /* < 64 */);
int32_t b200zk_event_elapsed_ms(b200zk_ctx* ctx, uint32_t from_slot, uint32_t to_slot, float* ms);

/* ---- device memory -------------------------------------------------------- */
int32_t b200zk_malloc(b200zk_ctx* ctx, size_t bytes, void** dptr);
int32_t b200zk_free(b200zk_ctx* ctx, void* dptr);
int32_t b200zk_upload(b200zk_ctx* ctx, void* dptr, const void* host, size_t bytes);
int32_t b200zk_download(b200zk_ctx* ctx, void* host, const void* dptr, size_t bytes);
int32_t b200zk_memset_zero(b200zk_ctx* ctx, void* dptr, size_t bytes);
/* pinned host staging buffers (cudaHostAlloc) for the end-to-end path */
int32_t b200zk_host_alloc(b200zk_ctx* ctx, size_t bytes, void** hptr);
int32_t b200zk_host_free(b200zk_ctx* ctx, void* hptr);

/* ---- arithmetic::best_multiexp(coeffs: &[Fr], bases: &[G1Affine]) -> G1 ----
 * halo2_proofs src/arithmetic.rs.  out = sum coeffs[i] * bases[i], returned as a
 * Jacobian point with z = 1 (or the identity (0,1,0)): the same group element the
 * CPU path returns, in normalised representation.  len == 0 gives the identity. */
int32_t b200zk_msm(b200zk_ctx* ctx, const void* coeffs, const void* bases, size_t len, void* out_g1);
int32_t b200zk_msm_dev(b200zk_ctx* ctx, const void* d_coeffs, const void* d_bases, size_t len, void* out_g1_host);
/* Host-side sum of `count` G1 points (96 B Jacobian each): combines the per-GPU partial results of a
 * point-range sharded best_multiexp after a 96-byte all-gather (no ctx, no device work). */
int32_t b200zk_g1_sum(const void* points_g1, size_t count, void* out_g1);
/* window size override for tuning (0 = automatic) */
int32_t b200zk_msm_set_window(b200zk_ctx* ctx, int32_t c);

/* ---- arithmetic::best_fft(a: &mut [Fr], omega: Fr, log_n: u32) --------------
 * In place, natural order in and out, unscaled:  a[i] <- sum_j a[j] omega^(ij). */
int32_t b200zk_fft(b200zk_ctx* ctx, void* a, const void* omega, uint32_t log_n);
int32_t b200zk_fft_dev(b200zk_ctx* ctx, void* d_a, const void* omega_host, uint32_t log_n);

/* Building blocks of one best_fft of size N = R*C sharded over several GPUs (four-step, SURVEY.md
 * 8(e)): colstep = this rank's [R][Cg] column block (Cg = 2^log_cg columns from global column
 * col0): R-point transforms down the columns + twiddle omega_n^((col0+c)*k_r), in place, R <= 2^10;
 * rows = nrows contiguous natural-order transforms of size 2^log_c (after the all-to-all). */
int32_t b200zk_fft_colstep_dev(b200zk_ctx* ctx, void* d_block, uint32_t log_r, uint32_t log_cg, uint32_t col0,
                               const void* omega_n, uint32_t log_n);
int32_t b200zk_fft_rows_dev(b200zk_ctx* ctx, void* d_rows, uint32_t nrows, const void* omega_c, uint32_t log_c);
/* Column step fused with the all-to-all that follows it: transformed row k is written straight into
 * peer_rows[k / (R / world)] (that rank's (R / world) x C row buffer, opened with b200zk_ipc_open) at
 * [k mod (R / world)][col0 + c] — NVLink / NVSwitch peer stores from inside the kernel, no staging
 * buffer and no separate exchange.  d_block is read only.  The caller synchronises the ranks
 * (every rank's stream, then a barrier) before the row step.  world: power of two <= 8. */
int32_t b200zk_fft_colstep_scatter_dev(b200zk_ctx* ctx, void* d_block, uint32_t log_r, uint32_t log_cg, uint32_t col0,
                                       const void* omega_n, uint32_t log_n, void* const* peer_rows, uint32_t world);
/* CUDA IPC for one-process-per-GPU hosts: export a b200zk_malloc'ed buffer (64-byte handle), open /
 * close a peer's handle in this process. */
int32_t b200zk_ipc_get_handle(b200zk_ctx* ctx, const void* d_ptr, void* handle64);
int32_t b200zk_ipc_open(b200zk_ctx* ctx, const void* handle64, void** d_ptr);
int32_t b200zk_ipc_close(b200zk_ctx* ctx, void* d_ptr);

/* ---- poly::EvaluationDomain<Fr> (src/poly/domain.rs) ------------------------
 * b200zk_domain_create(j, k) = EvaluationDomain::new(j, k). */
int32_t b200zk_domain_create(b200zk_ctx* ctx, uint32_t j, uint32_t k, b200zk_domain** out);
void b200zk_domain_destroy(b200zk_domain* dom);
uint32_t b200zk_domain_k(const b200zk_domain* dom);
uint32_t b200zk_domain_extended_k(const b200zk_domain* dom);
uint32_t b200zk_domain_quotient_poly_degree(const b200zk_domain* dom);
/* which: 0 omega, 1 omega_inv, 2 extended_omega, 3 extended_omega_inv, 4 g_coset,
 *        5 g_coset_inv, 6 ifft_divisor, 7 extended_ifft_divisor, 8 barycentric_weight */
int32_t b200zk_domain_constant(const b200zk_domain* dom, uint32_t which, void* out_fr);
/* rotate_omega(value, rotation) = value * omega^rotation;  l_i_range(x, x^n, rot_lo..=rot_hi): the Lagrange
 * basis polynomials l_i(x), i = rot_lo .. rot_hi (negative i counts from the end of the domain), rot_hi - rot_lo + 1
 * elements out;  rotate_extended: out[i] = in[(i + rotation * 2^(extended_k - k)) mod 2^extended_k] (out != in). */
int32_t b200zk_domain_rotate_omega(const b200zk_domain* dom, const void* value_fr, int32_t rotation, void* out_fr);
int32_t b200zk_domain_l_i_range(const b200zk_domain* dom, const void* x_fr, int32_t rot_lo, int32_t rot_hi, void* out_fr);
int32_t b200zk_rotate_extended_dev(b200zk_domain* dom, const void* d_in, int32_t rotation, void* d_out);
/* lagrange_to_coeff: n elements in place */
int32_t b200zk_lagrange_to_coeff(b200zk_domain* dom, void* a);
int32_t b200zk_lagrange_to_coeff_dev(b200zk_domain* dom, void* d_a);
/* coeff_to_extended: n coefficients in, 2^extended_k evaluations out */
int32_t b200zk_coeff_to_extended(b200zk_domain* dom, const void* coeffs, void* out_ext);
int32_t b200zk_coeff_to_extended_dev(b200zk_domain* dom, const void* d_coeffs, void* d_out_ext);
/* extended_to_coeff: 2^extended_k evaluations in (clobbered in the _dev variant),
 * n * quotient_poly_degree coefficients out */
int32_t b200zk_extended_to_coeff(b200zk_domain* dom, const void* ext, void* out_coeffs);
int32_t b200zk_extended_to_coeff_dev(b200zk_domain* dom, void* d_ext, void* d_out_coeffs);
/* divide_by_vanishing_poly: 2^extended_k evaluations in place */
int32_t b200zk_divide_by_vanishing_poly(b200zk_domain* dom, void* ext);
int32_t b200zk_divide_by_vanishing_poly_dev(b200zk_domain* dom, void* d_ext);

/* ---- poly::kzg::commitment::ParamsKZG<Bn256> ---------------------------------
 * load: upload an existing SRS (g, g_lagrange: n G1Affine each; g_lagrange may be
 * NULL).  setup: ParamsKZG::setup(k, rng) with the secret s supplied by the caller
 * (s = Fr::random(rng) on the Rust side); bases are generated on the device. */
int32_t b200zk_params_load(b200zk_ctx* ctx, uint32_t k, const void* g, const void* g_lagrange, b200zk_params** out);
int32_t b200zk_params_setup(b200zk_ctx* ctx, uint32_t k, const void* s_fr, b200zk_params** out);
void b200zk_params_destroy(b200zk_params* p);
/* copy the bases back (get_g / g_lagrange), n * 64 bytes each; either may be NULL */
int32_t b200zk_params_read(b200zk_params* p, void* g_out, void* g_lagrange_out);
/* commit(poly: Coeff) / commit_lagrange(poly: LagrangeCoeff); len <= n */
int32_t b200zk_commit(b200zk_params* p, const void* poly, size_t len, void* out_g1);
int32_t b200zk_commit_lagrange(b200zk_params* p, const void* poly, size_t len, void* out_g1);
int32_t b200zk_commit_dev(b200zk_params* p, const void* d_poly, size_t len, int32_t lagrange, void* out_g1_host);
/* `count` polynomials of the same length in one batched launch sequence — what create_proof's
 * column loops (`advice.iter().map(|poly| params.commit_lagrange(poly, blind))`, plonk/prover.rs)
 * amount to; d_polys: host array of `count` device pointers, out: count * 96 bytes on the host. */
int32_t b200zk_commit_many_dev(b200zk_params* p, const void* const* d_polys, uint32_t count, size_t len, int32_t lagrange,
                               void* out_g1_host);
/* arithmetic::g_to_lagrange(g, k): the Lagrange basis n^-1 · FFT_{ω^-1}(g) of n = 2^k G1Affine points
 * (any points; identity = (0,0)), as G1Affine.  out may alias g.  k <= 28. */
int32_t b200zk_g_to_lagrange(b200zk_ctx* ctx, const void* g, uint32_t k, void* out);
int32_t b200zk_g_to_lagrange_dev(b200zk_ctx* ctx, const void* d_g, uint32_t k, void* d_out);
/* ParamsKZG::downsize(k): new params on p's ctx holding g[..2^k] of p and its Lagrange basis, with
 * the fixed-base tables built as params_load builds them.  p is not changed; k <= p's k.
 * With k = p's k it derives the Lagrange basis of params loaded without one.
 * Upstream's downsize truncates `&mut self` in place; returning a new handle instead keeps every
 * proving key built on p valid.  Destroy both handles independently. */
int32_t b200zk_params_downsize(const b200zk_params* p, uint32_t k, b200zk_params** out);

/* ---- arithmetic::eval_polynomial / kate_division, ff::BatchInvert -----------------
 * eval_polynomial(poly, x) -> Fr (Horner);  kate_division(a, b): quotient of a(X) by
 * (X - b), len-1 coefficients;  batch_invert: in place, zeros stay zero.
 * field: 0 = Fr, 1 = Fq. */
int32_t b200zk_eval_polynomial(b200zk_ctx* ctx, const void* poly, size_t len, const void* x_fr, void* out_fr);
int32_t b200zk_eval_polynomial_dev(b200zk_ctx* ctx, const void* d_poly, size_t len, const void* x_fr, void* out_fr_host);
int32_t b200zk_kate_division_dev(b200zk_ctx* ctx, const void* d_a, size_t len, const void* b_fr, void* d_q);
int32_t b200zk_batch_invert_dev(b200zk_ctx* ctx, void* d_a, size_t len, int32_t field);
/* z[0] = z0, z[i] = z[i-1] * p[i-1]: the grand-product scan of the permutation and lookup
 * arguments (plonk/permutation/prover.rs, plonk/lookup/prover.rs).  d_z may alias d_p. */
int32_t b200zk_prefix_product_dev(b200zk_ctx* ctx, const void* d_p, void* d_z, size_t len, const void* z0_fr);

/* ---- plonk::keygen_pk / plonk::create_proof (src/plonk/keygen.rs, src/plonk/prover.rs) --------
 * The call `full_prover` makes at /root/reference/src/circuits/utils.rs:35 and :40-48, for one
 * circuit instance with KZGCommitmentScheme<Bn256>, ProverSHPLONK, Challenge255 and Blake2bWrite.
 *
 * pk_create: cs_blob is the constraint-system description (column counts, query lists, gate and
 * lookup expressions, permutation columns — the serialisation is documented in
 * halo2-experiments_b200/circuit.py::ConstraintSystem.to_blob); fixed_columns are the F fixed
 * columns (selectors already compressed into them) as n Lagrange values each; map_col/map_row are
 * the permutation Assembly's mapping (P x n, row-major): cell (c, r) maps to
 * (map_col[c*n+r], map_row[c*n+r]).  Everything derived (polys, cosets, sigma, l0/l_last/
 * l_active_row) is computed on the device and stays resident in HBM.
 *
 * create_proof: advice_columns = A columns of n Lagrange values as produced by witness synthesis
 * (batch-inverted, not yet blinded); instance_columns / instance_lens = the public inputs;
 * rng_wide = the 64-byte little-endian inputs of every Fr::random(rng) call create_proof makes, in
 * call order (b200zk_pk_rng_draws() of them: the Rust shim fills it from the caller's RngCore, so
 * the proof is a pure function of its inputs); transcript_repr = vk.transcript_repr (Fr).
 * The proof bytes are exactly what `transcript.finalize()` returns.
 * Returns B200ZK_ESYNTH for upstream's Error::ConstraintSystemFailure (lookup input not in table)
 * and Error::InstanceTooLarge. */
#define B200ZK_ESYNTH (-5)
typedef struct b200zk_pk b200zk_pk;
int32_t b200zk_pk_create(b200zk_params* params, const uint32_t* cs_blob, size_t blob_words,
                         const void* const* fixed_columns, const uint32_t* map_col, const uint32_t* map_row,
                         b200zk_pk** out);
void b200zk_pk_destroy(b200zk_pk* pk);
size_t b200zk_pk_proof_size(const b200zk_pk* pk);
size_t b200zk_pk_rng_draws(const b200zk_pk* pk);
uint32_t b200zk_pk_blinding_factors(const b200zk_pk* pk);
uint32_t b200zk_pk_degree(const b200zk_pk* pk);
int32_t b200zk_create_proof(b200zk_pk* pk, const void* const* advice_columns, const void* const* instance_columns,
                            const uint32_t* instance_lens, const void* rng_wide, const void* transcript_repr,
                            uint8_t* proof_out, size_t proof_cap, size_t* proof_len);
/* same, with the advice columns (A x n, contiguous) and the rng stream already in device memory */
int32_t b200zk_create_proof_dev(b200zk_pk* pk, const void* d_advice, const void* const* instance_columns,
                                const uint32_t* instance_lens, const void* d_rng_wide, const void* transcript_repr,
                                uint8_t* proof_out, size_t proof_cap, size_t* proof_len);
/* ---- many proofs of one pk on its device, side by side (an extension: upstream has no such call) --------
 * Proofs of `count` independent witnesses of one pk, run concurrently on the pk's device.  Proof i is byte for byte
 * what b200zk_create_proof returns for the inputs of proof i: advice_columns[i*A + c], instance_columns[i*I + c],
 * instance_lens[i*I + c], rng_wide[i]; one transcript_repr for all (one vk).  proofs_out holds
 * count * b200zk_pk_proof_size(pk) bytes, proof i starting at i * proof_size; status[i] is 0 or that proof's error.
 * Returns B200ZK_OK when every proof succeeded, B200ZK_ESYNTH when the only failures were ConstraintSystemFailure /
 * InstanceTooLarge (status says which; the other proofs are produced), any other code when a proof failed otherwise
 * (b200zk_last_error(pk's ctx) names the proof; proofs the call did not reach get that code in status).
 * B200ZK_EINVAL before any work for null pointers, count == 0, proofs_cap < count * proof_size, and for a pk whose ctx
 * is one rank of a sharded proof.  The pk and its ctx stay usable after any failure.
 * A lane is what one proof in flight needs: lane 0 is the pk's own state on its ctx; every further lane has an
 * internal ctx on the same device and its own arena (one arena and the workspaces of one proof, see DESIGN.md),
 * and shares the key, the SRS tables and the NTT plans.  Lanes run on library threads; the calling thread runs lane 0.
 * b200zk_pk_last_phase_ms / _last_trace / _debug_buffer describe the last proof lane 0 ran; b200zk_launch_count(ctx)
 * includes the launches of every lane.  The lane count is min(count, a cap, what fits in half of the free device
 * memory); B200ZK_PROOF_LANES=N replaces the cap.  Fewer lanes than asked when memory is short is not an error. */
int32_t b200zk_create_proofs(b200zk_pk* pk, uint32_t count, const void* const* advice_columns, const void* const* instance_columns,
                             const uint32_t* instance_lens, const void* const* rng_wide, const void* transcript_repr,
                             uint8_t* proofs_out, size_t proofs_cap, int32_t* status);
/* d_advice[i] = proof i's A x n advice block, d_rng_wide[i] = its draws, both in device memory (as create_proof_dev) */
int32_t b200zk_create_proofs_dev(b200zk_pk* pk, uint32_t count, const void* const* d_advice, const void* const* instance_columns,
                                 const uint32_t* instance_lens, const void* const* d_rng_wide, const void* transcript_repr,
                                 uint8_t* proofs_out, size_t proofs_cap, int32_t* status);
/* reserve up to `want` lanes now (0 = the planner's default) and use that request for later batches; *got = what
 * memory allowed, >= 1.  Before the pk's first proof the planner knows a lane's arena but not the workspaces a proof
 * needs, so *got is provisional then: a later batch reserves those workspaces and runs on fewer lanes if they do not
 * fit.  A lane that cannot get its memory is never an error. */
int32_t b200zk_pk_reserve_lanes(b200zk_pk* pk, uint32_t want, uint32_t* got);

/* ---- one create_proof sharded over several GPUs (BASELINE config 5; SURVEY.md 8(e)) ---------------
 * The reference's single prover call (/root/reference/src/circuits/utils.rs:40-48) spread over G GPUs of
 * one NVLink / NVSwitch box.  Every rank holds the SRS and the proving key (b200zk_params_* / b200zk_pk_create
 * on its own ctx) and receives the same inputs; inside the call each rank commits its share of the
 * columns, runs its lookups, extends and evaluates its quotient cosets and multiplies its point range of the
 * dense commitments (h pieces, random polynomial, SHPLONK), exchanging polynomials device to device and
 * 64-byte partial sums through the host, so that every rank's Blake2b transcript absorbs the same bytes.
 * The proof is byte-identical to the single-GPU one.
 *
 * (a) One process per GPU (torchrun / MPI style hosts): rank 0 calls b200zk_comm_unique_id and
 *     distributes the 128 bytes; every rank calls b200zk_ctx_comm_init (NCCL; collective), after which
 *     b200zk_create_proof[_dev] on that ctx is one rank of the sharded proof: all ranks call it with the
 *     same arguments and all receive the proof.  libnccl.so.2 is loaded on first use.
 * (b) One process driving several GPUs (what a Rust `create_proof` caller uses): b200zk_group_create
 *     makes one ctx per listed device with peer access between them; build params / pk on every
 *     b200zk_group_ctx(g, r), then b200zk_group_create_proof runs the ranks on internal threads (no
 *     NCCL, NVLink peer copies).  A device may be listed more than once (the ranks then share it):
 *     that is how the sharded prover is tested on a single GPU. */
typedef struct b200zk_group b200zk_group;
int32_t b200zk_comm_unique_id(void* id_out128);
int32_t b200zk_ctx_comm_init(b200zk_ctx* ctx, uint32_t world, uint32_t rank, const void* id128);
int32_t b200zk_ctx_comm_destroy(b200zk_ctx* ctx);
uint32_t b200zk_ctx_comm_world(const b200zk_ctx* ctx);
uint32_t b200zk_ctx_comm_rank(const b200zk_ctx* ctx);
int32_t b200zk_group_create(const int32_t* devices, uint32_t n, b200zk_group** out);
void b200zk_group_destroy(b200zk_group* g);            /* destroys the group's ctxs: free their params / pks first */
uint32_t b200zk_group_size(const b200zk_group* g);
b200zk_ctx* b200zk_group_ctx(b200zk_group* g, uint32_t rank);
int32_t b200zk_group_reset(b200zk_group* g);           /* after a failed group call */
/* arithmetic::best_multiexp / best_fft over the group's GPUs, host buffers in and out: the multiexp is split by point
 * range (partial sums added inside the call); the fft runs four-step with the exchange fused into the column-step
 * kernel (NVLink peer stores) when the group is 2, 4 or 8 devices and log_n >= 16, on rank 0 otherwise. */
int32_t b200zk_group_msm(b200zk_group* g, const void* coeffs, const void* bases, size_t len, void* out_g1);
int32_t b200zk_group_fft(b200zk_group* g, void* a, const void* omega, uint32_t log_n);
/* pks[r] = the proving key built on b200zk_group_ctx(g, r) */
int32_t b200zk_group_create_proof(b200zk_group* g, b200zk_pk* const* pks, const void* const* advice_columns,
                                  const void* const* instance_columns, const uint32_t* instance_lens, const void* rng_wide,
                                  const void* transcript_repr, uint8_t* proof_out, size_t proof_cap, size_t* proof_len);
/* d_advice_per_rank[r] / d_rng_wide_per_rank[r]: the inputs resident on rank r's device */
int32_t b200zk_group_create_proof_dev(b200zk_group* g, b200zk_pk* const* pks, const void* const* d_advice_per_rank,
                                      const void* const* instance_columns, const uint32_t* instance_lens,
                                      const void* const* d_rng_wide_per_rank, const void* transcript_repr,
                                      uint8_t* proof_out, size_t proof_cap, size_t* proof_len);

/* debugging aid: copy a named device buffer of the last proof (32-byte elements) to the host */
int32_t b200zk_pk_debug_buffer(b200zk_pk* pk, const char* name, void* host_out, size_t max_elems, size_t* count);
/* per-phase device times (ms) of the last create_proof: msm, ntt, quotient, lookup, permutation, evals+shplonk,
 * other (= time spent in / waiting at the exchanges of a sharded proof) */
int32_t b200zk_pk_last_phase_ms(const b200zk_pk* pk, float* out7);
/* host wall clock (ms since the call) at the synchronisation points of the last create_proof, as
 * "label:ms;label:ms;...": advice_commits, lookup_permuted_commits, perm_products, permutation_commits, lookup_product_commits,
 * quotient_and_h_commits, evaluations, shplonk_h1_commit, end */
int32_t b200zk_pk_last_trace(const b200zk_pk* pk, char* out, size_t cap);
/* field multiplications evaluate_h executes per row: {custom gates, permutation terms, all lookups, q, lookup cosets}
 * (the work model of bench.py's roofline_quotient) */
int32_t b200zk_pk_quotient_muls(const b200zk_pk* pk, uint32_t out5[5]);

/* ---- plonk::keygen_vk / plonk::verify_proof (src/plonk/keygen.rs, src/plonk/verifier.rs,
 *      src/poly/kzg/multiopen/shplonk/verifier.rs, src/poly/kzg/strategy.rs) ----------------------
 * The call `full_prover` makes at /root/reference/src/circuits/utils.rs:52-63 with VerifierSHPLONK,
 * SingleStrategy, Challenge255 and Blake2bRead, for one circuit instance.
 *
 * pk_vk_commitments: the commitments a VerifyingKey holds (keygen_vk's O(n) work, on the device):
 * F fixed-column commitments and P permutation (sigma) commitments, 64-byte G1Affine each.
 *
 * verify_proof runs on the caller's thread without a ctx or a device (O(#queries) field work, ~100
 * G1 scalar multiplications, two Miller loops) — like upstream's verifier it needs nothing of size n.
 * cs_blob as in pk_create; g1_generator = params.get_g()[0]; g2 / s_g2 = ParamsKZG's [1]_2 and
 * [s]_2 as G2Affine (x.c0, x.c1, y.c0, y.c1: 4 x 32-byte Montgomery Fq, halo2curves' layout).
 * Returns 0 for Ok(()), B200ZK_EVERIFY for every Err upstream returns (malformed or non-canonical
 * proof elements, instance too large, the final pairing check failing), B200ZK_EINVAL for a bad
 * argument.  Bytes after the last proof element are ignored, as upstream's reader ignores them. */
#define B200ZK_EVERIFY (-6)
int32_t b200zk_pk_vk_commitments(b200zk_pk* pk, void* fixed_out, void* sigma_out);
int32_t b200zk_verify_proof(const uint32_t* cs_blob, size_t blob_words, const void* fixed_commitments,
                            const void* sigma_commitments, const void* g1_generator, const void* g2, const void* s_g2,
                            const void* const* instance_columns, const uint32_t* instance_lens,
                            const void* transcript_repr, const uint8_t* proof, size_t proof_len);
/* ---- many proofs of one verifying key with one pairing check (an extension in the sense of b200zk_create_proofs) ----
 * Upstream's AccumulatorStrategy (src/poly/kzg/strategy.rs) over VerifierSHPLONK / Blake2bRead / Challenge255.
 * Inputs: as b200zk_verify_proof, for `count` proofs of one vk.  Proof i uses instance_columns[i*I + c],
 * instance_lens[i*I + c] (the indexing of b200zk_create_proofs) and proofs[i] / proof_lens[i]; all proofs share
 * transcript_repr.
 * Randomness: r_i = Fr::from_bytes_wide(rng_wide[64 i .. 64 i + 64]), one draw per proof, as `process` draws one
 * Fr::random per proof; the call is a pure function of its inputs.  The draws MUST be fresh and secret for every call
 * (the Rust shim fills them from OsRng): a prover who can predict them can make a batch with false proofs pass.
 * Stage 1, per proof, exactly the replay of b200zk_verify_proof: a proof that is malformed or truncated, has a
 * non-canonical scalar or point, a point off the curve, an instance that is too large, x^n = 1 or z_0 = 0 gets
 * status[i] = B200ZK_EVERIFY and adds nothing to the accumulator.  Bytes after the last proof element are ignored.
 * Points are decompressed on the device; the transcripts are replayed on a pool of library threads.
 * Accumulator: accumulator_out (if not NULL) receives (left, right) = sum_i c_i (h2_i, u_i h2_i + L_i / z0_i) over the
 * proofs that passed stage 1, c_i = r_{i+1} * ... * r_{count-1}, as two 64-byte G1Affine (identity (0,0)).  When every
 * proof passes stage 1 this is the DualMSM AccumulatorStrategy holds after `process` on proofs 0 .. count-1 in order.
 * Stage 2: one pairing check e(left, [s]_2) e(-right, [1]_2) = 1.  If it fails, one device call (the three kernels of
 * b200zk_pairing_checks) checks every stage-1 survivor's own c_i-scaled pair, so status[i] is then exactly
 * verify_proof's verdict for proof i, and the launch count does not depend on how many proofs fail.  Every status[i]
 * ends 0 or B200ZK_EVERIFY.
 * Returns B200ZK_OK when every proof is accepted, B200ZK_EVERIFY when at least one is rejected (status says which),
 * B200ZK_EINVAL before any device work for a bad argument (null pointers, count == 0, a cs blob that does not parse,
 * proofs[i] == NULL with a nonzero length, an invalid G2 point; b200zk_launch_count does not move), otherwise the CUDA
 * or memory code.  ctx may be any ctx, a rank of a sharded group or one holding a pk with lanes included: the call uses
 * only its stream and workspaces and leaves any pk on it untouched. */
int32_t b200zk_verify_proofs(b200zk_ctx* ctx, const uint32_t* cs_blob, size_t blob_words,
                             const void* fixed_commitments, const void* sigma_commitments,
                             const void* g1_generator, const void* g2, const void* s_g2,
                             uint32_t count, const void* const* instance_columns, const uint32_t* instance_lens,
                             const void* transcript_repr, const uint8_t* const* proofs, const size_t* proof_lens,
                             const void* rng_wide /* count * 64 bytes */, int32_t* status /* count */,
                             void* accumulator_out /* 2 x 64-byte G1Affine (left, right), or NULL */);
/* ParamsKZG::setup's G2 side: out = s * base (base NULL = the G2 generator, i.e. out = [s]_2). */
int32_t b200zk_g2_mul(const void* g2_or_null, const void* s_fr, void* out_g2);
/* prod e(g1_points[i], g2_points[i]) == 1 ?  0 = yes, B200ZK_EVERIFY = no (Engine::pairing product;
 * G1Affine 64 B, G2Affine 128 B each). */
int32_t b200zk_pairing_check(const void* g1_points, const void* g2_points, size_t count);
/* Many pairing-product checks in one call, on the device (halo2curves' multi_miller_loop(..).final_exponentiation()
 * compared with the identity, batched; e.g. one DualMSM::check per accumulator of a pile):
 * for j < count: prod_{i < m} e(g1_points[j*m + i], g2_points[j*m + i]) == 1 ?  status[j] = 0 or B200ZK_EVERIFY.
 * G1Affine 64 B, G2Affine 128 B (the layout of b200zk_pairing_check); a pair with an identity on either side
 * contributes 1.  The pairing is b200zk_pairing_check's, so every verdict is the one it gives for the same m pairs.
 * G2 points are compared by their bytes: each distinct point's Miller-loop lines are computed once per call.
 * Returns B200ZK_OK when every check holds, B200ZK_EVERIFY when at least one fails, B200ZK_EINVAL before any device
 * work (b200zk_launch_count does not move) for null pointers, count == 0, m == 0 or a point off its curve, otherwise
 * the CUDA or memory code.  Runs on the ctx stream with the ctx workspaces; three launches. */
int32_t b200zk_pairing_checks(b200zk_ctx* ctx, const void* g1_points, const void* g2_points,
                              uint32_t m, uint32_t count, int32_t* status);

/* ---- formats (SURVEY.md 8(f3)): halo2_proofs v2023_02_02 ParamsKZG::write / read (src/poly/kzg/commitment.rs),
 *      VerifyingKey::write / read commitments (src/plonk.rs), halo2curves G1Affine / G2Affine to_bytes / from_bytes,
 *      and vk.transcript_repr -------------------------------------------------------------------------------------
 * params_serialize = ParamsKZG::write: k (u32 LE) | n compressed G1 (g) | n compressed G1 (g_lagrange) | g2 | s_g2
 * (64-byte compressed G2 each); the 2n points are compressed / decompressed on the device (one Fq exponentiation per
 * point to recover y).  g2 / s_g2 cross as 128-byte G2Affine (x.c0, x.c1, y.c0, y.c1 Montgomery limbs).  deserialize
 * rejects non-canonical coordinates and points off the curve (B200ZK_EINVAL).
 * vk_serialize = the commitments VerifyingKey::write emits: fixed count (u32 BE) | fixed | permutation commitments.
 * vk_transcript_repr: the Fr create_proof / verify_proof absorb first.  Upstream hashes Rust's `{:?}` rendering of the
 * pinned key, which cannot be restated outside Rust, so a Rust host passes upstream's value; this entry derives a
 * value with the same role for other hosts: Blake2b-512 (personal "Halo2-Verify-Key") over (len u64 LE) | cs blob |
 * fixed | permutation commitments (uncompressed), then from_bytes_wide.  It binds k, the constraint system and the
 * commitments into every challenge; it is NOT upstream's value. */
size_t b200zk_params_serialized_size(uint32_t k, int32_t with_lagrange);
int32_t b200zk_params_serialize(b200zk_params* p, const void* g2, const void* s_g2, uint8_t* out, size_t cap, size_t* len);
int32_t b200zk_params_deserialize(b200zk_ctx* ctx, const uint8_t* in, size_t len, b200zk_params** out, void* g2_out, void* s_g2_out);
int32_t b200zk_g1_to_bytes(const void* affine_points, size_t count, uint8_t* out32);
int32_t b200zk_g1_from_bytes(const uint8_t* in32, size_t count, void* affine_out);     /* B200ZK_EVERIFY for an invalid encoding */
size_t b200zk_vk_serialized_size(uint32_t num_fixed, uint32_t num_sigma);
int32_t b200zk_vk_serialize(const void* fixed_commitments, uint32_t num_fixed, const void* sigma_commitments, uint32_t num_sigma,
                            uint8_t* out, size_t cap);
int32_t b200zk_vk_deserialize(const uint8_t* in, size_t len, uint32_t num_sigma, void* fixed_out, uint32_t fixed_cap,
                              uint32_t* num_fixed, void* sigma_out);
int32_t b200zk_vk_transcript_repr(const uint32_t* cs_blob, size_t blob_words, const void* fixed_commitments,
                                  const void* sigma_commitments, void* out_fr);

#ifdef __cplusplus
}
#endif
#endif /* B200ZK_H */
