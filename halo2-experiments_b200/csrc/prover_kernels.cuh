// Per-row device bodies of the prover's O(n) / O(ext) steps — everything in
// halo2_proofs v2023_02_02 create_proof (plonk/prover.rs, reached from
// /root/reference/src/circuits/utils.rs:40-48) that is neither an MSM, an NTT nor a scan:
//   plonk/permutation/prover.rs  Argument::commit           perm_denominator / perm_numerator
//   plonk/lookup/prover.rs       commit_product             lookup_den / lookup_num
//   plonk/evaluation.rs          evaluate_h (permutation and lookup parts)   quot_*
//   plonk/vanishing/prover.rs    evaluate (h pieces folded in x^n)           fold_pieces
//   poly/kzg/multiopen/shplonk/prover.rs  linear combinations of polynomials  axpy / scale
//   halo2curves Fr::random = from_u512                       from_u512_row
// Field arithmetic is exact, so any evaluation order gives the same canonical element.
#pragma once
#include "field.cuh"

namespace b200zk {

static constexpr int ZK_MAXC = 16;      // columns per permutation set (d - 2) / number of sets handled per launch
static constexpr int ZK_MAXCOSETS = 32; // cosets of the quotient domain (d - 1 <= 17)

// The prover's "extended" arrays hold C = d - 1 cosets of the size-n domain back to back:
// row idx = j * n + i is the evaluation at  zeta * extended_omega^j * omega^i  (j < C).  These are
// C of the 2^(extended_k - k) cosets that make up upstream's extended domain — enough points to
// determine h (degree < C n), so the other cosets are never computed (5 instead of 8 for the
// degree-6 circuits of the reference).  A rotation moves inside a coset: blocks of 2^log_size rows
// rotate independently, which is also the plain rotation of a Lagrange column (one block).

// ---- Fr::random(rng) = from_u512(8 x next_u64): lo * R^2 + hi * R^3 (Montgomery products) ----
ZK_D fe_t from_u512_row(const uint32_t* wide16) {
    fe_t lo, hi, r2, r3;
    for (int i = 0; i < 8; ++i) { lo.l[i] = wide16[i]; hi.l[i] = wide16[8 + i]; r2.l[i] = FrCfg::r2(i); r3.l[i] = FrCfg::r3(i); }
    // lo / hi are arbitrary 256-bit integers (not reduced).  They must be the SECOND operand: the
    // CIOS rounds keep the accumulator below 2p as long as the first operand is < p, whatever the
    // 32-bit digits of the second are; an unreduced first operand can overflow the 9-limb window.
    return Fr::add(Fr::mul(r2, lo), Fr::mul(r3, hi));
}

// ---- permutation grand product (Lagrange domain) ----
struct PermLagArgs {
    uint32_t ncols, n;
    const fe_t* values[ZK_MAXC];
    const fe_t* sigma[ZK_MAXC];
    fe_t coef[ZK_MAXC];                 // delta^(global column index) * beta
    fe_t beta, gamma;
    const fe_t* omega_pows;             // omega^i
    fe_t* out;
};
ZK_D void perm_denominator_row(const PermLagArgs& a, uint32_t i) {
    fe_t acc = Fr::one();
    for (uint32_t j = 0; j < a.ncols; ++j) {
        fe_t s = a.sigma[j][i], v = a.values[j][i];
        acc = Fr::mul(acc, Fr::add(Fr::add(Fr::mul(a.beta, s), a.gamma), v));
    }
    a.out[i] = acc;
}
ZK_D void perm_numerator_row(const PermLagArgs& a, uint32_t i) {
    fe_t acc = a.out[i], w = a.omega_pows[i];
    for (uint32_t j = 0; j < a.ncols; ++j) {
        fe_t v = a.values[j][i];
        acc = Fr::mul(acc, Fr::add(Fr::add(Fr::mul(w, a.coef[j]), a.gamma), v));
    }
    a.out[i] = acc;
}

// ---- lookup grand product (Lagrange domain) ----
struct LookupProdArgs {
    const fe_t *pin, *ptab, *cin, *ctab;
    fe_t beta, gamma;
    fe_t* out;
    uint32_t n;
};
ZK_D void lookup_den_row(const LookupProdArgs& a, uint32_t i) {
    fe_t x = a.pin[i], y = a.ptab[i];
    a.out[i] = Fr::mul(Fr::add(a.beta, x), Fr::add(a.gamma, y));
}
ZK_D void lookup_num_row(const LookupProdArgs& a, uint32_t i) {
    fe_t d = a.out[i], x = a.cin[i], y = a.ctab[i];
    a.out[i] = Fr::mul(Fr::mul(d, Fr::add(x, a.beta)), Fr::add(y, a.gamma));
}

// ---- evaluate_h: permutation part (extended domain) ----
struct QuotPermAArgs {
    fe_t* h;
    fe_t y;
    const fe_t *l0, *l_last;
    uint32_t rows;                      // rows evaluated: [row0, row0 + rows) of the C * n (a rank of a sharded proof owns whole cosets)
    uint32_t row0;
    uint32_t nsets, log_ext, rot_scale; // log_ext = log2 of the rotation block (k)
    int32_t last_rot;                   // -(blinding_factors + 1)
    const fe_t* z[ZK_MAXC];             // permutation_product_coset per set
};
ZK_D uint32_t rot_idx(uint32_t idx, int32_t rot, uint32_t rot_scale, uint32_t log_size) {
    const uint32_t mask = (1u << log_size) - 1;
    return (idx & ~mask) | ((idx + (uint32_t)(rot * (int32_t)rot_scale)) & mask);
}
ZK_D void quot_perm_a_row(const QuotPermAArgs& a, uint32_t idx) {
    fe_t h = a.h[idx], l0 = a.l0[idx], ll = a.l_last[idx];
    fe_t zf = a.z[0][idx], zl = a.z[a.nsets - 1][idx];
    // l_0 (1 - z_0)
    h = Fr::add(Fr::mul(h, a.y), Fr::mul(Fr::sub(Fr::one(), zf), l0));
    // l_last (z_l^2 - z_l)
    h = Fr::add(Fr::mul(h, a.y), Fr::mul(Fr::sub(Fr::sqr(zl), zl), ll));
    // l_0 (z_i - z_{i-1}(omega^last X))
    uint32_t r_last = rot_idx(idx, a.last_rot, a.rot_scale, a.log_ext);
    for (uint32_t s = 1; s < a.nsets; ++s) {
        fe_t zi = a.z[s][idx], zp = a.z[s - 1][r_last];
        h = Fr::add(Fr::mul(h, a.y), Fr::mul(Fr::sub(zi, zp), l0));
    }
    a.h[idx] = h;
}

struct QuotPermBArgs {
    fe_t* h;
    fe_t y, beta, gamma;
    const fe_t* l_active;
    const fe_t* z;
    uint32_t rows, row0, ncols, log_ext, rot_scale;
    const fe_t* values[ZK_MAXC];        // column cosets
    const fe_t* sigma[ZK_MAXC];         // permutation cosets
    fe_t cdelta[ZK_MAXC];               // beta * zeta * delta^(global column index)
    const fe_t* omega_pows;             // omega^i, i < n
    const fe_t* coset_fac;              // extended_omega^j, j < C (device)
};
ZK_D void quot_perm_b_row(const QuotPermBArgs& a, uint32_t idx) {
    fe_t wl = a.omega_pows[idx & ((1u << a.log_ext) - 1)], wh = a.coset_fac[idx >> a.log_ext];
    fe_t beta_term = Fr::mul(wl, wh);                                       // extended_omega^j * omega^i = X / zeta
    fe_t left = a.z[rot_idx(idx, 1, a.rot_scale, a.log_ext)], right = a.z[idx];
    for (uint32_t j = 0; j < a.ncols; ++j) {
        fe_t v = a.values[j][idx], s = a.sigma[j][idx];
        left = Fr::mul(left, Fr::add(Fr::add(v, Fr::mul(a.beta, s)), a.gamma));
        right = Fr::mul(right, Fr::add(Fr::add(v, Fr::mul(a.cdelta[j], beta_term)), a.gamma));
    }
    fe_t h = a.h[idx], la = a.l_active[idx];
    a.h[idx] = Fr::add(Fr::mul(h, a.y), Fr::mul(Fr::sub(left, right), la));
}

// ---- evaluate_h: one lookup argument (extended domain) ----
struct QuotLookupArgs {
    fe_t* h;
    fe_t y, beta, gamma;
    const fe_t *l0, *l_last, *l_active;
    const fe_t *z, *a, *s;              // product / permuted input / permuted table cosets
    const fe_t* table_value;            // (compressed input + beta)(compressed table + gamma)
    uint32_t log_ext, rot_scale, rows, row0;
    fe_t ypow[4];                       // y^2, y^3, y^4, y^5
};
// The five terms upstream folds one by one (h <- h*y + term):
//   l_0 (1 - z);  l_last (z^2 - z);  l_active (z(wX)(a' + beta)(s' + gamma) - z * table_value);
//   l_0 (a' - s');  l_active (a' - s')(a' - a'(w^-1 X))
// are accumulated grouped by their Lagrange factor — the same polynomial value with 13 instead of
// 15 multiplications per row:
//   h y^5 + l_0 [(1 - z) y^4 + (a' - s') y] + l_last (z^2 - z) y^3 + l_active [(lhs - z tv) y^2 + (a' - s')(a' - a'_prev)]
ZK_D void quot_lookup_row(const QuotLookupArgs& q, uint32_t idx) {
    fe_t h = q.h[idx], l0 = q.l0[idx], ll = q.l_last[idx], la = q.l_active[idx];
    fe_t z = q.z[idx], zn = q.z[rot_idx(idx, 1, q.rot_scale, q.log_ext)];
    fe_t a = q.a[idx], ap = q.a[rot_idx(idx, -1, q.rot_scale, q.log_ext)], s = q.s[idx], tv = q.table_value[idx];
    fe_t a_minus_s = Fr::sub(a, s);
    fe_t t0 = Fr::add(Fr::mul(Fr::sub(Fr::one(), z), q.ypow[2]), Fr::mul(a_minus_s, q.y));
    fe_t t1 = Fr::mul(Fr::sub(Fr::sqr(z), z), q.ypow[1]);
    fe_t lhs = Fr::mul(Fr::mul(zn, Fr::add(a, q.beta)), Fr::add(s, q.gamma));
    fe_t t2 = Fr::add(Fr::mul(Fr::sub(lhs, Fr::mul(z, tv)), q.ypow[0]), Fr::mul(a_minus_s, Fr::sub(a, ap)));
    h = Fr::mul(h, q.ypow[3]);
    h = Fr::add(h, Fr::mul(l0, t0));
    h = Fr::add(h, Fr::mul(ll, t1));
    h = Fr::add(h, Fr::mul(la, t2));
    q.h[idx] = h;
}

// ---- vanishing::construct without the extended iNTT ----
// g[j*n + r] are the coefficients (in Y = X / c_j) of h restricted to coset j, i.e. after the
// per-coset iNTT.  With h(X) = sum_r X^r H_r(X^n), deg H_r < C:  H_r(c_j^n) = g[j][r] * c_j^(-r), and
// the C coefficients of H_r — the r-th coefficient of every h piece — follow from the fixed C x C
// inverse Vandermonde matrix of the points c_j^n:   out[t*n + r] = sum_j vinv[t*C + j] * H_r(c_j^n).
// `extra` (optional): a second summand already in H-space, extra[j*n + r] = H'_r(c_j^n) — the lookup part of the
// quotient when it was evaluated on fewer cosets (lookup_extrapolate_row).
// `lin` (optional): a part of h of degree < n, lin[r] = its r-th coefficient in Y = X / c_0 (the per-coset iNTT of coset 0);
// it adds lin[r] * c_0^(-r) to piece 0.
ZK_D void coset_interpolate_row(const fe_t* g, const fe_t* inv_pow, const fe_t* vinv, uint32_t C, size_t n, fe_t* out, size_t r,
                                const fe_t* extra = nullptr, const fe_t* lin = nullptr) {
    fe_t v[ZK_MAXCOSETS];
    for (uint32_t j = 0; j < C; ++j) {
        fe_t x = g[(size_t)j * n + r], w = inv_pow[(size_t)j * n + r];
        v[j] = Fr::mul(x, w);
        if (extra) { fe_t e = extra[(size_t)j * n + r]; v[j] = Fr::add(v[j], e); }
    }
    for (uint32_t t = 0; t < C; ++t) {
        fe_t acc = Fr::mul(v[0], vinv[t * C]);
        for (uint32_t j = 1; j < C; ++j) acc = Fr::add(acc, Fr::mul(v[j], vinv[t * C + j]));
        if (t == 0 && lin) acc = Fr::add(acc, Fr::mul(lin[r], inv_pow[r]));
        out[(size_t)t * n + r] = acc;
    }
}

// ---- lookup terms and low-degree gates on fewer cosets ----
// The lookup terms of evaluate_h have degree < CL * n with CL = 2 + deg(input) + deg(table) (4 for a plain column
// lookup) while the gates of the highest degree need all C = d - 1 cosets; gates of degree <= CL + 1 join them
// (quot_plan.hpp).  Their sum h_L is therefore evaluated on the first CL cosets only — the three coset extensions per
// lookup and the two lookup kernels shrink by CL / C — and carried to the other cosets in H-space: with
// h_L(X) = sum_r X^r H_r(X^n), deg H_r < CL, the per-coset iNTT gives g[j][r] = c_j^r H_r(y_j) (y_j = c_j^n) for j < CL,
// and H_r(y_j') for j' >= CL is the Lagrange extrapolation sum_j lambda[j' - CL][j] H_r(y_j).  Output (in place, C * n
// elements): H_r(y_j) * tinv[j] for every coset j (tinv null: 1), the summand coset_interpolate_row adds to the gate /
// permutation part.  The prover divides by the vanishing polynomial in the iNTT already (tinv null): the numerator of a
// gate of degree CL + 1 has degree CL * n + n - CL - 1, more than CL cosets determine, its quotient has degree < CL * n.
ZK_D void lookup_extrapolate_row(fe_t* g, const fe_t* inv_pow, const fe_t* lambda, const fe_t* tinv, uint32_t CL, uint32_t C, size_t n, size_t r) {
    fe_t u[ZK_MAXCOSETS];
    for (uint32_t j = 0; j < CL; ++j) { fe_t x = g[(size_t)j * n + r], w = inv_pow[(size_t)j * n + r]; u[j] = Fr::mul(x, w); }
    for (uint32_t jp = CL; jp < C; ++jp) {
        fe_t acc = Fr::mul(u[0], lambda[(jp - CL) * CL]);
        for (uint32_t j = 1; j < CL; ++j) acc = Fr::add(acc, Fr::mul(u[j], lambda[(jp - CL) * CL + j]));
        g[(size_t)jp * n + r] = tinv ? Fr::mul(acc, tinv[jp]) : acc;
    }
    for (uint32_t j = 0; j < CL; ++j) g[(size_t)j * n + r] = tinv ? Fr::mul(u[j], tinv[j]) : u[j];
}

// ---- vanishing::evaluate: h_poly = sum_j (x^n)^j piece_j  (pieces contiguous, n apart) ----
ZK_D void fold_pieces_row(const fe_t* pieces, uint32_t npieces, size_t n, const fe_t& xn, fe_t* out, size_t i) {
    fe_t acc = pieces[(size_t)(npieces - 1) * n + i];
    for (uint32_t j = npieces - 1; j-- > 0;) { fe_t p = pieces[(size_t)j * n + i]; acc = Fr::add(Fr::mul(acc, xn), p); }
    out[i] = acc;
}

// ---- polynomial linear algebra ----
ZK_D void axpy_row(fe_t* acc, const fe_t* p, const fe_t& s, size_t i, bool init) {
    fe_t v = p[i];
    fe_t t = Fr::mul(v, s);
    if (!init) { fe_t a = acc[i]; t = Fr::add(a, t); }
    acc[i] = t;
}
ZK_D void scale_row(fe_t* a, const fe_t& s, size_t i) { fe_t v = a[i]; a[i] = Fr::mul(v, s); }
// out = 1 - (a + b)   (l_active_row)
ZK_D void one_minus_sum_row(const fe_t* a, const fe_t* b, fe_t* out, size_t i) {
    fe_t x = a[i], y = b[i];
    out[i] = Fr::sub(Fr::one(), Fr::add(x, y));
}
// sigma[i] = delta^col * omega^row of the mapped cell (permutation keygen)
ZK_D void sigma_row(const uint32_t* map_col, const uint32_t* map_row, const fe_t* delta_pows, const fe_t* omega_pows, fe_t* out, size_t i) {
    fe_t d = delta_pows[map_col[i]], w = omega_pows[map_row[i]];
    out[i] = Fr::mul(d, w);
}

}  // namespace b200zk
