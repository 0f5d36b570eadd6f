// bn256 pairing products on the device: the pairing of csrc/pairing.hpp, f_{t-1,Q}(P)^((q^12-1)/r) with t - 1 = 6 x^2,
// over the same tower (Fq2 = Fq[u]/(u^2 + 1), Fq12 = Fq2[w]/(w^6 - xi), xi = 9 + u, six Fq2 coefficients of w^i).
// Every value is fully reduced, so each result is byte for byte the host's final_exponentiation(prod miller_loop).
//
// Miller loop: the host's loop over the bits of t - 1 (126 doublings, 69 additions), with the G2 point T kept in
// homogeneous projective coordinates (X : Y : Z) on the twist.  Each line is the host's affine line times a factor
// in Fq2 (-2YZ for a tangent, X - xQ Z for a chord), which the final exponentiation removes:
//   line(P) = c0 * yP + c1 * xP * w + c2 * w^3.
// The steps depend on Q only, so g2_prepare writes the 195 coefficient triples of one Q once (upstream's G2Prepared);
// a product then costs one Fq12 squaring per bit and one sparse product per line and pair.
// Final exponentiation: the easy part (q^6 - 1)(q^2 + 1) with one inversion and a q^2-Frobenius; the hard part
// (q^4 - q^2 + 1)/r = l0 + l1 q + l2 q^2 + q^3 (Scott et al., "On the final exponentiation for calculating pairings
// on ordinary elliptic curves", 2009) through three exponentiations by x with cyclotomic squarings (Granger-Scott)
// and Frobenius maps.  The exponent is exactly the host's, not a multiple of it.
// Per-thread bodies only; the launches are in pairing.cu, and the same bodies run on a host compiler under
// ptx_chain.cuh emulation (tests/pairing_harness.cpp).
#pragma once
#include "curve.cuh"

// The tower's products are calls on the device: inlined, one final exponentiation would be millions of instructions.
#if defined(__CUDACC__)
#define PC_CALL static __device__ __noinline__
#else
#define PC_CALL static inline
#endif

namespace b200zk {

struct fq2_t { fe_t a, b; };                 // a + b u
struct fq12_t { fq2_t c[6]; };               // sum c_i w^i
struct pc_line_t { fq2_t c0, c1, c2; };      // c0 yP + c1 xP w + c2 w^3

static constexpr uint32_t PC_T_BITS = 126;   // bits of t - 1 below the top one
static constexpr uint32_t PC_LINES = 195;    // 126 doubling lines + 69 addition lines
static constexpr unsigned long long PC_X = 4965661367192848881ULL;

ZK_D bool pc_t_bit(int i) {                  // bit i of t - 1 = 6 x^2
    return (((i < 64 ? 0xf83e9682e87cfd46ULL : 0x6f4d8248eeb859fbULL) >> (i & 63)) & 1) != 0;
}

// ---- Fq2 ----
ZK_D fq2_t fq2_zero() { fq2_t r; r.a = Fq::zero(); r.b = Fq::zero(); return r; }
ZK_D fq2_t fq2_one() { fq2_t r; r.a = Fq::one(); r.b = Fq::zero(); return r; }
ZK_D fq2_t fq2_add(const fq2_t& x, const fq2_t& y) { fq2_t r; r.a = Fq::add(x.a, y.a); r.b = Fq::add(x.b, y.b); return r; }
ZK_D fq2_t fq2_sub(const fq2_t& x, const fq2_t& y) { fq2_t r; r.a = Fq::sub(x.a, y.a); r.b = Fq::sub(x.b, y.b); return r; }
ZK_D fq2_t fq2_neg(const fq2_t& x) { fq2_t r; r.a = Fq::neg(x.a); r.b = Fq::neg(x.b); return r; }
ZK_D fq2_t fq2_dbl(const fq2_t& x) { return fq2_add(x, x); }
ZK_D fq2_t fq2_conj(const fq2_t& x) { fq2_t r; r.a = x.a; r.b = Fq::neg(x.b); return r; }
PC_CALL fq2_t fq2_mul(const fq2_t& x, const fq2_t& y) {
    fe_t t0 = Fq::mul(x.a, y.a), t1 = Fq::mul(x.b, y.b);
    fq2_t r;
    r.a = Fq::sub(t0, t1);
    r.b = Fq::sub(Fq::sub(Fq::mul(Fq::add(x.a, x.b), Fq::add(y.a, y.b)), t0), t1);
    return r;
}
PC_CALL fq2_t fq2_sqr(const fq2_t& x) {
    fq2_t r;
    r.a = Fq::mul(Fq::add(x.a, x.b), Fq::sub(x.a, x.b));
    r.b = Fq::dbl(Fq::mul(x.a, x.b));
    return r;
}
ZK_D fq2_t fq2_scale(const fq2_t& x, const fe_t& s) { fq2_t r; r.a = Fq::mul(x.a, s); r.b = Fq::mul(x.b, s); return r; }
ZK_D fq2_t fq2_mul_xi(const fq2_t& x) {      // (a + b u)(9 + u) = (9a - b) + (9b + a) u
    fe_t a8 = Fq::dbl(Fq::dbl(Fq::dbl(x.a))), b8 = Fq::dbl(Fq::dbl(Fq::dbl(x.b)));
    fq2_t r;
    r.a = Fq::sub(Fq::add(a8, x.a), x.b);
    r.b = Fq::add(Fq::add(b8, x.b), x.a);
    return r;
}
PC_CALL fq2_t fq2_inv(const fq2_t& x) {         // inv(0) = 0
    fe_t d = Fq::inv_gcd(Fq::add(Fq::sqr(x.a), Fq::sqr(x.b)));
    fq2_t r;
    r.a = Fq::mul(x.a, d);
    r.b = Fq::neg(Fq::mul(x.b, d));
    return r;
}

// ---- Fq6 = Fq2[v]/(v^3 - xi), v = w^2: the even (g = c0, c2, c4) and odd (h = c1, c3, c5) halves of an Fq12 ----
struct fq6_t { fq2_t c[3]; };
ZK_D fq6_t fq6_add(const fq6_t& x, const fq6_t& y) { fq6_t r; for (int i = 0; i < 3; ++i) r.c[i] = fq2_add(x.c[i], y.c[i]); return r; }
ZK_D fq6_t fq6_sub(const fq6_t& x, const fq6_t& y) { fq6_t r; for (int i = 0; i < 3; ++i) r.c[i] = fq2_sub(x.c[i], y.c[i]); return r; }
ZK_D fq6_t fq6_mul_v(const fq6_t& x) { fq6_t r; r.c[0] = fq2_mul_xi(x.c[2]); r.c[1] = x.c[0]; r.c[2] = x.c[1]; return r; }
PC_CALL fq6_t fq6_mul(const fq6_t& x, const fq6_t& y) {          // Karatsuba: 6 Fq2 products
    fq2_t t0 = fq2_mul(x.c[0], y.c[0]), t1 = fq2_mul(x.c[1], y.c[1]), t2 = fq2_mul(x.c[2], y.c[2]);
    fq6_t r;
    r.c[0] = fq2_add(t0, fq2_mul_xi(fq2_sub(fq2_sub(fq2_mul(fq2_add(x.c[1], x.c[2]), fq2_add(y.c[1], y.c[2])), t1), t2)));
    r.c[1] = fq2_add(fq2_sub(fq2_sub(fq2_mul(fq2_add(x.c[0], x.c[1]), fq2_add(y.c[0], y.c[1])), t0), t1), fq2_mul_xi(t2));
    r.c[2] = fq2_add(fq2_sub(fq2_sub(fq2_mul(fq2_add(x.c[0], x.c[2]), fq2_add(y.c[0], y.c[2])), t0), t2), t1);
    return r;
}
PC_CALL fq6_t fq6_mul_by_01(const fq6_t& x, const fq2_t& b0, const fq2_t& b1) {     // x (b0 + b1 v): 5 Fq2 products
    fq2_t t0 = fq2_mul(x.c[0], b0), t1 = fq2_mul(x.c[1], b1);
    fq6_t r;
    r.c[0] = fq2_add(t0, fq2_mul_xi(fq2_sub(fq2_mul(fq2_add(x.c[1], x.c[2]), b1), t1)));
    r.c[1] = fq2_sub(fq2_sub(fq2_mul(fq2_add(x.c[0], x.c[1]), fq2_add(b0, b1)), t0), t1);
    r.c[2] = fq2_add(fq2_sub(fq2_mul(fq2_add(x.c[0], x.c[2]), b0), t0), t1);
    return r;
}
PC_CALL fq6_t fq6_inv(const fq6_t& x) {
    fq2_t t0 = fq2_sub(fq2_sqr(x.c[0]), fq2_mul_xi(fq2_mul(x.c[1], x.c[2])));
    fq2_t t1 = fq2_sub(fq2_mul_xi(fq2_sqr(x.c[2])), fq2_mul(x.c[0], x.c[1]));
    fq2_t t2 = fq2_sub(fq2_sqr(x.c[1]), fq2_mul(x.c[0], x.c[2]));
    fq2_t d = fq2_inv(fq2_add(fq2_mul(x.c[0], t0), fq2_mul_xi(fq2_add(fq2_mul(x.c[2], t1), fq2_mul(x.c[1], t2)))));
    fq6_t r;
    r.c[0] = fq2_mul(t0, d); r.c[1] = fq2_mul(t1, d); r.c[2] = fq2_mul(t2, d);
    return r;
}
ZK_D fq6_t fq12_even(const fq12_t& f) { fq6_t r; r.c[0] = f.c[0]; r.c[1] = f.c[2]; r.c[2] = f.c[4]; return r; }
ZK_D fq6_t fq12_odd(const fq12_t& f) { fq6_t r; r.c[0] = f.c[1]; r.c[1] = f.c[3]; r.c[2] = f.c[5]; return r; }
ZK_D fq12_t fq12_join(const fq6_t& g, const fq6_t& h) {
    fq12_t r;
    for (int i = 0; i < 3; ++i) { r.c[2 * i] = g.c[i]; r.c[2 * i + 1] = h.c[i]; }
    return r;
}

// ---- Fq12 = Fq6[w]/(w^2 - v) ----
ZK_D fq12_t fq12_one() { fq12_t r; r.c[0] = fq2_one(); for (int i = 1; i < 6; ++i) r.c[i] = fq2_zero(); return r; }
ZK_D bool fq12_is_one(const fq12_t& f) {
    bool one = Fq::eq(f.c[0].a, Fq::one()) && Fq::is_zero(f.c[0].b);
    for (int i = 1; i < 6; ++i) one = one && Fq::is_zero(f.c[i].a) && Fq::is_zero(f.c[i].b);
    return one;
}
PC_CALL fq12_t fq12_mul(const fq12_t& x, const fq12_t& y) {      // 3 Fq6 products (18 Fq2)
    fq6_t g0 = fq12_even(x), h0 = fq12_odd(x), g1 = fq12_even(y), h1 = fq12_odd(y);
    fq6_t t0 = fq6_mul(g0, g1), t1 = fq6_mul(h0, h1);
    fq6_t s = fq6_mul(fq6_add(g0, h0), fq6_add(g1, h1));
    return fq12_join(fq6_add(t0, fq6_mul_v(t1)), fq6_sub(fq6_sub(s, t0), t1));
}
PC_CALL fq12_t fq12_sqr(const fq12_t& x) {                        // complex squaring: 2 Fq6 products
    fq6_t g = fq12_even(x), h = fq12_odd(x);
    fq6_t t = fq6_mul(g, h);
    fq6_t s = fq6_mul(fq6_add(g, h), fq6_add(g, fq6_mul_v(h)));
    return fq12_join(fq6_sub(fq6_sub(s, t), fq6_mul_v(t)), fq6_add(t, t));
}
ZK_D fq12_t fq12_conj(const fq12_t& x) {                       // x^(q^6): w -> -w
    fq12_t r = x;
    for (int i = 1; i < 6; i += 2) r.c[i] = fq2_neg(x.c[i]);
    return r;
}
PC_CALL fq12_t fq12_inv(const fq12_t& x) {                        // (g + h w)^-1 = (g - h w) / (g^2 - v h^2)
    fq6_t g = fq12_even(x), h = fq12_odd(x);
    fq6_t d = fq6_inv(fq6_sub(fq6_mul(g, g), fq6_mul_v(fq6_mul(h, h))));
    fq6_t rh = fq6_mul(h, d);
    for (int i = 0; i < 3; ++i) rh.c[i] = fq2_neg(rh.c[i]);
    return fq12_join(fq6_mul(g, d), rh);
}
// f * line(P): the line is c0 yP + (c1 xP) w + c2 w^3, i.e. a + b w with a = (c0 yP, 0, 0), b = (c1 xP, c2, 0) in Fq6
PC_CALL fq12_t fq12_mul_by_line(const fq12_t& f, const pc_line_t& l, const affine_t& p) {
    fq2_t a = fq2_scale(l.c0, p.y), b0 = fq2_scale(l.c1, p.x);
    fq6_t g = fq12_even(f), h = fq12_odd(f);
    fq6_t ga;
    for (int i = 0; i < 3; ++i) ga.c[i] = fq2_mul(g.c[i], a);
    fq6_t hb = fq6_mul_by_01(h, b0, l.c2);
    fq6_t s = fq6_mul_by_01(fq6_add(g, h), fq2_add(a, b0), l.c2);
    return fq12_join(fq6_add(ga, fq6_mul_v(hb)), fq6_sub(fq6_sub(s, ga), hb));
}

// ---- Frobenius maps: f^(q^k) = sum frob_k(c_i) gamma_{k,i} w^i (constants from tools/gen_pairing_frobenius.py) ----
ZK_D constexpr uint64_t pc_frob_limb(int row, int j) {
    constexpr uint64_t t[30 * 4] = {
#include "pairing_frobenius.inc"
    };
    return t[row * 4 + j];
}
ZK_D fe_t pc_frob_const(int row) {
    fe_t r;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        r.l[2 * j] = (uint32_t)pc_frob_limb(row, j);
        r.l[2 * j + 1] = (uint32_t)(pc_frob_limb(row, j) >> 32);
    }
    return r;
}
PC_CALL fq12_t fq12_frob(const fq12_t& x, int k) {                // k = 1, 2 or 3
    fq12_t r;
    r.c[0] = k == 2 ? x.c[0] : fq2_conj(x.c[0]);
#pragma unroll
    for (int i = 1; i < 6; ++i) {
        if (k == 2) { r.c[i] = fq2_scale(x.c[i], pc_frob_const(12 + i)); continue; }
        const int row = (k == 1 ? 0 : 18) + 2 * i;
        fq2_t g;
        g.a = pc_frob_const(row);
        g.b = pc_frob_const(row + 1);
        r.c[i] = fq2_mul(fq2_conj(x.c[i]), g);
    }
    return r;
}

// ---- the cyclotomic subgroup (f^(q^6 + 1) = 1, every value after the easy part) ----
// Granger-Scott squaring over Fq12 = Fq4^3, Fq4 = Fq2[s]/(s^2 - xi), s = w^3: the pairs (c0, c3), (c1, c4), (c2, c5)
PC_CALL fq12_t fq12_cyc_sqr(const fq12_t& x) {
    const fq2_t* c = x.c;
    fq2_t t0 = fq2_sqr(c[3]), t1 = fq2_sqr(c[0]);
    fq2_t t6 = fq2_sub(fq2_sub(fq2_sqr(fq2_add(c[3], c[0])), t0), t1);              // 2 c0 c3
    fq2_t t2 = fq2_sqr(c[4]), t3 = fq2_sqr(c[1]);
    fq2_t t7 = fq2_sub(fq2_sub(fq2_sqr(fq2_add(c[4], c[1])), t2), t3);              // 2 c1 c4
    fq2_t t4 = fq2_sqr(c[5]), t5 = fq2_sqr(c[2]);
    fq2_t t8 = fq2_mul_xi(fq2_sub(fq2_sub(fq2_sqr(fq2_add(c[5], c[2])), t4), t5));  // 2 xi c2 c5
    t0 = fq2_add(fq2_mul_xi(t0), t1);                                               // (c0 + c3 s)^2, s-free part
    t2 = fq2_add(fq2_mul_xi(t2), t3);
    t4 = fq2_add(fq2_mul_xi(t4), t5);
    fq12_t r;
    r.c[0] = fq2_add(fq2_dbl(fq2_sub(t0, c[0])), t0);                              // 3 t - 2 c
    r.c[2] = fq2_add(fq2_dbl(fq2_sub(t2, c[2])), t2);
    r.c[4] = fq2_add(fq2_dbl(fq2_sub(t4, c[4])), t4);
    r.c[1] = fq2_add(fq2_dbl(fq2_add(t8, c[1])), t8);                              // 3 t + 2 c
    r.c[3] = fq2_add(fq2_dbl(fq2_add(t6, c[3])), t6);
    r.c[5] = fq2_add(fq2_dbl(fq2_add(t7, c[5])), t7);
    return r;
}
PC_CALL fq12_t fq12_cyc_exp_x(const fq12_t& f) {                  // f^x, x = 4965661367192848881 (63 bits, 28 set)
    fq12_t acc = f;
    for (int i = 61; i >= 0; --i) {
        acc = fq12_cyc_sqr(acc);
        if ((PC_X >> i) & 1) acc = fq12_mul(acc, f);
    }
    return acc;
}

// f^((q^12 - 1)/r)
PC_CALL fq12_t fq12_easy_part(const fq12_t& f) {                  // f^((q^6 - 1)(q^2 + 1))
    fq12_t t = fq12_mul(fq12_conj(f), fq12_inv(f));
    return fq12_mul(fq12_frob(t, 2), t);
}
PC_CALL fq12_t fq12_hard_part(const fq12_t& t1) {                 // t1^(l0 + l1 q + l2 q^2 + q^3), t1 cyclotomic
    fq12_t fu = fq12_cyc_exp_x(t1), fu2 = fq12_cyc_exp_x(fu), fu3 = fq12_cyc_exp_x(fu2);
    fq12_t fp2 = fq12_frob(t1, 2);
    fq12_t y0 = fq12_mul(fq12_mul(fq12_frob(t1, 1), fp2), fq12_frob(fp2, 1));        // t1^(q + q^2 + q^3)
    fq12_t y1 = fq12_conj(t1);                                                        // t1^-1
    fq12_t y2 = fq12_frob(fu2, 2);                                                    // t1^(x^2 q^2)
    fq12_t y3 = fq12_conj(fq12_frob(fu, 1));                                          // t1^(-x q)
    fq12_t y4 = fq12_conj(fq12_mul(fu, fq12_frob(fu2, 1)));                           // t1^(-x - x^2 q)
    fq12_t y5 = fq12_conj(fu2);                                                       // t1^(-x^2)
    fq12_t y6 = fq12_conj(fq12_mul(fu3, fq12_frob(fu3, 1)));                          // t1^(-x^3 - x^3 q)
    // y0 y1^2 y2^6 y3^12 y4^18 y5^30 y6^36 (a vector addition chain)
    fq12_t t0 = fq12_mul(fq12_mul(fq12_cyc_sqr(y6), y4), y5);
    fq12_t t = fq12_mul(fq12_mul(y3, y5), t0);
    t0 = fq12_mul(t0, y2);
    t = fq12_cyc_sqr(fq12_mul(fq12_cyc_sqr(t), t0));
    t0 = fq12_mul(t, y1);
    t = fq12_mul(t, y0);
    return fq12_mul(fq12_cyc_sqr(t0), t);
}
ZK_D fq12_t fq12_final_exp(const fq12_t& f) { return fq12_hard_part(fq12_easy_part(f)); }

// ---- G2Prepared: the 195 lines of the Miller loop of Q (affine, on the twist, not the identity) ----
struct pc_g2_proj_t { fq2_t x, y, z; };
// tangent at T, T <- 2T;  line = -2YZ times the host's tangent
PC_CALL pc_line_t pc_dbl_step(pc_g2_proj_t& t, const fe_t& two_inv, const fq2_t& b_twist) {
    fq2_t a = fq2_scale(fq2_mul(t.x, t.y), two_inv);
    fq2_t b = fq2_sqr(t.y), c = fq2_sqr(t.z);
    fq2_t e = fq2_mul(b_twist, fq2_add(fq2_dbl(c), c));                             // 3 b' Z^2
    fq2_t f = fq2_add(fq2_dbl(e), e);
    fq2_t g = fq2_scale(fq2_add(b, f), two_inv);
    fq2_t h = fq2_sub(fq2_sqr(fq2_add(t.y, t.z)), fq2_add(b, c));                  // 2YZ
    fq2_t j = fq2_sqr(t.x);
    fq2_t e2 = fq2_sqr(e);
    t.x = fq2_mul(a, fq2_sub(b, f));
    t.y = fq2_sub(fq2_sqr(g), fq2_add(fq2_dbl(e2), e2));
    t.z = fq2_mul(b, h);
    pc_line_t l;
    l.c0 = fq2_neg(h);
    l.c1 = fq2_add(fq2_dbl(j), j);
    l.c2 = fq2_sub(e, b);
    return l;
}
// chord through T and Q, T <- T + Q;  line = (X - xQ Z) times the host's chord
PC_CALL pc_line_t pc_add_step(pc_g2_proj_t& t, const fq2_t& qx, const fq2_t& qy) {
    fq2_t theta = fq2_sub(t.y, fq2_mul(qy, t.z));
    fq2_t lambda = fq2_sub(t.x, fq2_mul(qx, t.z));
    fq2_t c = fq2_sqr(theta), d = fq2_sqr(lambda);
    fq2_t e = fq2_mul(lambda, d), f = fq2_mul(t.z, c), g = fq2_mul(t.x, d);
    fq2_t h = fq2_sub(fq2_add(e, f), fq2_dbl(g));
    t.x = fq2_mul(lambda, h);
    t.y = fq2_sub(fq2_mul(theta, fq2_sub(g, h)), fq2_mul(e, t.y));
    t.z = fq2_mul(t.z, e);
    pc_line_t l;
    l.c0 = lambda;
    l.c1 = fq2_neg(theta);
    l.c2 = fq2_sub(fq2_mul(theta, qx), fq2_mul(lambda, qy));
    return l;
}
// lines[0 .. PC_LINES) in loop order: for i = 125 .. 0, the doubling line, then the addition line when bit i is set
ZK_D void g2_prepare(const fq2_t& qx, const fq2_t& qy, pc_line_t* lines) {
    const fe_t two_inv = Fq::inv_gcd(Fq::dbl(Fq::one()));
    fq2_t xi; xi.a = Fq::add(Fq::dbl(Fq::dbl(Fq::dbl(Fq::one()))), Fq::one()); xi.b = Fq::one();
    const fq2_t b_twist = fq2_scale(fq2_inv(xi), Fq::add(Fq::dbl(Fq::one()), Fq::one()));     // 3 / xi
    pc_g2_proj_t t; t.x = qx; t.y = qy; t.z = fq2_one();
    uint32_t n = 0;
    for (int i = (int)PC_T_BITS - 1; i >= 0; --i) {
        lines[n++] = pc_dbl_step(t, two_inv, b_twist);
        if (pc_t_bit(i)) lines[n++] = pc_add_step(t, qx, qy);
    }
}

// prod_j f_{t-1,Q_j}(P_j) up to factors in Fq2 over the m pairs (p[j], Q_j), Q_j's lines at tables + q[j] * PC_LINES;
// q[j] == PC_SKIP leaves a pair out (an identity on either side contributes 1)
static constexpr uint32_t PC_SKIP = 0xffffffffu;
ZK_D fq12_t pc_miller_product(const affine_t* p, const uint32_t* q, const pc_line_t* tables, uint32_t m) {
    fq12_t f = fq12_one();
    uint32_t n = 0;
    for (int i = (int)PC_T_BITS - 1; i >= 0; --i) {
        f = fq12_sqr(f);
        for (uint32_t j = 0; j < m; ++j) if (q[j] != PC_SKIP) f = fq12_mul_by_line(f, tables[(size_t)q[j] * PC_LINES + n], p[j]);
        ++n;
        if (pc_t_bit(i)) {
            for (uint32_t j = 0; j < m; ++j) if (q[j] != PC_SKIP) f = fq12_mul_by_line(f, tables[(size_t)q[j] * PC_LINES + n], p[j]);
            ++n;
        }
    }
    return f;
}

}  // namespace b200zk
