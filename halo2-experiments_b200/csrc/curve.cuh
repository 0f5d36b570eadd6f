// bn256 G1 (y^2 = x^3 + 3 over Fq) on the device.
//
// Memory formats match halo2curves 0.3.1 (src/bn256/curve.rs, src/derive/curve.rs;
// G1Affine is named at /root/reference/src/circuits/utils.rs:2,43,45):
//   affine_t = G1Affine {x, y}   64 B, identity = (0, 0)
//   jac_t    = G1 {x, y, z}      96 B, identity z = 0
// Bucket accumulators use extended Jacobian (XYZZ) coordinates: x = X/ZZ,
// y = Y/ZZZ, ZZ^3 = ZZZ^2, identity ZZ = 0.  A mixed addition is 8M + 2S and a
// full addition 12M + 2S, all on the IMAD pipe.  Every operation is complete
// (handles identity, P + P and P + (-P)), because best_multiexp accepts arbitrary
// bases, including repeated ones.
#pragma once
#include "field.cuh"

namespace b200zk {

struct alignas(32) affine_t { fe_t x, y; };
struct alignas(32) jac_t { fe_t x, y, z; };
struct alignas(32) xyzz_t { fe_t x, y, zz, zzz; };

ZK_D bool affine_is_identity(const affine_t& p) { return Fq::is_zero(p.x) && Fq::is_zero(p.y); }

ZK_D xyzz_t xyzz_identity() {
    xyzz_t r; r.x = Fq::zero(); r.y = Fq::zero(); r.zz = Fq::zero(); r.zzz = Fq::zero(); return r;
}
ZK_D bool xyzz_is_identity(const xyzz_t& p) { return Fq::is_zero(p.zz); }

ZK_D xyzz_t xyzz_from_affine(const affine_t& p) {
    if (affine_is_identity(p)) return xyzz_identity();
    xyzz_t r; r.x = p.x; r.y = p.y; r.zz = Fq::one(); r.zzz = Fq::one(); return r;
}

// dbl-2008-s-1 (a = 0)
ZK_D xyzz_t xyzz_dbl(const xyzz_t& p) {
    if (xyzz_is_identity(p)) return p;
    fe_t u = Fq::dbl(p.y), v = Fq::sqr(u), w = Fq::mul(u, v), s = Fq::mul(p.x, v);
    fe_t xx = Fq::sqr(p.x), m = Fq::add(Fq::dbl(xx), xx);
    xyzz_t r;
    r.x = Fq::sub(Fq::sqr(m), Fq::dbl(s));
    r.y = Fq::sub(Fq::mul(m, Fq::sub(s, r.x)), Fq::mul(w, p.y));
    r.zz = Fq::mul(v, p.zz);
    r.zzz = Fq::mul(w, p.zzz);
    return r;
}

// acc += q (affine); `negate` adds -q.   madd-2008-s
ZK_D void xyzz_madd(xyzz_t& acc, const affine_t& q_in, bool negate) {
    if (affine_is_identity(q_in)) return;
    affine_t q = q_in;
    if (negate) q.y = Fq::neg(q.y);
    if (xyzz_is_identity(acc)) { acc = xyzz_from_affine(q); return; }
    fe_t u2 = Fq::mul(q.x, acc.zz), s2 = Fq::mul(q.y, acc.zzz);
    fe_t p = Fq::sub(u2, acc.x), r = Fq::sub(s2, acc.y);
    if (Fq::is_zero(p)) {
        if (Fq::is_zero(r)) acc = xyzz_dbl(xyzz_from_affine(q)); else acc = xyzz_identity();
        return;
    }
    fe_t pp = Fq::sqr(p), ppp = Fq::mul(p, pp), qq = Fq::mul(acc.x, pp);
    fe_t x3 = Fq::sub(Fq::sub(Fq::sqr(r), ppp), Fq::dbl(qq));
    fe_t y3 = Fq::sub(Fq::mul(r, Fq::sub(qq, x3)), Fq::mul(acc.y, ppp));
    acc.x = x3; acc.y = y3;
    acc.zz = Fq::mul(acc.zz, pp);
    acc.zzz = Fq::mul(acc.zzz, ppp);
}

// acc += q (XYZZ).   add-2008-s
ZK_D void xyzz_add(xyzz_t& acc, const xyzz_t& q) {
    if (xyzz_is_identity(q)) return;
    if (xyzz_is_identity(acc)) { acc = q; return; }
    fe_t u1 = Fq::mul(acc.x, q.zz), u2 = Fq::mul(q.x, acc.zz);
    fe_t s1 = Fq::mul(acc.y, q.zzz), s2 = Fq::mul(q.y, acc.zzz);
    fe_t p = Fq::sub(u2, u1), r = Fq::sub(s2, s1);
    if (Fq::is_zero(p)) {
        if (Fq::is_zero(r)) acc = xyzz_dbl(acc); else acc = xyzz_identity();
        return;
    }
    fe_t pp = Fq::sqr(p), ppp = Fq::mul(p, pp), qq = Fq::mul(u1, pp);
    fe_t x3 = Fq::sub(Fq::sub(Fq::sqr(r), ppp), Fq::dbl(qq));
    fe_t y3 = Fq::sub(Fq::mul(r, Fq::sub(qq, x3)), Fq::mul(s1, ppp));
    acc.x = x3; acc.y = y3;
    acc.zz = Fq::mul(Fq::mul(acc.zz, q.zz), pp);
    acc.zzz = Fq::mul(Fq::mul(acc.zzz, q.zzz), ppp);
}

// G1Affine::from_bytes (halo2curves 0.3.1 compressed form) of one point: x8 = the 32 bytes as 8 little-endian words,
// x canonical < q with the parity of y in bit 31 of word 7, identity = all zero.  y = sqrt(x^3 + 3) with the stored parity.
// Returns false (and the identity) for a non-canonical x, a sign bit on the identity or a point off the curve.
ZK_D bool g1_decompress(const uint32_t x8[8], affine_t* out) {
    fe_t x;
#pragma unroll
    for (int j = 0; j < 8; ++j) x.l[j] = x8[j];
    const uint32_t sign = x.l[7] >> 31;
    x.l[7] &= 0x7fffffffu;
    out->x = Fq::zero(); out->y = Fq::zero();
    bool ge = true;                                              // x >= q ?
    for (int j = 7; j >= 0; --j) { uint32_t pj = FqCfg::p(j); if (x.l[j] != pj) { ge = x.l[j] > pj; break; } }
    if (ge) return false;
    bool zero = true;
    for (int j = 0; j < 8; ++j) zero &= x.l[j] == 0;
    if (zero) return !sign;
    fe_t xm = Fq::to_mont(x);
    fe_t three = Fq::add(Fq::add(Fq::one(), Fq::one()), Fq::one());
    fe_t rhs = Fq::add(Fq::mul(Fq::sqr(xm), xm), three);
    // (q + 1) / 4
    const uint32_t e[8] = {0xb61f3f52u, 0x4f082305u, 0x5a1c72a3u, 0x65e05aa4u, 0xa0605617u, 0x6e14116du, 0xb84c680au, 0x0c19139cu};
    fe_t y = Fq::pow(rhs, e);
    bool same = true;
    fe_t y2 = Fq::sqr(y);
    for (int j = 0; j < 8; ++j) same &= y2.l[j] == rhs.l[j];
    if (!same) return false;
    fe_t yc = Fq::from_mont(y);
    if ((yc.l[0] & 1u) != sign) y = Fq::neg(y);
    out->x = xm; out->y = y;
    return true;
}

// k * p for a small scalar (double-and-add, MSB first)
ZK_D xyzz_t xyzz_mul_small(const xyzz_t& p, uint32_t k) {
    xyzz_t acc = xyzz_identity();
    for (int i = 31; i >= 0; --i) {
        acc = xyzz_dbl(acc);
        if ((k >> i) & 1) xyzz_add(acc, p);
    }
    return acc;
}

}  // namespace b200zk
