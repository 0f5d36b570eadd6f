// Number-theoretic transform over G1 points: halo2_proofs v2023_02_02 `arithmetic::g_to_lagrange`
// (src/arithmetic.rs), which ParamsKZG::downsize (src/poly/kzg/commitment.rs) uses to rebuild the
// Lagrange basis of a truncated SRS:
//   g_lagrange[i] = n^-1 * sum_j w^(-ij) * g[j],   n = 2^k, w the primitive n-th root of unity of Fr.
// Radix-2 decimation in time on XYZZ points (curve.cuh): bit-reversed load, k stages of butterflies
// (a, b) -> (a + t*b, a - t*b), then the n^-1 scaling.  Each multiplication by a twiddle is a full
// variable-base scalar multiplication, so the transform is arithmetic bound (about 3 300 Fq
// multiplications per butterfly against 512 B of traffic).  Per-thread bodies only; the launches
// are in setup.cu, and the same bodies run on a host compiler under ptx_chain.cuh emulation.
#pragma once
#include "curve.cuh"

namespace b200zk {

ZK_D xyzz_t xyzz_neg(const xyzz_t& p) {
    xyzz_t r = p;
    r.y = Fq::neg(p.y);
    return r;
}

// s * p for a canonical (non-Montgomery) Fr scalar s < r < 2^254.  Signed 4-bit windows
// d_i = nibble_i - 16 * bit(4i + 3) + bit(4i - 1), so sum d_i 16^i = s and |d_i| <= 8: a table of
// 1p ... 8p, 63 * 4 doublings and at most 64 additions.  Each digit depends on its own bits only,
// so the recoding runs most significant window first with no carry state.  Complete: xyzz_add and
// xyzz_dbl handle the identity, P + P and P + (-P).
ZK_D xyzz_t xyzz_mul(const xyzz_t& p, const fe_t& s) {
    xyzz_t tab[8];
    tab[0] = p;
    tab[1] = xyzz_dbl(p);
    for (int i = 2; i < 8; ++i) { tab[i] = tab[i - 1]; xyzz_add(tab[i], p); }
    xyzz_t acc = xyzz_identity();
    for (int i = 63; i >= 0; --i) {
        if (i != 63) for (int d = 0; d < 4; ++d) acc = xyzz_dbl(acc);
        uint32_t nib = (s.l[i >> 3] >> ((i & 7) * 4)) & 0xf;
        uint32_t below = i ? (s.l[(4 * i - 1) >> 5] >> ((4 * i - 1) & 31)) & 1 : 0;
        int32_t dig = (int32_t)nib - (int32_t)((nib >> 3) << 4) + (int32_t)below;
        if (dig > 0) xyzz_add(acc, tab[dig - 1]);
        else if (dig < 0) xyzz_add(acc, xyzz_neg(tab[-dig - 1]));
    }
    return acc;
}

// One butterfly of a stage with twiddle w (canonical).  `trivial` (w = 1) skips the multiplication.
ZK_D void g1_ntt_butterfly(xyzz_t& a, xyzz_t& b, const fe_t& w, bool trivial) {
    xyzz_t t = trivial ? b : xyzz_mul(b, w);
    b = a;
    xyzz_add(a, t);
    xyzz_add(b, xyzz_neg(t));
}

// Butterfly t of stage s (half-length h = 2^s) of a 2^k-point transform, j-major: j = t / B, block
// t mod B with B = n / 2h blocks.  While B >= 32, a warp shares one j, so the twiddle-1 butterflies
// (j = 0) of a stage are whole warps.  Pairs (i0, i0 + h); twiddle w^(-j * B) = tw[j * B].
struct G1NttPair { size_t i0, i1, tw; };
ZK_D G1NttPair g1_ntt_pair(size_t t, uint32_t s, uint32_t k) {
    const uint32_t log_b = k - 1 - s;
    const size_t j = t >> log_b, blk = t & (((size_t)1 << log_b) - 1);
    G1NttPair r;
    r.i0 = (blk << (s + 1)) + j;
    r.i1 = r.i0 + ((size_t)1 << s);
    r.tw = j << log_b;
    return r;
}

// Butterfly t of stage s in place over a[]; tw holds w^-j, j < n/2, in Montgomery form.
ZK_D void g1_ntt_stage_body(xyzz_t* a, const fe_t* tw, size_t t, uint32_t s, uint32_t k) {
    G1NttPair pr = g1_ntt_pair(t, s, k);
    bool trivial = pr.tw == 0;
    fe_t w = trivial ? Fr::zero() : Fr::from_mont(tw[pr.tw]);
    xyzz_t x = a[pr.i0], y = a[pr.i1];
    g1_ntt_butterfly(x, y, w, trivial);
    a[pr.i0] = x;
    a[pr.i1] = y;
}

}  // namespace b200zk
