// TEST AID: the per-thread bodies of csrc/g1_ntt.cuh compiled with a host compiler (carry flag emulated,
// see csrc/ptx_chain.cuh) and driven in the launch order of g_to_lagrange_run (csrc/setup.cu), next to a
// statement-for-statement restatement of halo2_proofs v2023_02_02 `arithmetic::g_to_lagrange`
// (src/arithmetic.rs) over the reference types of oracle/.  Built together with oracle/arith.cpp into one
// shared object by tests/g1_ntt_ref.py.  Never linked into the product library.
#include <thread>
#include <vector>
#include <cstring>
#include "../halo2-experiments_b200/csrc/g1_ntt.cuh"
#include "../halo2-experiments_b200/csrc/poly.cuh"
#include "../halo2-experiments_b200/csrc/host_field.hpp"
#include "../oracle/arith.hpp"

namespace {

using b200zk::affine_t;
using b200zk::fe_t;
using b200zk::xyzz_t;

// the device types are 32-byte aligned, numpy's buffers need not be: every array crosses the boundary by memcpy
template <class T> std::vector<T> load(const void* src, size_t n) {
    std::vector<T> v(n);
    memcpy(v.data(), src, n * sizeof(T));
    return v;
}

// setup_normalize_kernel after batch_invert_run(.., 1), one lane; out unaligned
void normalize(std::vector<xyzz_t>& p, void* out_bytes) {
    std::vector<affine_t> out(p.size());
    size_t n = p.size();
    std::vector<fe_t> zzz(n), scratch(n);
    for (size_t i = 0; i < n; ++i) zzz[i] = p[i].zzz;
    b200zk::batch_invert_lane<b200zk::Fq>(zzz.data(), scratch.data(), n, 0, 1);
    for (size_t i = 0; i < n; ++i) {
        if (b200zk::Fq::is_zero(p[i].zz)) { out[i].x = b200zk::Fq::zero(); out[i].y = b200zk::Fq::zero(); continue; }
        fe_t t = b200zk::Fq::mul(p[i].zz, zzz[i]);
        out[i].x = b200zk::Fq::mul(p[i].x, b200zk::Fq::sqr(t));
        out[i].y = b200zk::Fq::mul(p[i].y, zzz[i]);
    }
    memcpy(out_bytes, out.data(), n * sizeof(affine_t));
}

// ---- restatement of upstream (G = G1 projective) ----
using orc::Fr;
using orc::G1;

size_t bitreverse(size_t n, unsigned l) {
    size_t r = 0;
    for (unsigned i = 0; i < l; ++i) { r = (r << 1) | (n & 1); n >>= 1; }
    return r;
}
// recursive_butterfly_arithmetic: `let t = a[n/2 + i] * twiddle; a[n/2 + i] = a[i]; a[i] += t; a[n/2 + i] -= t`,
// with the halves joined on two threads down to par_depth levels, as the Fr restatement of best_fft does
void butterfly_layer(G1* left, G1* right, size_t half, size_t twiddle_chunk, const Fr* tw) {
    G1 t = right[0]; right[0] = left[0]; left[0] = left[0].add(t); right[0] = right[0].add(t.neg());
    for (size_t i = 1; i < half; ++i) {
        G1 t2 = right[i].mul(tw[i * twiddle_chunk]);
        right[i] = left[i]; left[i] = left[i].add(t2); right[i] = right[i].add(t2.neg());
    }
}
void recursive_butterfly(G1* a, size_t n, size_t twiddle_chunk, const Fr* tw, int par_depth) {
    if (n == 2) { G1 t = a[1]; a[1] = a[0]; a[0] = a[0].add(t); a[1] = a[1].add(t.neg()); return; }
    if (par_depth > 0) {
        std::thread other([=] { recursive_butterfly(a, n / 2, twiddle_chunk * 2, tw, par_depth - 1); });
        recursive_butterfly(a + n / 2, n / 2, twiddle_chunk * 2, tw, par_depth - 1);
        other.join();
    } else {
        recursive_butterfly(a, n / 2, twiddle_chunk * 2, tw, 0);
        recursive_butterfly(a + n / 2, n / 2, twiddle_chunk * 2, tw, 0);
    }
    butterfly_layer(a, a + n / 2, n / 2, twiddle_chunk, tw);
}
// arithmetic::best_fft
void best_fft(G1* a, const Fr& omega, unsigned log_n) {
    size_t n = (size_t)1 << log_n;
    int threads = orc::num_threads();
    unsigned log_threads = 0; while ((2 << log_threads) <= threads) ++log_threads;
    for (size_t k = 0; k < n; ++k) { size_t rk = bitreverse(k, log_n); if (k < rk) std::swap(a[rk], a[k]); }
    std::vector<Fr> tw(n / 2 ? n / 2 : 1, Fr::one());
    orc::parallelize(n / 2, [&](size_t s, size_t e) { Fr w = omega.pow_u64(s); for (size_t i = s; i < e; ++i) { tw[i] = w; w *= omega; } });
    if (log_n <= log_threads) {
        size_t chunk = 2, twiddle_chunk = n / 2;
        for (unsigned l = 0; l < log_n; ++l) {
            for (size_t s = 0; s < n; s += chunk) butterfly_layer(a + s, a + s + chunk / 2, chunk / 2, twiddle_chunk, tw.data());
            chunk *= 2; twiddle_chunk /= 2;
        }
    } else {
        recursive_butterfly(a, n, 1, tw.data(), (int)log_threads);
    }
}

}  // namespace

extern "C" {

// out[i] = s[i] * p[i] through xyzz_mul; s canonical (4 x u64), p and out G1Affine
void g1h_xyzz_mul(const void* p_bytes, const void* s_bytes, void* out, size_t n) {
    std::vector<affine_t> p = load<affine_t>(p_bytes, n);
    std::vector<fe_t> s = load<fe_t>(s_bytes, n);
    std::vector<xyzz_t> r(n);
    for (size_t i = 0; i < n; ++i) r[i] = b200zk::xyzz_mul(b200zk::xyzz_from_affine(p[i]), s[i]);
    normalize(r, out);
}

// g_to_lagrange_run on the host: bit-reversed load, k stages of g1_ntt_stage_body, n^-1, normalisation
void g1h_g_to_lagrange_emu(const void* g_bytes, uint32_t k, void* out) {
    using b200zk::host::HFr;
    const size_t n = (size_t)1 << k, half = n / 2;
    std::vector<affine_t> g = load<affine_t>(g_bytes, n);
    HFr omega_inv = b200zk::host::fr_root_of_unity();
    for (uint32_t i = k; i < b200zk::host::FR_TWO_ADICITY; ++i) omega_inv = omega_inv.sqr();
    omega_inv = omega_inv.inv();
    std::vector<fe_t> tw(half);
    HFr w = HFr::one();
    for (size_t j = 0; j < half; ++j) { memcpy(tw[j].l, w.v, 32); w = w * omega_inv; }
    std::vector<xyzz_t> a(n);
    for (size_t i = 0; i < n; ++i) a[i] = b200zk::xyzz_from_affine(g[k ? bitreverse(i, k) : 0]);
    for (uint32_t s = 0; s < k; ++s)
        for (size_t t = 0; t < half; ++t) b200zk::g1_ntt_stage_body(a.data(), tw.data(), t, s, k);
    uint64_t n_inv[4];
    HFr::from_u64(n).inv().to_canonical(n_inv);
    fe_t n_inv_d; memcpy(n_inv_d.l, n_inv, 32);
    for (size_t i = 0; i < n; ++i) a[i] = b200zk::xyzz_mul(a[i], n_inv_d);
    normalize(a, out);
}

// arithmetic::g_to_lagrange(g_projective, k), on `threads` host threads (0 = all cores)
void g1h_g_to_lagrange_ref(const uint64_t* g_aff, uint32_t k, uint64_t* out_aff, int threads) {
    orc::init_fields();
    if (threads > 0) orc::set_num_threads(threads);
    const size_t n = (size_t)1 << k;
    const orc::G1Affine* g = (const orc::G1Affine*)g_aff;
    // let n_inv = C::Scalar::TWO_INV.pow_vartime(&[k as u64, 0, 0, 0]);
    Fr n_inv = Fr::from_u64(2).inv().pow_u64(k);
    // let mut omega_inv = C::Scalar::ROOT_OF_UNITY_INV; for _ in k..C::Scalar::S { omega_inv = omega_inv.square(); }
    Fr omega_inv = orc::FR_ROOT_OF_UNITY.inv();
    for (uint32_t i = k; i < 28; ++i) omega_inv = omega_inv.sqr();
    std::vector<G1> gp(n);
    for (size_t i = 0; i < n; ++i) gp[i] = G1::from_affine(g[i]);
    // best_fft(&mut g_lagrange_projective, omega_inv, k);
    best_fft(gp.data(), omega_inv, k);
    // parallelize(&mut g_lagrange_projective, |g, _| for g in g.iter_mut() { *g *= n_inv; });
    orc::parallelize(n, [&](size_t s, size_t e) { for (size_t i = s; i < e; ++i) gp[i] = gp[i].mul(n_inv); });
    // parallelize(&mut g_lagrange, |g_lagrange, starts| C::Curve::batch_normalize(&projective[starts..], g_lagrange));
    orc::G1Affine* out = (orc::G1Affine*)out_aff;
    orc::parallelize(n, [&](size_t s, size_t e) { orc::batch_normalize(gp.data() + s, out + s, e - s); });
    if (threads > 0) orc::set_num_threads(0);
}

}  // extern "C"
