// TEST AID: the per-thread bodies of csrc/pairing.cuh compiled with a host compiler (carry flag emulated, see
// csrc/ptx_chain.cuh), next to the host pairing of csrc/pairing.hpp that b200zk_pairing_check and verify_proof use.
// Built into one shared object by tests/pairing_ref.py.  Never linked into the product library.
// Every array crosses the boundary by memcpy: the device types are 32-byte aligned, numpy's buffers need not be.
// `which` selects the implementation: 0 = the device bodies, 1 = the host pairing.
#include <cstring>
#include <vector>
#include "../halo2-experiments_b200/csrc/pairing.cuh"
#include "../halo2-experiments_b200/csrc/pairing.hpp"

namespace {

using namespace b200zk;
using host::F2;
using host::F12;

template <class T> T load1(const void* src, size_t i) { T v; memcpy(&v, (const uint8_t*)src + i * sizeof(T), sizeof(T)); return v; }
template <class T> void store1(void* dst, size_t i, const T& v) { memcpy((uint8_t*)dst + i * sizeof(T), &v, sizeof(T)); }

static_assert(sizeof(fq2_t) == sizeof(F2) && sizeof(fq12_t) == sizeof(F12), "device and host towers share one layout");

F12 host_pow(const F12& a, const uint64_t* e, size_t nlimbs) {
    F12 acc = host::f12_one();
    for (size_t i = nlimbs * 64; i-- > 0;) {
        acc = host::f12_mul(acc, acc);
        if ((e[i >> 6] >> (i & 63)) & 1) acc = host::f12_mul(acc, a);
    }
    return acc;
}

}  // namespace

extern "C" {

// op 0: a * b, 1: a^2, 2: a^-1
void ph_fq2(int op, const void* a, const void* b, void* out, size_t n, int which) {
    for (size_t i = 0; i < n; ++i) {
        if (which == 0) {
            fq2_t x = load1<fq2_t>(a, i), y = load1<fq2_t>(b, i);
            store1(out, i, op == 0 ? fq2_mul(x, y) : op == 1 ? fq2_sqr(x) : fq2_inv(x));
        } else {
            F2 x = load1<F2>(a, i), y = load1<F2>(b, i);
            store1(out, i, op == 0 ? host::f2_mul(x, y) : op == 1 ? host::f2_mul(x, x) : host::f2_inv(x));
        }
    }
}

// op 0: a * b, 1: a^2, 2: a^-1, 3: cyclotomic a^2, 4: easy part, 5: final exponentiation, 6 / 7 / 8: a^q, a^(q^2), a^(q^3).
// The host implements 0, 1 and 5.
void ph_fq12(int op, const void* a, const void* b, void* out, size_t n, int which) {
    for (size_t i = 0; i < n; ++i) {
        if (which == 0) {
            fq12_t x = load1<fq12_t>(a, i), y = load1<fq12_t>(b, i), r;
            switch (op) {
            case 0: r = fq12_mul(x, y); break;
            case 1: r = fq12_sqr(x); break;
            case 2: r = fq12_inv(x); break;
            case 3: r = fq12_cyc_sqr(x); break;
            case 4: r = fq12_easy_part(x); break;
            case 5: r = fq12_final_exp(x); break;
            default: r = fq12_frob(x, op - 5); break;
            }
            store1(out, i, r);
        } else {
            F12 x = load1<F12>(a, i), y = load1<F12>(b, i);
            store1(out, i, op == 0 ? host::f12_mul(x, y) : op == 1 ? host::f12_mul(x, x) : host::final_exponentiation(x));
        }
    }
}

// a^e on the host, e as nlimbs little-endian u64 limbs (plain square-and-multiply)
void ph_fq12_pow(const void* a, const uint64_t* e, size_t nlimbs, void* out, size_t n) {
    for (size_t i = 0; i < n; ++i) store1(out, i, host_pow(load1<F12>(a, i), e, nlimbs));
}

// f * line(P): device fq12_mul_by_line, or the host's dense product with the same line
void ph_line(const void* f, const void* lines, const void* p, void* out, size_t n, int which) {
    for (size_t i = 0; i < n; ++i) {
        pc_line_t l = load1<pc_line_t>(lines, i);
        affine_t pa = load1<affine_t>(p, i);
        if (which == 0) { store1(out, i, fq12_mul_by_line(load1<fq12_t>(f, i), l, pa)); continue; }
        F12 d = host::f12_one();
        F2 c0, c1, c2; memcpy(&c0, &l.c0, 64); memcpy(&c1, &l.c1, 64); memcpy(&c2, &l.c2, 64);
        host::HFq px, py; memcpy(px.v, pa.x.l, 32); memcpy(py.v, pa.y.l, 32);
        d.c[0] = host::f2_scale(c0, py); d.c[1] = host::f2_scale(c1, px); d.c[2] = host::f2_zero(); d.c[3] = c2;
        d.c[4] = host::f2_zero(); d.c[5] = host::f2_zero();
        store1(out, i, host::f12_mul(load1<F12>(f, i), d));
    }
}

// prod_{i < m} e(g1[j m + i], g2[j m + i]) for j < count, before the verdict: device = one line table per distinct G2
// point (by bytes), pc_miller_product and fq12_final_exp; host = final_exponentiation(prod miller_loop), identities skipped
void ph_pairing(const void* g1, const void* g2, uint32_t m, size_t count, void* out, int which) {
    for (size_t j = 0; j < count; ++j) {
        if (which == 1) {
            F12 f = host::f12_one();
            for (uint32_t i = 0; i < m; ++i) {
                const uint8_t* pq = (const uint8_t*)g2 + 128 * (j * m + i);
                host::HAffine p = load1<host::HAffine>(g1, j * m + i);
                host::G2A q = host::g2_from_limbs(pq);
                if ((p.x.is_zero() && p.y.is_zero()) || host::g2_is_identity(q)) continue;
                f = host::f12_mul(f, host::miller_loop(q, p));
            }
            store1(out, j, host::final_exponentiation(f));
            continue;
        }
        std::vector<affine_t> ps(m);
        std::vector<uint32_t> qi(m);
        std::vector<const uint8_t*> distinct;
        std::vector<pc_line_t> tables;
        for (uint32_t i = 0; i < m; ++i) {
            const uint8_t* pq = (const uint8_t*)g2 + 128 * (j * m + i);
            ps[i] = load1<affine_t>(g1, j * m + i);
            fq2_t qx = load1<fq2_t>(pq, 0), qy = load1<fq2_t>(pq, 1);
            bool q_id = Fq::is_zero(qx.a) && Fq::is_zero(qx.b) && Fq::is_zero(qy.a) && Fq::is_zero(qy.b);
            if (affine_is_identity(ps[i]) || q_id) { qi[i] = PC_SKIP; continue; }
            uint32_t k = 0;
            while (k < distinct.size() && memcmp(distinct[k], pq, 128)) ++k;
            if (k == distinct.size()) {
                distinct.push_back(pq);
                tables.resize(distinct.size() * PC_LINES);
                g2_prepare(qx, qy, &tables[k * PC_LINES]);
            }
            qi[i] = k;
        }
        store1(out, j, fq12_final_exp(pc_miller_product(ps.data(), qi.data(), tables.data(), m)));
    }
}

// s[i] * G1 generator and s[i] * G2 generator on the host (s canonical, 4 x u64); G1Affine 64 B, G2Affine 128 B
void ph_g1_mul(const uint64_t* s, void* out, size_t n) {
    const host::HAffine gen = {host::HFq::from_u64(1), host::HFq::from_u64(2)};
    for (size_t i = 0; i < n; ++i) {
        host::HXyzz acc = host::hx_identity(), base = host::hx_from_affine(gen);
        for (int b = 255; b >= 0; --b) {
            acc = host::hx_dbl(acc);
            if ((s[4 * i + (b >> 6)] >> (b & 63)) & 1) acc = host::hx_add(acc, base);
        }
        store1(out, i, host::hx_to_affine(acc));
    }
}
void ph_g2_mul(const uint64_t* s, void* out, size_t n) {
    for (size_t i = 0; i < n; ++i) host::g2_store(host::g2_mul(host::g2_generator(), host::HFr::from_canonical(s + 4 * i)), (uint8_t*)out + 128 * i);
}

}  // extern "C"
