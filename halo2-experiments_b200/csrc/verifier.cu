// plonk::verify_proof + VerifierSHPLONK + the KZG pairing check on the host: halo2_proofs
// v2023_02_02 src/plonk/verifier.rs, src/poly/kzg/multiopen/shplonk/verifier.rs and
// src/poly/kzg/strategy.rs — the call `full_prover` makes at
// /root/reference/src/circuits/utils.rs:52-63 (`verify_proof(..).is_ok()`, the reference's only
// assertion on the hot path).  SURVEY.md §8 row f3.
//
// Verification is O(#queries) field work, one ~100-term G1 combination and two Miller loops: it runs
// on the caller's thread with no device and no ctx, exactly like the Blake2b transcript of the
// prover.  replay_proof (verify_replay.hpp) is the transcript replay; it returns the opening as
// linear terms, which b200zk_verify_proof evaluates here and b200zk_verify_proofs (verify_batch.cu)
// evaluates on the device for many proofs at once.  The O(n) work a verifying key needs — the commitments to the fixed and permutation
// polynomials (keygen_vk) — is done on the device by b200zk_pk_vk_commitments (prover.cu).
#include <cstring>
#include <vector>
#include "../../include/b200zk.h"
#include "cs_desc.hpp"
#include "pairing.hpp"
#include "transcript.hpp"
#include "verify_replay.hpp"

using namespace b200zk;
using namespace b200zk::host;

namespace {

int cmp_canon(const HFr& a, const HFr& b) {
    uint64_t x[4], y[4]; a.to_canonical(x); b.to_canonical(y);
    for (int i = 3; i >= 0; --i) if (x[i] != y[i]) return x[i] < y[i] ? -1 : 1;
    return 0;
}

// G1Affine::from_bytes (halo2curves 0.3.1 compressed form): x little-endian, the parity of y in
// bit 7 of byte 31, identity = all zero.  Returns false for a non-canonical x or a point off the curve.
bool decompress_g1(const uint8_t* b, HAffine* out) {
    uint8_t t[32]; memcpy(t, b, 32);
    unsigned sign = t[31] >> 7;
    t[31] &= 0x7f;
    uint64_t xc[4]; memcpy(xc, t, 32);
    if (HFq::ge_p(xc)) return false;
    if ((xc[0] | xc[1] | xc[2] | xc[3]) == 0) {
        if (sign) return false;
        *out = {HFq::zero(), HFq::zero()};
        return true;
    }
    HFq x = HFq::from_canonical(xc);
    HFq rhs = x.sqr() * x + HFq::from_u64(3);
    static const uint64_t E[4] = {0x4f082305b61f3f52ULL, 0x65e05aa45a1c72a3ULL, 0x6e14116da0605617ULL, 0x0c19139cb84c680aULL};   // (q + 1) / 4
    HFq y = rhs.pow(E);
    if (y.sqr() != rhs) return false;
    uint64_t yc[4]; y.to_canonical(yc);
    if ((yc[0] & 1) != sign) y = y.neg();
    *out = {x, y};
    return true;
}

HXyzz g1_mul(const HAffine& p, const HFr& s) {
    uint64_t e[4]; s.to_canonical(e);
    HXyzz base = hx_from_affine(p), acc = hx_identity();
    for (int i = 255; i >= 0; --i) {
        acc = hx_dbl(acc);
        if ((e[i >> 6] >> (i & 63)) & 1) acc = hx_add(acc, base);
    }
    return acc;
}

}  // namespace

namespace b200zk {
HAffine open_base_point(const VkPoints& vk, const HAffine* proof_points, const OpenBase& b) {
    auto at = [](const void* base, size_t i) {
        const uint64_t* p = (const uint64_t*)base + 8 * i;
        return HAffine{HFq::from_limbs(p), HFq::from_limbs(p + 4)};
    };
    switch (b.kind) {
    case OpenBase::FIXED: return at(vk.fixed, b.idx);
    case OpenBase::SIGMA: return at(vk.sigma, b.idx);
    case OpenBase::GEN: return at(vk.g1, 0);
    default: return proof_points[b.idx];
    }
}
}  // namespace b200zk

namespace {

// TranscriptRead side of Blake2bRead<_, G1Affine, Challenge255<_>> (src/transcript.rs).  Points are decompressed here,
// or taken from `pre` (the proof's points decompressed by the caller, in read order); either way they are kept in `pts`.
struct Reader {
    Transcript tr;
    const uint8_t* buf; size_t len, pos = 0; bool ok = true;
    const HAffine* pre;
    std::vector<HAffine> pts;
    Reader(const uint8_t* b, size_t l, const HAffine* p) : buf(b), len(l), pre(p) {}
    uint32_t read_point() {
        HAffine p = {HFq::zero(), HFq::zero()};
        if (!ok || pos + 32 > len) ok = false;
        else if (pre) p = pre[pts.size()];
        else if (!decompress_g1(buf + pos, &p)) ok = false;
        if (ok) { pos += 32; tr.common_point(p); }
        else p = {HFq::zero(), HFq::zero()};
        pts.push_back(p);
        return (uint32_t)(pts.size() - 1);
    }
    HFr read_scalar() {
        if (!ok || pos + 32 > len) { ok = false; return HFr::zero(); }
        uint64_t c[4]; memcpy(c, buf + pos, 32);
        if (HFr::ge_p(c)) { ok = false; return HFr::zero(); }
        pos += 32;
        HFr s = HFr::from_canonical(c);
        tr.common_scalar(s);
        return s;
    }
    HFr squeeze() { return tr.squeeze_challenge(); }
};

// Expression::evaluate at the opening point (verifier.rs: gate / lookup expressions over the *_evals)
bool eval_expr_at(const CsDesc& cs, uint32_t off, uint32_t len, const std::vector<HFr>& fx, const std::vector<HFr>& ad,
                  const std::vector<HFr>& in, HFr* out) {
    std::vector<HFr> st;
    for (uint32_t i = off; i < off + len; ++i) {
        uint32_t op = cs.prog[i] & 0xff, arg = cs.prog[i] >> 8;
        switch (op) {
        case EX_CONST: st.push_back(cs.consts[arg]); break;
        case EX_FIXED: st.push_back(fx[arg]); break;
        case EX_ADVICE: st.push_back(ad[arg]); break;
        case EX_INSTANCE: st.push_back(in[arg]); break;
        case EX_NEG: if (st.empty()) return false; st.back() = st.back().neg(); break;
        case EX_SCALE: if (st.empty()) return false; st.back() = st.back() * cs.consts[arg]; break;
        case EX_ADD: case EX_MUL: {
            if (st.size() < 2) return false;
            HFr b = st.back(); st.pop_back();
            st.back() = op == EX_ADD ? st.back() + b : st.back() * b;
            break;
        }
        default: return false;
        }
    }
    if (st.size() != 1) return false;
    *out = st[0];
    return true;
}

int find_query(const std::vector<int32_t>& q, uint32_t col, int32_t rot) {
    for (size_t i = 0; i + 1 < q.size(); i += 2) if ((uint32_t)q[i] == col && q[i + 1] == rot) return (int)(i / 2);
    return -1;
}

struct Query { int cid; OpenBase c; HFr pt, eval; };
struct CommitSet { int cid; OpenBase c; std::vector<HFr> pts, evals; };     // one commitment, its points in first-seen order
struct RotSet { std::vector<HFr> pts; std::vector<size_t> members; };        // sorted point set, commitments in first-seen order

std::vector<HFr> interpolate(const std::vector<HFr>& pts, const std::vector<HFr>& evals) {
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

}  // namespace

extern "C" {

int32_t b200zk_g2_mul(const void* g2_or_null, const void* s_fr, void* out_g2) {
    if (!s_fr || !out_g2) return B200ZK_EINVAL;
    G2A base = g2_or_null ? g2_from_limbs(g2_or_null) : g2_generator();
    if (!g2_on_curve(base)) return B200ZK_EINVAL;
    g2_store(g2_mul(base, HFr::from_limbs(s_fr)), out_g2);
    return B200ZK_OK;
}

int32_t b200zk_pairing_check(const void* g1_points, const void* g2_points, size_t count) {
    if (count && (!g1_points || !g2_points)) return B200ZK_EINVAL;
    std::vector<HAffine> ps(count);
    std::vector<G2A> qs(count);
    for (size_t i = 0; i < count; ++i) {
        const uint64_t* p = (const uint64_t*)g1_points + 8 * i;
        ps[i] = {HFq::from_limbs(p), HFq::from_limbs(p + 4)};
        qs[i] = g2_from_limbs((const uint8_t*)g2_points + 128 * i);
        bool id1 = ps[i].x.is_zero() && ps[i].y.is_zero();
        if (!id1 && ps[i].y.sqr() != ps[i].x.sqr() * ps[i].x + HFq::from_u64(3)) return B200ZK_EINVAL;
        if (!g2_on_curve(qs[i])) return B200ZK_EINVAL;
    }
    return pairing_product_is_one(ps.data(), qs.data(), count) ? B200ZK_OK : B200ZK_EVERIFY;
}


}  // extern "C"

namespace b200zk {

size_t proof_point_offsets(const CsDesc& cs, std::vector<size_t>* offs) {
    const size_t L = cs.lookups.size(), P = cs.perm.size(), chunk = cs.degree - 2, S = (P + chunk - 1) / chunk;
    const size_t commitments = cs.A + 2 * L + S + L + 1 + (cs.degree - 1);
    const size_t evals = cs.adv_q.size() / 2 + cs.fix_q.size() / 2 + 1 + P + (S ? 3 * S - 1 : 0) + 5 * L;
    offs->clear();
    for (size_t i = 0; i < commitments; ++i) offs->push_back(32 * i);
    offs->push_back(32 * (commitments + evals));           // h1
    offs->push_back(32 * (commitments + evals + 1));       // h2
    return 32 * (commitments + evals + 2);
}

int32_t replay_proof(const CsDesc& cs, const VkPoints& vk, const void* const* instance_columns, const uint32_t* instance_lens,
                     const void* transcript_repr, const uint8_t* proof, size_t proof_len, const HAffine* points, Opening* out) {
    const uint32_t k = cs.k, bf = cs.bf;
    const uint64_t n = 1ull << k;
    const size_t A = cs.A, L = cs.lookups.size(), P = cs.perm.size();
    const size_t chunk = cs.degree - 2, S = (P + chunk - 1) / chunk, q = cs.degree - 1;

    // ---- instances: length check (Error::InstanceTooLarge), absorbed as scalars (KZG: query_instance = false)
    std::vector<std::vector<HFr>> inst(cs.I);
    for (uint32_t c = 0; c < cs.I; ++c) {
        if (instance_lens[c] > n - (bf + 1)) return B200ZK_EVERIFY;
        if (instance_lens[c] && !instance_columns[c]) return B200ZK_EINVAL;
        for (uint32_t i = 0; i < instance_lens[c]; ++i) inst[c].push_back(HFr::from_limbs((const uint8_t*)instance_columns[c] + 32 * (size_t)i));
    }
    Reader rd(proof, proof_len, points);
    rd.tr.common_scalar(HFr::from_limbs(transcript_repr));
    for (auto& col : inst) for (auto& v : col) rd.tr.common_scalar(v);

    // ---- commitments (indices into rd.pts) and challenges, in the prover's order (verifier.rs)
    std::vector<uint32_t> advice_c(A), lk_a(L), lk_s(L), perm_c(S), lk_z(L), h_c(q);
    for (auto& c : advice_c) c = rd.read_point();
    HFr theta = rd.squeeze();
    for (size_t i = 0; i < L; ++i) { lk_a[i] = rd.read_point(); lk_s[i] = rd.read_point(); }
    HFr beta = rd.squeeze(), gamma = rd.squeeze();
    for (auto& c : perm_c) c = rd.read_point();
    for (auto& c : lk_z) c = rd.read_point();
    uint32_t random_c = rd.read_point();
    HFr y = rd.squeeze();
    for (auto& c : h_c) c = rd.read_point();
    HFr x = rd.squeeze();

    // ---- evaluations
    size_t naq = cs.adv_q.size() / 2, nfq = cs.fix_q.size() / 2, niq = cs.inst_q.size() / 2;
    std::vector<HFr> advice_ev(naq), fixed_ev(nfq), sigma_ev(P), instance_ev(niq);
    for (auto& e : advice_ev) e = rd.read_scalar();
    for (auto& e : fixed_ev) e = rd.read_scalar();
    HFr random_ev = rd.read_scalar();
    for (auto& e : sigma_ev) e = rd.read_scalar();
    struct PermEv { HFr z, z_next, z_last; };
    std::vector<PermEv> perm_ev(S);
    for (size_t s = 0; s < S; ++s) {
        perm_ev[s].z = rd.read_scalar(); perm_ev[s].z_next = rd.read_scalar();
        perm_ev[s].z_last = s + 1 < S ? rd.read_scalar() : HFr::zero();
    }
    struct LkEv { HFr z, z_next, a, a_prev, s; };
    std::vector<LkEv> lk_ev(L);
    for (auto& e : lk_ev) { e.z = rd.read_scalar(); e.z_next = rd.read_scalar(); e.a = rd.read_scalar(); e.a_prev = rd.read_scalar(); e.s = rd.read_scalar(); }
    if (!rd.ok) return B200ZK_EVERIFY;                     // Error::Transcript / malformed proof

    // ---- domain constants (EvaluationDomain::new)
    HFr omega = fr_root_of_unity();
    for (uint32_t i = k; i < FR_TWO_ADICITY; ++i) omega = omega.sqr();
    HFr omega_inv = omega.inv(), n_inv = HFr::from_u64(n).inv();
    auto rotate = [&](const HFr& pt, int rot) { return rot >= 0 ? pt * omega.pow_u64((uint64_t)rot) : pt * omega_inv.pow_u64((uint64_t)(-(int64_t)rot)); };
    auto pow_n = [&](HFr v) { for (uint32_t i = 0; i < k; ++i) v = v.sqr(); return v; };
    // l_i(pt) = (pt^n - 1) / n * omega^i / (pt - omega^i); i taken mod n
    auto l_i = [&](const HFr& pt, const HFr& ptn, int64_t i) {
        HFr wi = i >= 0 ? omega.pow_u64((uint64_t)i) : omega_inv.pow_u64((uint64_t)(-i));
        return (ptn - HFr::one()) * n_inv * wi * (pt - wi).inv();
    };
    HFr xn = pow_n(x);
    if (xn == HFr::one()) return B200ZK_EVERIFY;          // x in the domain: probability 2^-226, upstream would divide by zero
    // instance evaluations from the public inputs (Lagrange basis)
    for (size_t qi = 0; qi < niq; ++qi) {
        uint32_t col = (uint32_t)cs.inst_q[2 * qi];
        HFr xr = rotate(x, cs.inst_q[2 * qi + 1]), xrn = pow_n(xr), acc = HFr::zero();
        for (size_t i = 0; i < inst[col].size(); ++i) acc = acc + inst[col][i] * l_i(xr, xrn, (int64_t)i);
        instance_ev[qi] = acc;
    }
    HFr l_0 = l_i(x, xn, 0), l_last = l_i(x, xn, -(int64_t)(bf + 1)), l_blind = HFr::zero();
    for (uint32_t j = 1; j <= bf; ++j) l_blind = l_blind + l_i(x, xn, -(int64_t)j);
    HFr one = HFr::one(), l_active = one - l_last - l_blind;

    // ---- expected h(x): every term of evaluate_h at x, folded in y
    HFr expected = HFr::zero();
    auto fold = [&](const HFr& t) { expected = expected * y + t; };
    for (auto& g : cs.gates) {
        HFr v;
        if (!eval_expr_at(cs, g.first, g.second, fixed_ev, advice_ev, instance_ev, &v)) return B200ZK_EINVAL;
        fold(v);
    }
    if (S) {
        std::vector<HFr> col_ev(P);
        for (size_t j = 0; j < P; ++j) {
            uint32_t ct = cs.perm[j].first, ci = cs.perm[j].second;
            int qi = find_query(ct == 0 ? cs.adv_q : ct == 1 ? cs.fix_q : cs.inst_q, ci, 0);
            if (qi < 0 || ct > 2) return B200ZK_EINVAL;
            col_ev[j] = ct == 0 ? advice_ev[qi] : ct == 1 ? fixed_ev[qi] : instance_ev[qi];
        }
        fold(l_0 * (one - perm_ev[0].z));
        HFr zl = perm_ev[S - 1].z;
        fold(l_last * (zl.sqr() - zl));
        for (size_t s = 1; s < S; ++s) fold(l_0 * (perm_ev[s].z - perm_ev[s - 1].z_last));
        HFr delta = fr_delta(), cur = beta * x;
        for (size_t s = 0; s < S; ++s) {
            HFr left = perm_ev[s].z_next, right = perm_ev[s].z;
            for (size_t j = s * chunk; j < std::min(P, (s + 1) * chunk); ++j) {
                left = left * (col_ev[j] + beta * sigma_ev[j] + gamma);
                right = right * (col_ev[j] + cur + gamma);
                cur = cur * delta;
            }
            fold(l_active * (left - right));
        }
    }
    for (size_t li = 0; li < L; ++li) {
        auto compress = [&](const std::vector<std::pair<uint32_t, uint32_t>>& exprs, HFr* out) {
            HFr acc = HFr::zero();
            for (auto& e : exprs) {
                HFr v;
                if (!eval_expr_at(cs, e.first, e.second, fixed_ev, advice_ev, instance_ev, &v)) return false;
                acc = acc * theta + v;
            }
            *out = acc;
            return true;
        };
        HFr in_c, tab_c;
        if (!compress(cs.lookups[li].ins, &in_c) || !compress(cs.lookups[li].tabs, &tab_c)) return B200ZK_EINVAL;
        const LkEv& e = lk_ev[li];
        fold(l_0 * (one - e.z));
        fold(l_last * (e.z.sqr() - e.z));
        fold(l_active * (e.z_next * (e.a + beta) * (e.s + gamma) - e.z * (in_c + beta) * (tab_c + gamma)));
        fold(l_0 * (e.a - e.s));
        fold(l_active * ((e.a - e.s) * (e.a - e.a_prev)));
    }
    expected = expected * (xn - one).inv();

    // ---- queries, in upstream's order (prover and verifier must agree on it: it fixes the y / v powers).  The h
    // commitment is sum_i x^(n i) h_i: its query carries the marker H and is expanded into the h pieces below.
    const OpenBase H = {OpenBase::PROOF, UINT32_MAX};
    auto pt_of = [](uint32_t i) { return OpenBase{OpenBase::PROOF, i}; };
    std::vector<Query> Q;
    HFr x_next = rotate(x, 1), x_prev = rotate(x, -1), x_last = rotate(x, -(int)(bf + 1));
    int cid_pz = (int)A, cid_lk = cid_pz + (int)S, cid_fix = cid_lk + 3 * (int)L, cid_sig = cid_fix + (int)cs.F, cid_h = cid_sig + (int)P, cid_rand = cid_h + 1;
    for (size_t i = 0; i < naq; ++i) Q.push_back({cs.adv_q[2 * i], pt_of(advice_c[cs.adv_q[2 * i]]), rotate(x, cs.adv_q[2 * i + 1]), advice_ev[i]});
    for (size_t s = 0; s < S; ++s) {
        Q.push_back({cid_pz + (int)s, pt_of(perm_c[s]), x, perm_ev[s].z});
        Q.push_back({cid_pz + (int)s, pt_of(perm_c[s]), x_next, perm_ev[s].z_next});
    }
    for (size_t s = S > 0 ? S - 1 : 0; s-- > 0;) Q.push_back({cid_pz + (int)s, pt_of(perm_c[s]), x_last, perm_ev[s].z_last});
    for (size_t li = 0; li < L; ++li) {
        int b = cid_lk + 3 * (int)li;
        const LkEv& e = lk_ev[li];
        Q.push_back({b, pt_of(lk_z[li]), x, e.z});
        Q.push_back({b + 1, pt_of(lk_a[li]), x, e.a});
        Q.push_back({b + 2, pt_of(lk_s[li]), x, e.s});
        Q.push_back({b + 1, pt_of(lk_a[li]), x_prev, e.a_prev});
        Q.push_back({b, pt_of(lk_z[li]), x_next, e.z_next});
    }
    for (size_t i = 0; i < nfq; ++i) Q.push_back({cid_fix + cs.fix_q[2 * i], {OpenBase::FIXED, (uint32_t)cs.fix_q[2 * i]}, rotate(x, cs.fix_q[2 * i + 1]), fixed_ev[i]});
    for (size_t j = 0; j < P; ++j) Q.push_back({cid_sig + (int)j, {OpenBase::SIGMA, (uint32_t)j}, x, sigma_ev[j]});
    Q.push_back({cid_h, H, x, expected});
    Q.push_back({cid_rand, pt_of(random_c), x, random_ev});

    // ---- SHPLONK (shplonk/verifier.rs)
    HFr ch_y = rd.squeeze(), ch_v = rd.squeeze();
    uint32_t h1 = rd.read_point();
    HFr u = rd.squeeze();
    uint32_t h2 = rd.read_point();
    if (!rd.ok) return B200ZK_EVERIFY;
    // construct_intermediate_sets: commitments in first-seen order; rotation sets keyed by the point set
    std::vector<CommitSet> csets;
    std::vector<HFr> super_pts;
    auto has = [](const std::vector<HFr>& v, const HFr& p) { for (auto& e : v) if (e == p) return true; return false; };
    for (auto& qy : Q) {
        if (!has(super_pts, qy.pt)) super_pts.push_back(qy.pt);
        CommitSet* cset = nullptr;
        for (auto& c : csets) if (c.cid == qy.cid) { cset = &c; break; }
        if (!cset) { csets.push_back({qy.cid, qy.c, {}, {}}); cset = &csets.back(); }
        bool seen = false;
        for (size_t i = 0; i < cset->pts.size(); ++i) if (cset->pts[i] == qy.pt) { cset->evals[i] = qy.eval; seen = true; }
        if (!seen) { cset->pts.push_back(qy.pt); cset->evals.push_back(qy.eval); }
    }
    auto sort_pts = [](std::vector<HFr>& v) { std::sort(v.begin(), v.end(), [](const HFr& a, const HFr& b) { return cmp_canon(a, b) < 0; }); };
    sort_pts(super_pts);
    std::vector<RotSet> rsets;
    for (size_t ci = 0; ci < csets.size(); ++ci) {
        std::vector<HFr> pts = csets[ci].pts;
        sort_pts(pts);
        RotSet* rs = nullptr;
        for (auto& r : rsets) if (r.pts.size() == pts.size() && std::equal(pts.begin(), pts.end(), r.pts.begin())) { rs = &r; break; }
        if (!rs) { rsets.push_back({pts, {}}); rs = &rsets.back(); }
        rs->members.push_back(ci);
    }
    auto vanish = [&](const std::vector<HFr>& roots, const std::vector<HFr>* except) {
        HFr acc = HFr::one();
        for (auto& r : roots) if (!except || !has(*except, r)) acc = acc * (u - r);
        return acc;
    };
    // L = sum_i v^i z_i sum_j y^j (C_ij - [r_ij(u)] G) - Z_T(u) h1;  the opening is (h2, u h2 + L / z_0)
    HFr z0 = vanish(super_pts, rsets.empty() ? nullptr : &rsets[0].pts);
    if (rsets.empty() || z0.is_zero()) return B200ZK_EVERIFY;
    const HFr z0_inv = z0.inv();
    out->points = std::move(rd.pts);
    out->h2 = h2;
    out->right.clear();
    out->right.push_back({pt_of(h2), u});
    HFr g_scalar = HFr::zero(), v_pow = HFr::one();
    for (size_t ri = 0; ri < rsets.size(); ++ri) {
        const RotSet& rs = rsets[ri];
        HFr y_pow = HFr::one(), zv = vanish(super_pts, &rs.pts) * v_pow;
        for (size_t ci : rs.members) {
            const CommitSet& c = csets[ci];
            std::vector<HFr> ev(rs.pts.size());
            for (size_t i = 0; i < rs.pts.size(); ++i)
                for (size_t j = 0; j < c.pts.size(); ++j) if (c.pts[j] == rs.pts[i]) ev[i] = c.evals[j];
            std::vector<HFr> low = interpolate(rs.pts, ev);
            HFr r_eval = HFr::zero();
            for (size_t i = low.size(); i-- > 0;) r_eval = r_eval * u + low[i];
            HFr sc = zv * y_pow;
            if (c.c.kind == H.kind && c.c.idx == H.idx) {
                HFr w = sc * z0_inv;
                for (size_t i = 0; i < q; ++i) { out->right.push_back({pt_of(h_c[i]), w}); w = w * xn; }
            } else {
                out->right.push_back({c.c, sc * z0_inv});
            }
            g_scalar = g_scalar - sc * r_eval;
            y_pow = y_pow * ch_y;
        }
        v_pow = v_pow * ch_v;
    }
    out->right.push_back({{OpenBase::GEN, 0}, g_scalar * z0_inv});
    out->right.push_back({pt_of(h1), vanish(super_pts, nullptr).neg() * z0_inv});
    return B200ZK_OK;
}

}  // namespace b200zk

extern "C" {

int32_t b200zk_verify_proof(const uint32_t* cs_blob, size_t blob_words, const void* fixed_commitments,
                            const void* sigma_commitments, const void* g1_generator, const void* g2, const void* s_g2,
                            const void* const* instance_columns, const uint32_t* instance_lens, const void* transcript_repr,
                            const uint8_t* proof, size_t proof_len) {
    CsDesc cs;
    if (!cs_blob || !parse_cs(cs_blob, blob_words, cs)) return B200ZK_EINVAL;
    if (!g1_generator || !g2 || !s_g2 || !transcript_repr || (!proof && proof_len)) return B200ZK_EINVAL;
    if ((cs.F && !fixed_commitments) || (!cs.perm.empty() && !sigma_commitments)) return B200ZK_EINVAL;
    if (cs.I && (!instance_columns || !instance_lens)) return B200ZK_EINVAL;
    if (cs.k < 1 || cs.k > FR_TWO_ADICITY) return B200ZK_EINVAL;
    const VkPoints vk = {fixed_commitments, sigma_commitments, g1_generator};
    Opening op;
    int32_t rc = replay_proof(cs, vk, instance_columns, instance_lens, transcript_repr, proof, proof_len, nullptr, &op);
    if (rc != B200ZK_OK) return rc;
    // accept iff e(h2, [s]_2) = e(right, [1]_2)
    HXyzz rhs = hx_identity();
    for (const OpenTerm& t : op.right) rhs = hx_add(rhs, g1_mul(open_base_point(vk, op.points.data(), t.base), t.scalar));
    HAffine rhs_a = hx_to_affine(rhs);
    HAffine ps[2] = {op.points[op.h2], {rhs_a.x, rhs_a.y.neg()}};
    if (rhs_a.x.is_zero() && rhs_a.y.is_zero()) ps[1] = rhs_a;
    G2A qs[2] = {g2_from_limbs(s_g2), g2_from_limbs(g2)};
    if (!g2_on_curve(qs[0]) || !g2_on_curve(qs[1]) || g2_is_identity(qs[0]) || g2_is_identity(qs[1])) return B200ZK_EINVAL;
    return pairing_product_is_one(ps, qs, 2) ? B200ZK_OK : B200ZK_EVERIFY;
}

}  // extern "C"
