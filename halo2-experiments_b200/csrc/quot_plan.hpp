// Host-side planner of the quotient evaluation (evaluate_h): on how many cosets each gate polynomial is
// evaluated and each advice / instance column is extended (pure C++, no CUDA types).
//
// A term of degree d of the numerator of h = (sum_i y^i g_i) / Z_H contributes a polynomial of degree
// < (d - 1) n to h, so d - 1 cosets of size n determine it.  Three classes, their sizes in cosets:
//   main (q)    gates with d - 1 above `low`, and the permutation terms: evaluated into h on all q cosets
//   low         gates with 1 < d - 1 <= low (and below 2^QUOT_LINEAR_MIN_K rows those with d <= 2): evaluated with the lookup terms into their accumulator h_lk,
//               carried to the other cosets after the per-coset iNTT (lookup_extrapolate_row).  `low` is
//               the lookups' coset count.  low == q: no such class (the gates stay in main).  Without lookups
//               there is none either: an accumulator of its own costs `low` iNTTs and the extrapolation, more
//               than the gates save (Merkle v3, 5 gates of degree <= 4: 2 x 13 multiplications per row saved
//               against ~3 log2(n) / 2 + 9 spent; measured 6.18 -> 6.34 ms at k = 14)
//   linear (1)  gates with d <= 2 from 2^QUOT_LINEAR_MIN_K rows on: evaluated on coset 0 only; their part of
//               h has degree < n and goes to piece 0 after an iNTT of its own.  Below that size the gates
//               join the low class (or main): the extra launches cost more than the rows they save
//               (Merkle v3, k = 14: 6.15 -> 6.20 ms with the class, 3 launches more)
// Each gate keeps its power of y in evaluate_h wherever it runs (see ExprArgs::wts).
#pragma once
#include <algorithm>
#include <cstdint>
#include <vector>
#include "cs_desc.hpp"

namespace b200zk {

enum : uint32_t { QC_MAIN = 0, QC_LOW = 1, QC_LINEAR = 2 };
// The linear class saves (q - 1) n rows of its gates for one size-n iNTT and three launches (≈ 30 us on a B200):
// with the 60 multiplications per row it saves in the Merkle circuits (≈ 0.9 ns per row at the IMAD rate), that is
// worth it from n ≈ 2^15 on.
static constexpr uint32_t QUOT_LINEAR_MIN_K = 16;

struct QuotPlan {
    uint32_t q = 0, low = 0;
    std::vector<uint32_t> gate_class;               // per gate polynomial
    std::vector<uint32_t> adv_need, inst_need;      // cosets the quotient reads of each advice / instance column
    uint32_t cosets(uint32_t cls) const { return cls == QC_MAIN ? q : cls == QC_LOW ? low : 1; }
};

// cosets the lookup terms need: their degree is < (2 + deg input + deg table) * n  (circuit.rs, lookup
// Argument::required_degree; the max(4, .) floor does not matter, it is >= 4 already); q without lookups
inline uint32_t lookup_cosets(const CsDesc& cs, uint32_t q) {
    if (cs.lookups.empty()) return q;
    uint32_t need = 0;
    for (auto& lk : cs.lookups) {
        uint32_t di = 1, dt = 1;
        for (auto& e : lk.ins) di = std::max(di, expr_degree(cs, e.first, e.second));
        for (auto& e : lk.tabs) dt = std::max(dt, expr_degree(cs, e.first, e.second));
        need = std::max(need, 2 + di + dt);
    }
    return std::min(q, need);
}

// advice / instance columns an expression reads (query indices resolved to columns)
inline void expr_columns(const CsDesc& cs, uint32_t off, uint32_t len, std::vector<uint32_t>& adv, std::vector<uint32_t>& inst, uint32_t cosets) {
    for (uint32_t i = off; i < off + len; ++i) {
        uint32_t op = cs.prog[i] & 0xff, arg = cs.prog[i] >> 8;
        if (op == EX_ADVICE) { uint32_t c = (uint32_t)cs.adv_q[2 * arg]; adv[c] = std::max(adv[c], cosets); }
        else if (op == EX_INSTANCE) { uint32_t c = (uint32_t)cs.inst_q[2 * arg]; inst[c] = std::max(inst[c], cosets); }
    }
}

// q: cosets of the quotient (degree - 1); CL: cosets of the lookup terms (lookup_cosets)
inline QuotPlan quot_plan(const CsDesc& cs, uint32_t q, uint32_t CL) {
    QuotPlan p;
    p.q = q;
    std::vector<uint32_t> deg;
    for (auto& g : cs.gates) deg.push_back(expr_degree(cs, g.first, g.second));
    p.low = CL;                                     // == q without lookups
    const bool linear = cs.k >= QUOT_LINEAR_MIN_K;
    for (uint32_t d : deg)
        p.gate_class.push_back(d <= 2 && linear ? QC_LINEAR : (d <= 2 || d - 1 <= p.low) && p.low < q ? QC_LOW : QC_MAIN);
    p.adv_need.assign(cs.A, 0);
    p.inst_need.assign(cs.I, 0);
    for (size_t i = 0; i < cs.gates.size(); ++i)
        expr_columns(cs, cs.gates[i].first, cs.gates[i].second, p.adv_need, p.inst_need, p.cosets(p.gate_class[i]));
    for (auto& lk : cs.lookups) {
        for (auto& e : lk.ins) expr_columns(cs, e.first, e.second, p.adv_need, p.inst_need, CL);
        for (auto& e : lk.tabs) expr_columns(cs, e.first, e.second, p.adv_need, p.inst_need, CL);
    }
    for (auto& pc : cs.perm) {
        if (pc.first == 0 && pc.second < cs.A) p.adv_need[pc.second] = q;
        else if (pc.first == 2 && pc.second < cs.I) p.inst_need[pc.second] = q;
    }
    return p;
}

}  // namespace b200zk
