// TEST AID for tests/test_quotient_classes.py: the quotient planner (quot_plan.hpp) and the class programs
// (expr_share.hpp) on a constraint-system blob, and coset_interpolate_row's linear-class summand, compiled with a
// host compiler like tests/emu/emu_harness.cpp.  Never linked into the product library.
#include <algorithm>
#include <vector>
#include "../halo2-experiments_b200/csrc/field.cuh"
#include "../halo2-experiments_b200/csrc/prover_kernels.cuh"
#include "../halo2-experiments_b200/csrc/cs_desc.hpp"
#include "../halo2-experiments_b200/csrc/expr_share.hpp"
#include "../halo2-experiments_b200/csrc/quot_plan.hpp"

using namespace b200zk;

extern "C" {

// q = degree - 1 as the prover's domain has it.  out: q, lookup cosets, low, multiplications per row of the main / low /
// linear gate programs (as the prover compiles them), then the class of every gate and the cosets of every advice and
// instance column.  Returns the number of words, 0 for a malformed blob.
size_t quot_plan_words(const uint32_t* blob, size_t nw, uint32_t* out, size_t cap) {
    CsDesc cs;
    if (!parse_cs(blob, nw, cs)) return 0;
    const uint32_t q = cs.degree - 1, CL = lookup_cosets(cs, q);
    QuotPlan p = quot_plan(cs, q, CL);
    std::vector<uint32_t> o{q, CL, p.low};
    for (uint32_t cls = 0; cls < 3; ++cls) {
        std::vector<ExFold> items;
        for (size_t i = 0; i < cs.gates.size(); ++i)
            if (p.gate_class[i] == cls) items.push_back({cs.gates[i].first, cs.gates[i].second, EX_WSUM | ((EXW_ACC0 | (uint32_t)i) << 8)});
        std::vector<uint32_t> prog;
        if (!ex_share_common(cs.prog, items, prog, true)) return 0;
        o.push_back(ex_program_muls(prog.data(), prog.size()));
    }
    o.insert(o.end(), p.gate_class.begin(), p.gate_class.end());
    o.insert(o.end(), p.adv_need.begin(), p.adv_need.end());
    o.insert(o.end(), p.inst_need.begin(), p.inst_need.end());
    if (o.size() > cap) return 0;
    std::copy(o.begin(), o.end(), out);
    return o.size();
}

void coset_interpolate_lin(const fe_t* g, const fe_t* inv_pow, const fe_t* vinv, uint32_t C, size_t n, fe_t* out, const fe_t* lin) {
    for (size_t r = 0; r < n; ++r) coset_interpolate_row(g, inv_pow, vinv, C, n, out, r, nullptr, lin);
}

}  // extern "C"
