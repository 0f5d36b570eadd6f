// Host-side compiler of evaluator programs (expr.cuh): pure C++, shared by the prover and the host tests.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <map>
#include <vector>
#include "expr.cuh"

namespace b200zk {

// One evaluator program = a list of expressions (postfix ranges of cs.prog), each followed by a
// FOLD or WSUM word.  The trees are hash-consed (ADD / MUL operands unordered); a node that the emission
// reaches more than once and that contains at least one multiplication is computed once and kept
// in a TEE/TMP slot (expr.cuh).  When more than EX_TMPS nodes qualify, those saving the most
// multiplications win.
struct ExFold { uint32_t off, len, fold_word; };

inline bool ex_share_common(const std::vector<uint32_t>& src, const std::vector<ExFold>& items, std::vector<uint32_t>& out,
                            bool group_common_factor = false) {
    struct Node { uint32_t op, arg; int l, r; uint32_t muls; };
    std::vector<Node> nodes;
    std::map<std::array<int64_t, 4>, int> intern;
    auto make = [&](uint32_t op, uint32_t arg, int l, int r) {
        int a = l, b = r;
        if ((op == EX_ADD || op == EX_MUL) && a > b) std::swap(a, b);
        std::array<int64_t, 4> key{(int64_t)op, (int64_t)arg, a, b};
        auto it = intern.find(key);
        if (it != intern.end()) return it->second;
        uint32_t muls = (op == EX_MUL || op == EX_SCALE ? 1u : 0u) + (l >= 0 ? nodes[l].muls : 0u) + (r >= 0 ? nodes[r].muls : 0u);
        nodes.push_back({op, arg, l, r, muls});
        intern[key] = (int)nodes.size() - 1;
        return (int)nodes.size() - 1;
    };
    std::vector<int> roots;
    for (auto& it : items) {
        std::vector<int> st;
        for (uint32_t i = it.off; i < it.off + it.len; ++i) {
            uint32_t op = src[i] & 0xff, arg = src[i] >> 8;
            if (op <= EX_INSTANCE) st.push_back(make(op, arg, -1, -1));
            else if (op == EX_NEG || op == EX_SCALE) { if (st.empty()) return false; st.back() = make(op, arg, st.back(), -1); }
            else if (op == EX_ADD || op == EX_MUL) {
                if (st.size() < 2) return false;
                int r = st.back(); st.pop_back();
                st.back() = make(op, 0, st.back(), r);
            } else return false;
        }
        if (st.size() != 1) return false;
        roots.push_back(st[0]);
    }
    // how often the emission asks for each node when shared nodes are expanded once
    std::vector<uint32_t> req(nodes.size(), 0);
    std::vector<int> work;
    for (int root : roots) {
        work.push_back(root);
        while (!work.empty()) {
            int id = work.back(); work.pop_back();
            if (++req[id] == 1) { if (nodes[id].l >= 0) work.push_back(nodes[id].l); if (nodes[id].r >= 0) work.push_back(nodes[id].r); }
        }
    }
    std::vector<int> cand;
    for (size_t id = 0; id < nodes.size(); ++id) if (req[id] >= 2 && nodes[id].muls >= 1) cand.push_back((int)id);
    std::sort(cand.begin(), cand.end(), [&](int a, int b) {
        uint64_t sa = (uint64_t)(req[a] - 1) * nodes[a].muls, sb = (uint64_t)(req[b] - 1) * nodes[b].muls;
        return sa != sb ? sa > sb : a < b;
    });
    if (cand.size() > (size_t)EX_TMPS) cand.resize(EX_TMPS);
    std::vector<int> slot(nodes.size(), -1);
    for (size_t i = 0; i < cand.size(); ++i) slot[cand[i]] = (int)i;
    std::vector<char> done(nodes.size(), 0);
    // iterative postfix emission: (node, phase)
    auto emit = [&](int root) {
        std::vector<std::pair<int, int>> stk{{root, 0}};
        while (!stk.empty()) {
            auto [id, phase] = stk.back(); stk.pop_back();
            const Node& nd = nodes[id];
            if (phase == 0) {
                if (slot[id] >= 0 && done[id]) { out.push_back(EX_TMP | ((uint32_t)slot[id] << 8)); continue; }
                stk.push_back({id, 1});
                if (nd.r >= 0) stk.push_back({nd.r, 0});
                if (nd.l >= 0) stk.push_back({nd.l, 0});
            } else {
                out.push_back(nd.op | (nd.arg << 8));
                if (slot[id] >= 0) { out.push_back(EX_TEE | ((uint32_t)slot[id] << 8)); done[id] = 1; }
            }
        }
    };
    // common factor of two product roots (-1 if none)
    auto common = [&](int a, int b) {
        if (nodes[a].op != EX_MUL || nodes[b].op != EX_MUL) return -1;
        for (int x : {nodes[a].l, nodes[a].r}) if (x == nodes[b].l || x == nodes[b].r) return x;
        return -1;
    };
    for (size_t k = 0; k < roots.size();) {
        size_t m = 1;
        int f = -1;
        if (group_common_factor && k + 1 < roots.size()) {
            f = common(roots[k], roots[k + 1]);
            if (f >= 0) {
                m = 2;
                while (k + m < roots.size() && nodes[roots[k + m]].op == EX_MUL &&
                       (nodes[roots[k + m]].l == f || nodes[roots[k + m]].r == f)) ++m;
            }
        }
        if (f < 0) {
            emit(roots[k]);
            out.push_back(items[k].fold_word);
            ++k;
            continue;
        }
        for (size_t j = 0; j < m; ++j) {                        // weighted cofactors into acc1
            const Node& nd = nodes[roots[k + j]];
            emit(nd.l == f ? nd.r : nd.l);
            out.push_back(EX_WSUM | (((items[k + j].fold_word >> 8 & EXW_INDEX) | (j == 0 ? EXW_SET1 : EXW_ACC1)) << 8));
        }
        emit(f);
        out.push_back(EX_GROUP);
        k += m;
    }
    return true;
}

// Field multiplications one row of a program executes.
inline uint32_t ex_program_muls(const uint32_t* prog, size_t len) {
    uint32_t m = 0;
    for (size_t i = 0; i < len; ++i) {
        uint32_t op = prog[i] & 0xff;
        if (op == EX_MUL || op == EX_SCALE || op == EX_FOLD || op == EX_WSUM || op == EX_GROUP) m += 1;
    }
    return m;
}

}  // namespace b200zk
