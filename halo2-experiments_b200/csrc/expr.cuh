// Row-wise expression evaluation: the device counterpart of halo2_proofs v2023_02_02
// plonk/evaluation.rs (`GraphEvaluator::evaluate`, `evaluate`) — reached from create_proof at
// /root/reference/src/circuits/utils.rs:40-48.  One thread evaluates the whole program for one
// row of the (extended or Lagrange) domain, so every column element is read once and all
// intermediates stay on chip.
//
// The program is the constraint system's expressions in postfix order over a small value
// stack, plus instructions that accumulate them:
//   custom gates : every gate polynomial followed by WSUM:  acc0 <- acc0 + pop() * w[i], where
//                  w[i] = y^e_i is gate i's power of y in evaluate_h (uploaded per proof, see
//                  quot_plan.hpp) — one multiplication per gate, as upstream's Horner fold in y,
//                  but independent of which other gates the program holds, so that gates of
//                  different degree can run as separate programs on different numbers of cosets
//   lookups      : input expressions with FOLD(acc0, theta), table expressions with FOLD(acc1, theta)
//                  (FOLD is the Horner step acc <- acc * factor + pop())
// Like upstream's GraphEvaluator (which interns every Calculation once), repeated sub-expressions
// are evaluated once per row: the host (ex_share_common in expr_share.hpp) hash-conses the expression
// trees, and a shared node is computed at its first use, kept with TEE(slot) and re-read with
// TMP(slot).  In the Merkle Sum Tree circuit the five (state + rc)^5 terms of Pow5Chip's
// "full round" gate appear in five polynomials each, and the compressed-selector products
// q(1-q)(2-q).. in every polynomial they gate: 281 -> ~150 multiplications per row.
// Consecutive gate polynomials with a common factor (every constraint of a gate is
// selector * poly) are accumulated as  acc0 <- acc0 + s * (p_0 w_0 + ... + p_(m-1) w_(m-1)):  the inner
// sum runs in acc1 (WSUM into acc1), GROUP multiplies it by the factor once — m - 1
// multiplications less than accumulating s * p_i one by one.
// Upstream orders the same arithmetic differently; the value per row is the same field element,
// hence bit-exact.
#pragma once
#include "field.cuh"

namespace b200zk {

enum : uint32_t { EX_CONST = 0, EX_FIXED = 1, EX_ADVICE = 2, EX_INSTANCE = 3, EX_NEG = 4, EX_ADD = 5, EX_MUL = 6, EX_SCALE = 7, EX_FOLD = 8, EX_TEE = 9, EX_TMP = 10, EX_WSUM = 11, EX_GROUP = 12 };
// WSUM argument: weight index | target (acc0 += v w, acc1 += v w, acc1 = v w)
enum : uint32_t { EXW_ACC0 = 0u << 20, EXW_ACC1 = 1u << 20, EXW_SET1 = 2u << 20, EXW_INDEX = (1u << 20) - 1 };
enum : uint32_t { EXF_THETA = 0, EXF_BETA = 1, EXF_GAMMA = 2, EXF_Y = 3 };
// output modes
enum : uint32_t {
    EXM_ACC0 = 0,        // out0[idx] = acc0                                  (custom gates: h)
    EXM_ACC01 = 1,       // out0[idx] = acc0, out1[idx] = acc1                (lookup compressed input / table)
    EXM_LOOKUP_PROD = 2  // out0[idx] = (acc0 + beta) * (acc1 + gamma)        (lookup "table_value" in evaluate_h)
};

static constexpr int EX_STACK = 16;
static constexpr int EX_TMPS = 24;          // shared sub-expression slots per row

struct ExprArgs {
    const uint32_t* prog;
    uint32_t prog_len;
    const fe_t* consts;                 // Montgomery form
    const fe_t* const* fixed;           // device arrays of column base pointers
    const fe_t* const* advice;
    const fe_t* const* instance;
    const int32_t* q_fixed;             // (column, rotation) pairs
    const int32_t* q_advice;
    const int32_t* q_instance;
    uint32_t log_size;                  // rotations wrap inside blocks of 2^log_size rows (= n: one coset / the Lagrange domain)
    uint32_t rows;                      // rows evaluated: n, or C * n on the quotient cosets
    uint32_t row0;                      // first row (a rank of a sharded proof evaluates its own cosets only)
    uint32_t rot_scale;                 // 1
    fe_t factors[4];                    // theta, beta, gamma, y
    const fe_t* wts;                    // per-gate weights y^e_i of WSUM (gate programs only)
    uint32_t mode;
    fe_t* out0;
    fe_t* out1;
};

ZK_D fe_t expr_load(const fe_t* const* cols, const int32_t* q, uint32_t qi, uint32_t idx, const ExprArgs& a) {
    int32_t col = q[2 * qi], rot = q[2 * qi + 1];
    uint32_t mask = (1u << a.log_size) - 1;
    uint32_t r = (idx & ~mask) | ((idx + (uint32_t)(rot * (int32_t)a.rot_scale)) & mask);   // rem_euclid inside the coset
    return cols[col][r];
}

ZK_D void expr_eval_row(const ExprArgs& a, uint32_t idx) {
    fe_t stk[EX_STACK];
    fe_t tmp[EX_TMPS];
    int sp = 0;
    fe_t acc0 = Fr::zero(), acc1 = Fr::zero();
    for (uint32_t pc = 0; pc < a.prog_len; ++pc) {
        uint32_t w = a.prog[pc], op = w & 0xff, arg = w >> 8;
        switch (op) {
            case EX_CONST: stk[sp++] = a.consts[arg]; break;
            case EX_FIXED: stk[sp++] = expr_load(a.fixed, a.q_fixed, arg, idx, a); break;
            case EX_ADVICE: stk[sp++] = expr_load(a.advice, a.q_advice, arg, idx, a); break;
            case EX_INSTANCE: stk[sp++] = expr_load(a.instance, a.q_instance, arg, idx, a); break;
            case EX_NEG: stk[sp - 1] = Fr::neg(stk[sp - 1]); break;
            case EX_ADD: stk[sp - 2] = Fr::add(stk[sp - 2], stk[sp - 1]); --sp; break;
            case EX_MUL: stk[sp - 2] = Fr::mul(stk[sp - 2], stk[sp - 1]); --sp; break;
            case EX_SCALE: stk[sp - 1] = Fr::mul(stk[sp - 1], a.consts[arg]); break;
            case EX_FOLD: {
                fe_t v = stk[--sp];
                const fe_t f = a.factors[arg & 0xf];
                if ((arg >> 4) == 0) acc0 = Fr::add(Fr::mul(acc0, f), v);
                else acc1 = Fr::add(Fr::mul(acc1, f), v);
                break;
            }
            case EX_WSUM: {
                fe_t v = Fr::mul(stk[--sp], a.wts[arg & EXW_INDEX]);
                const uint32_t to = arg & ~EXW_INDEX;
                if (to == EXW_ACC0) acc0 = Fr::add(acc0, v);
                else if (to == EXW_ACC1) acc1 = Fr::add(acc1, v);
                else acc1 = v;
                break;
            }
            case EX_GROUP: acc0 = Fr::add(acc0, Fr::mul(stk[--sp], acc1)); break;
            case EX_TEE: tmp[arg] = stk[sp - 1]; break;
            case EX_TMP: stk[sp++] = tmp[arg]; break;
            default: break;
        }
    }
    if (a.mode == EXM_ACC0) {
        a.out0[idx] = acc0;
    } else if (a.mode == EXM_ACC01) {
        a.out0[idx] = acc0; a.out1[idx] = acc1;
    } else {
        a.out0[idx] = Fr::mul(Fr::add(acc0, a.factors[EXF_BETA]), Fr::add(acc1, a.factors[EXF_GAMMA]));
    }
}

}  // namespace b200zk
