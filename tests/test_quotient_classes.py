"""Degree-aware quotient (csrc/quot_plan.hpp): which gate polynomials run on how many cosets, which cosets of each
column are extended, and that evaluating the classes on their own cosets gives the same h as evaluating everything
on all q cosets."""
import ctypes
import hashlib
import importlib
import os
import random
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import pyref as P

_HARNESS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "quot_plan_harness.cpp")


@pytest.fixture(scope="module")
def harness():
    """tests/quot_plan_harness.cpp built with the host compiler into a temporary directory (the tree may be read-only)."""
    csrc = os.path.join(os.path.dirname(_HARNESS), "..", "halo2-experiments_b200", "csrc")
    h = hashlib.sha256()
    for f in [_HARNESS] + sorted(os.path.join(csrc, x) for x in os.listdir(csrc) if x.endswith((".cuh", ".hpp"))):
        h.update(open(f, "rb").read())
    so = os.path.join(tempfile.gettempdir(), f"quot_plan_harness_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = so + f".{os.getpid()}"
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-w", "-x", "c++", "-o", tmp, _HARNESS])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    lib.quot_plan_words.restype = ctypes.c_size_t
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def quot_plan(lib, blob):
    """quot_plan.hpp on a constraint-system blob: dict(q, lookup_cosets, low, muls (main, low, linear per row),
    gate_class (0 main, 1 low, 2 linear), adv_need, inst_need)."""
    blob = np.ascontiguousarray(blob, dtype=np.uint32)
    out = np.zeros(6 + len(blob), dtype=np.uint32)
    ln = lib.quot_plan_words(_p(blob), ctypes.c_size_t(len(blob)), _p(out), ctypes.c_size_t(len(out)))
    assert ln, "malformed blob"
    G, A, I = int(blob[9]), int(blob[3]), int(blob[5])
    v = [int(x) for x in out[:ln]]
    return {"q": v[0], "lookup_cosets": v[1], "low": v[2], "muls": tuple(v[3:6]), "gate_class": v[6:6 + G],
            "adv_need": v[6 + G:6 + G + A], "inst_need": v[6 + G + A:6 + G + A + I]}


@pytest.fixture(scope="module")
def fe(zk):
    return importlib.import_module(zk.__name__ + ".frontend")


@pytest.fixture(scope="module")
def chips(zk):
    return importlib.import_module(zk.__name__ + ".chips")


@pytest.fixture(scope="module")
def synth(zk):
    return importlib.import_module(zk.__name__ + ".circuits_synth")


def _columns(cs, e, out):
    """(kind, column) of every advice / instance query an expression reads."""
    if e.kind == "advice":
        out.add(("advice", cs.advice_queries[e.a][0]))
    elif e.kind == "instance":
        out.add(("instance", cs.instance_queries[e.a][0]))
    elif e.kind in ("neg", "scaled"):
        _columns(cs, e.a, out)
    elif e.kind in ("sum", "prod"):
        _columns(cs, e.a, out); _columns(cs, e.b, out)
    return out


LINEAR_MIN_K = 16                                       # quot_plan.hpp QUOT_LINEAR_MIN_K


def _restated_plan(cs, k):
    q = cs.degree() - 1
    CL = min(q, max(2 + max([1] + [e.degree() for e in ins]) + max([1] + [e.degree() for e in tabs]) for ins, tabs in cs.lookups)) if cs.lookups else q
    degs = [g.degree() for g in cs.gates]
    low = CL if cs.lookups else q
    cls = [2 if d <= 2 and k >= LINEAR_MIN_K else 1 if ((d <= 2 or d - 1 <= low) and low < q) else 0 for d in degs]
    size = {0: q, 1: low, 2: 1}
    need = {("advice", c): 0 for c in range(cs.num_advice)}
    need.update({("instance", c): 0 for c in range(cs.num_instance)})

    def bump(cols, v):
        for c in cols:
            need[c] = max(need[c], v)
    for g, c in zip(cs.gates, cls):
        bump(_columns(cs, g, set()), size[c])
    for ins, tabs in cs.lookups:
        for e in ins + tabs:
            bump(_columns(cs, e, set()), CL)
    for t, c in cs.permutation:
        if t != 1:
            need[({0: "advice", 2: "instance"}[t], c)] = q
    return {"q": q, "lookup_cosets": CL, "low": low, "gate_class": cls,
            "adv_need": [need[("advice", c)] for c in range(cs.num_advice)],
            "inst_need": [need[("instance", c)] for c in range(cs.num_instance)]}


def _jobs(name, chips, fe, synth):
    if name == "mst":
        return chips.merkle_sum_tree_job(10)
    if name == "merkle_v3":
        return chips.merkle_v3_job(10)
    if name == "less_than":
        return fe.synthesize_job(chips.LessThanCircuit(755), 10, [list(range(800))])
    if name == "safe_accumulator":
        return fe.synthesize_job(chips.SafeAccumulatorCircuit([4], [0, 0, 14, 13]), 8, [[0, 0, 15, 1]])
    fn, k = name.split(":")
    return getattr(synth, fn)(int(k))


@pytest.mark.parametrize("name", ["mst", "merkle_v3", "less_than", "safe_accumulator", "generic_shapes:6", "generic_shapes:10",
                                  "small:5", "mst_shaped:9", "v3_shaped:6"])
@pytest.mark.parametrize("k", [None, 20])
def test_plan_matches_restatement(harness, chips, fe, synth, name, k):
    """At the job's own size and, with the same constraint system, at k = 20 (where the linear class exists)."""
    job = _jobs(name, chips, fe, synth)
    k = job.k if k is None else k
    got = quot_plan(harness, job.cs.to_blob(k))
    want = _restated_plan(job.cs, k)
    assert {key: got[key] for key in want} == want
    if name == "safe_accumulator":
        assert got["q"] == 16


def test_mst_plan(harness, chips):
    """The headline circuit at k = 20: 7 gate polynomials of degree 6 on 5 cosets, 12 of degree 3..5 on the lookups' 4,
    the 4 degree-2 partial-round gates on 1; advice columns 0-10 and the instance column on 5 cosets, 11-19 on 4.
    Below 2^16 rows the degree-2 gates run with the low class."""
    cs = chips.merkle_sum_tree_job(10).cs
    p = quot_plan(harness, cs.to_blob(20))
    assert (p["q"], p["low"]) == (5, 4)
    assert [p["gate_class"].count(c) for c in range(3)] == [7, 12, 4]
    assert p["adv_need"] == [5] * 11 + [4] * 9 and p["inst_need"] == [5]
    assert sum(p["adv_need"]) + sum(p["inst_need"]) == 96
    small = quot_plan(harness, cs.to_blob(10))
    assert [small["gate_class"].count(c) for c in range(3)] == [7, 16, 0]


# ---- the class split in a small prime field: p = 12289 = 3 * 2^12 + 1, generator 11
PR, GEN = 12289, 11


def _poly_eval(c, x):
    acc = 0
    for v in reversed(c):
        acc = (acc * x + v) % PR
    return acc


def _intt(vals, w):
    n = len(vals)
    wi, ni = pow(w, PR - 2, PR), pow(n, PR - 2, PR)
    return [sum(v * pow(wi, i * r, PR) for i, v in enumerate(vals)) * ni % PR for r in range(n)]


@pytest.mark.parametrize("q,CL,L,S,seed", [(5, 4, 2, 2, 1), (5, 4, 1, 1, 2), (7, 4, 1, 0, 3), (4, 3, 2, 2, 4), (5, 5, 0, 2, 5)])
def test_class_split_gives_the_same_h(q, CL, L, S, seed):
    """Gates of every degree, permutation terms and lookup terms folded in y in halo2's order give h = N / Z_H; the same
    h from: main gates + permutation on q cosets (weights y^(G-1-i), Horner in y through the permutation terms, y^(5L)
    in the iNTT), low gates + lookups on CL cosets (weights y^(G-1-i+2S+1), y^5 per lookup) extrapolated to the other
    cosets in H-space, linear gates on coset 0 (weights y^(G-1-i+2S+1+5L)) added to piece 0."""
    rnd = random.Random(seed)
    n, ext = 8, 8                                        # extended domain of ext * n points: cosets c_j = zeta * w_ext^j
    w = pow(GEN, (PR - 1) // n, PR)
    w_ext = pow(GEN, (PR - 1) // (n * ext), PR)
    cj = [GEN * pow(w_ext, j, PR) % PR for j in range(q)]
    yj = [pow(c, n, PR) for c in cj]
    zh = lambda x: (pow(x, n, PR) - 1) % PR
    y = rnd.randrange(2, PR)
    low = CL if L else q
    # random quotient parts t of degree < (d - 1) n - d + 1 (numerator t Z_H of degree <= d (n - 1)), gates of degree 2..q+1
    rand_t = lambda d: [rnd.randrange(PR) for _ in range(d * (n - 1) - n + 1)]
    degs = [rnd.randrange(2, q + 2) for _ in range(9)] + [2, q + 1, low + 1]
    gates = [rand_t(d) for d in degs]
    perm = [rand_t(q + 1) for _ in range(2 * S + 1 if S else 0)]
    lks = [[rand_t(CL + 1) for _ in range(5)] for _ in range(L)]
    G, PT = len(gates), len(perm)
    # reference: Horner in y over all terms, in halo2's order
    terms = gates + perm + [t for lk in lks for t in lk]
    h = [0] * (q * n)
    for t in terms:
        h = [v * y % PR for v in h]
        for i, v in enumerate(t):
            h[i] = (h[i] + v) % PR
    want = [h[t * n:(t + 1) * n] for t in range(q)]
    # split: numerator values on coset rows, as the kernels see them
    num = lambda t, x: _poly_eval(t, x) * zh(x) % PR
    rows = lambda j: [cj[j] * pow(w, i, PR) % PR for i in range(n)]
    cls = [2 if d <= 2 else 1 if d - 1 <= low and low < q else 0 for d in degs]
    yp = lambda e: pow(y, e, PR)
    # main class + permutation on all q cosets, y^(5L) in the per-coset iNTT post factor
    g = []
    for j in range(q):
        vals = []
        for x in rows(j):
            acc = sum(yp(G - 1 - i) * num(gates[i], x) for i in range(G) if cls[i] == 0) % PR
            for t in perm:
                acc = (acc * y + num(t, x)) % PR
            vals.append(acc * yp(5 * L) * pow(zh(x), PR - 2, PR) % PR)
        g.append(_intt(vals, w))
    # low class + lookups on the first `low` cosets, extrapolated to the others (lookup_extrapolate_row)
    Hlow = []
    for j in range(low):
        vals = []
        for x in rows(j):
            acc = sum(yp(G - 1 - i + PT) * num(gates[i], x) for i in range(G) if cls[i] == 1) % PR
            for lk in lks:
                acc = (acc * yp(5) + sum(yp(4 - m) * num(t, x) for m, t in enumerate(lk))) % PR
            vals.append(acc * pow(zh(x), PR - 2, PR) % PR)
        b = _intt(vals, w)
        Hlow.append([b[r] * pow(cj[j], (PR - 1 - r) % (PR - 1), PR) % PR for r in range(n)])
    for jp in range(low, q):
        lam = []
        for j in range(low):
            nu = de = 1
            for m in range(low):
                if m != j:
                    nu = nu * (yj[jp] - yj[m]) % PR; de = de * (yj[j] - yj[m]) % PR
            lam.append(nu * pow(de, PR - 2, PR) % PR)
        Hlow.append([sum(lam[j] * Hlow[j][r] for j in range(low)) % PR for r in range(n)])
    # interpolation across the q cosets (coset_interpolate_row): V^-1 of the y_j applied to H_r(y_j)
    pieces = [[0] * n for _ in range(q)]
    for r in range(n):
        v = [(g[j][r] * pow(cj[j], (PR - 1 - r) % (PR - 1), PR) + Hlow[j][r]) % PR for j in range(q)]
        # solve sum_t c_t y_j^t = v_j
        A = [[pow(yj[j], t, PR) for t in range(q)] + [v[j]] for j in range(q)]
        for c in range(q):
            piv = next(rr for rr in range(c, q) if A[rr][c])
            A[c], A[piv] = A[piv], A[c]
            inv = pow(A[c][c], PR - 2, PR)
            A[c] = [a * inv % PR for a in A[c]]
            for rr in range(q):
                if rr != c and A[rr][c]:
                    f = A[rr][c]
                    A[rr] = [(a - f * b2) % PR for a, b2 in zip(A[rr], A[c])]
        for t in range(q):
            pieces[t][r] = A[t][q]
    # linear class on coset 0: iNTT with 1 / Z_H(c_0), times c_0^(-r), into piece 0
    vals = [sum(yp(G - 1 - i + PT + 5 * L) * num(gates[i], x) for i in range(G) if cls[i] == 2) * pow(zh(x), PR - 2, PR) % PR for x in rows(0)]
    b = _intt(vals, w)
    for r in range(n):
        pieces[0][r] = (pieces[0][r] + b[r] * pow(cj[0], (PR - 1 - r) % (PR - 1), PR)) % PR
    assert pieces == want


def test_coset_interpolate_adds_the_linear_part(harness, orc):
    """coset_interpolate_row with `lin`: piece 0 gains lin[r] * c_0^(-r), the other pieces are unchanged."""
    rnd = random.Random(77)
    R, n, C = P.R_MOD, 8, 5
    cs = [rnd.randrange(1, R) for _ in range(C)]
    ys = [pow(c, n, R) for c in cs]
    M = lambda v: orc.ints_to_mont([x % R for x in v])
    ev = lambda coeffs, x: sum(cf * pow(x, t, R) for t, cf in enumerate(coeffs)) % R
    H = [[rnd.randrange(R) for _ in range(C)] for _ in range(n)]
    lin = [rnd.randrange(R) for _ in range(n)]
    A = [[pow(ys[j], t, R) for t in range(C)] + [int(i == j) for i in range(C)] for j in range(C)]
    for c in range(C):
        inv = pow(A[c][c], -1, R)
        A[c] = [v * inv % R for v in A[c]]
        for r in range(C):
            if r != c and A[r][c]:
                f = A[r][c]
                A[r] = [(a - f * b) % R for a, b in zip(A[r], A[c])]
    vinv = M([A[t][C + j] for t in range(C) for j in range(C)])
    g = M([pow(cs[j], r, R) * ev(H[r], ys[j]) for j in range(C) for r in range(n)])
    inv_pow = M([pow(c, -r, R) for c in cs for r in range(n)])
    out = np.zeros((C * n, 4), dtype=np.uint64)
    lin_m = np.ascontiguousarray(M([pow(cs[0], r, R) * lin[r] for r in range(n)]), dtype=np.uint64)
    harness.coset_interpolate_lin(_p(np.ascontiguousarray(g, dtype=np.uint64)), _p(np.ascontiguousarray(inv_pow, dtype=np.uint64)),
                                  _p(np.ascontiguousarray(vinv, dtype=np.uint64)), ctypes.c_uint32(C), ctypes.c_size_t(n), _p(out), _p(lin_m))
    got = orc.mont_to_ints(out)
    assert got == [(H[r][t] + (lin[r] if t == 0 else 0)) % R for t in range(C) for r in range(n)]
