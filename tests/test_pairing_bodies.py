"""CPU: the device pairing bodies of csrc/pairing.cuh, compiled for the host (tests/pairing_harness.cpp), against the host
pairing of csrc/pairing.hpp that b200zk_pairing_check and verify_proof use.  Every comparison is byte for byte."""
import os
import sys

import numpy as np
import pytest

from tests import pairing_ref as P

sys.path.insert(0, os.path.join(P.ROOT, "tools"))
import gen_pairing_frobenius  # noqa: E402

ONE12 = np.array(P.mont(1) + [0] * 44, dtype=np.uint64)


@pytest.fixture(scope="module")
def rng():
    return np.random.default_rng(20261022)


def test_frobenius_constants_match_their_recomputation():
    path = os.path.join(P._CSRC, "pairing_frobenius.inc")
    assert open(path).read() == gen_pairing_frobenius.render()


@pytest.mark.parametrize("op", [0, 1, 2])
def test_fq2_ops_equal_host(rng, op):
    a, b = P.rand_fq(rng, 32, 2), P.rand_fq(rng, 32, 2)
    a[0] = 0                                                 # inv(0) = 0 on both sides
    assert (P.fq2(op, a, b, which=0) == P.fq2(op, a, b, which=1)).all()


@pytest.mark.parametrize("op", ["mul", "sqr"])
def test_fq12_mul_and_sqr_equal_host(rng, op):
    a, b = P.rand_fq(rng, 8, 12), P.rand_fq(rng, 8, 12)
    assert (P.fq12(op, a, b, which=0) == P.fq12(op, a, b, which=1)).all()


def test_fq12_inverse(rng):
    a = P.rand_fq(rng, 8, 12)
    assert (P.fq12("mul", P.fq12("inv", a), a, which=1) == ONE12).all()


def test_line_product_equals_dense_host_product(rng):
    f, lines = P.rand_fq(rng, 8, 12), P.rand_fq(rng, 8, 6)
    pts = P.g1_mul([int(x) for x in rng.integers(1, 2**62, 8)])
    assert (P.line(f, lines, pts, which=0) == P.line(f, lines, pts, which=1)).all()


@pytest.mark.parametrize("k", [1, 2, 3])
def test_frobenius_equals_plain_power(rng, k):
    a = P.rand_fq(rng, 3, 12)
    assert (P.fq12(f"frob{k}", a) == P.fq12_pow(a, P.Q**k)).all()


def test_cyclotomic_squaring(rng):
    e = P.fq12("easy", P.rand_fq(rng, 6, 12))
    assert (P.fq12("mul", e, P.fq12("frob3", P.fq12("frob3", e)), which=1) == ONE12).all()    # e^(q^6 + 1) = 1
    assert (P.fq12("cyc_sqr", e) == P.fq12("sqr", e, which=1)).all()


def test_final_exponentiation_equals_host(rng):
    a = P.rand_fq(rng, 3, 12)
    assert (P.fq12("final_exp", a) == P.fq12("final_exp", a, which=1)).all()


def _cases(rng):
    """(g1, g2, m) products of 1..4 pairs: random pairs, identities on either side, P / -P, repeated G2 points, and a
    true product e(aP, bQ) e(-abP, Q)."""
    sc = lambda n: [int(x) for x in rng.integers(1, 2**62, n)]       # noqa: E731
    out = []
    for m in (1, 2, 3, 4):
        out.append((P.g1_mul(sc(m)), P.g2_mul(sc(m)), m))
    z1, z2 = np.zeros((1, 8), np.uint64), np.zeros((1, 16), np.uint64)
    p, q = P.g1_mul(sc(2)), P.g2_mul(sc(2))
    out.append((np.vstack([z1, p[:1]]), np.vstack([q[:1], q[1:]]), 2))          # identity on the G1 side
    out.append((p, np.vstack([z2, q[1:]]), 2))                                  # identity on the G2 side
    out.append((np.vstack([p[:1], P.g1_neg(p[:1])]), np.vstack([q[:1], q[:1]]), 2))   # e(P, Q) e(-P, Q) = 1
    out.append((P.g1_mul(sc(3)), np.vstack([q[:1]] * 3), 3))                   # one G2 point three times
    a, b = sc(2)
    out.append((np.vstack([P.g1_mul([a]), P.g1_neg(P.g1_mul([a * b]))]), np.vstack([P.g2_mul([b]), P.g2_mul([1])]), 2))
    return out


def test_prepared_miller_loop_and_final_exponentiation_equal_host_pairing(rng):
    truths = []
    for g1, g2, m in _cases(rng):
        dev, host = P.pairing(g1, g2, m, which=0), P.pairing(g1, g2, m, which=1)
        assert (dev == host).all(), m
        truths.append(bool((dev == ONE12).all()))
    assert truths[:4] == [False] * 4 and truths[6] and truths[8]
