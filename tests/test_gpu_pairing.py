"""GPU: b200zk_pairing_checks — many pairing-product checks in one call — against the host pairing of
b200zk_pairing_check, and verify_proofs, whose failing batches are now judged proof by proof with it."""
import ctypes
import importlib

import numpy as np
import pytest

from tests import pairing_ref as P
from tests import verify_batch_ref as VB
from tests.test_gpu_verify_batch import Batch, _g1_mont, _oracle_vk, _rng, _tamper_eval

pytestmark = pytest.mark.gpu

Z1, Z2 = np.zeros((1, 8), np.uint64), np.zeros((1, 16), np.uint64)


def _check(rng, m, g2_pool, truth):
    """m pairs whose product is one (truth) or not: e(a_0 P, Q_0) ... e(a_{m-2} P, Q_{m-2}) e(-(sum a_i b_i) P, Q) with
    Q_i = b_i Q, Q the last pool point; a false one adds 1 to the last scalar.  m = 1: e(identity, Q) or e(aP, Q)."""
    if m == 1:
        return (Z1 if truth else P.g1_mul([int(rng.integers(1, 2**60))])), g2_pool[-1][1][None]
    idx = rng.integers(0, len(g2_pool) - 1, m - 1)
    a = [int(x) for x in rng.integers(1, 2**60, m - 1)]
    s = sum(ai * g2_pool[i][0] for ai, i in zip(a, idx)) + (0 if truth else 1)
    g1 = np.vstack([P.g1_mul(a), P.g1_neg(P.g1_mul([s]))])
    g2 = np.vstack([g2_pool[i][1] for i in idx] + [g2_pool[-1][1]])
    return g1, g2


@pytest.fixture(scope="module")
def g2_pool():
    bs = [3, 5, 7, 11, 13, 1]
    return list(zip(bs, P.g2_mul(bs)))


def test_verdicts_equal_host_pairing_check(zk, backend, g2_pool):
    """64 checks with m = 1 .. 4: true products from bilinearity, false ones one scalar off, identities, shared and
    all-distinct G2 points; each verdict equals b200zk_pairing_check's."""
    rng = np.random.default_rng(5)
    for m in (1, 2, 3, 4):
        g1s, g2s, want = [], [], []
        for j in range(16):
            g1, g2 = _check(rng, m, g2_pool, truth=j % 3 != 1)
            if j == 5:                                                  # all-distinct G2 points, never seen before
                bs = [int(x) for x in rng.integers(2, 2**40, m)]
                g2 = P.g2_mul(bs)
            if j == 7:
                g2 = np.vstack([Z2, g2[1:]])                            # identity on the G2 side
            g1s.append(g1); g2s.append(g2)
            want.append(0 if zk.pairing_check(g1, g2) else zk.EVERIFY)
        status = zk.pairing_checks(backend, np.vstack(g1s), np.vstack(g2s), m)
        assert list(status) == want, m
        assert want.count(0) not in (0, 16)


@pytest.mark.parametrize("count", [1, 33, 1024, 16384])
def test_verdicts_at_scale(zk, backend, g2_pool, count):
    """2-pair checks, true and false interleaved at known positions (every 7th and the last are false)."""
    rng = np.random.default_rng(count)
    pool = [_check(rng, 2, g2_pool, truth) for truth in [True] * 24 + [False] * 8]
    truth = [j % 7 != 3 and j != count - 1 for j in range(count)]
    pick = [int(rng.integers(0, 24)) if t else 24 + int(rng.integers(0, 8)) for t in truth]
    g1 = np.vstack([pool[i][0] for i in pick])
    g2 = np.vstack([pool[i][1] for i in pick])
    status = zk.pairing_checks(backend, g1, g2, 2)
    assert list(status) == [0 if t else zk.EVERIFY for t in truth]


def test_bad_arguments_leave_the_ctx_usable(zk, backend, orc, g2_pool):
    """null pointers, count == 0, m == 0 and points off either curve return EINVAL with the launch count unmoved; the
    ctx then checks, and a pk with lanes on it proves the same bytes as before."""
    from tests.test_gpu_verify_batch import _synth
    g1, g2 = _check(np.random.default_rng(1), 2, g2_pool, True)
    g1 = np.ascontiguousarray(g1); g2 = np.ascontiguousarray(g2)
    st = np.zeros(1, dtype=np.int32)
    fn = zk.lib().b200zk_pairing_checks
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)                    # noqa: E731
    b = Batch(zk, backend, orc, [_synth(zk).small(5)], 3)
    try:
        b.pk.reserve_lanes(2)
        l0 = backend.launch_count()
        off1 = g1.copy(); off1[0, 0] ^= np.uint64(1)
        off2 = g2.copy(); off2[0, 0] ^= np.uint64(1)
        cases = [(None, vp(g2), 2, 1, vp(st)), (vp(g1), None, 2, 1, vp(st)), (vp(g1), vp(g2), 2, 1, None),
                 (vp(g1), vp(g2), 2, 0, vp(st)), (vp(g1), vp(g2), 0, 1, vp(st)),
                 (vp(off1), vp(g2), 2, 1, vp(st)), (vp(g1), vp(off2), 2, 1, vp(st))]
        for c in cases:
            assert fn(backend._ctx, c[0], c[1], ctypes.c_uint32(c[2]), ctypes.c_uint32(c[3]), c[4]) == zk.EINVAL
        assert backend.launch_count() == l0
        assert list(zk.pairing_checks(backend, g1, g2, 2)) == [0]
        assert backend.launch_count() == l0 + 3
        assert b.pk.create_proofs([j.advice for j in b.jobs], b.insts, b.wides, b.tr) == b.proofs
    finally:
        b.close()


@pytest.fixture(scope="module")
def mst1024(zk, backend, orc):
    jobs = [importlib.import_module(zk.__name__ + ".chips").merkle_sum_tree_job(9, levels=5, seed=s) for s in (1, 2, 3, 4)]
    b = Batch(zk, backend, orc, jobs, 1024)
    yield b
    b.close()


def _launches_of(backend, fn):
    l0 = backend.launch_count()
    out = fn()
    return out, backend.launch_count() - l0


@pytest.mark.parametrize("bad", [[777], [0, 1023], list(range(3, 1024, 16)), list(range(1024))])
def test_verify_proofs_judges_each_proof(zk, backend, mst1024, bad):
    """1 024 MST k = 9 proofs with 1, 2, 64 and all tampered: the statuses are exactly the tampered set, sampled
    proofs agree with verify_proof, and one and 64 tampered proofs cost the same launches."""
    b = mst1024
    proofs = list(b.proofs)
    for i in bad:
        proofs[i] = _tamper_eval(proofs[i])
    got, launches = _launches_of(backend, lambda: b.vk.verify_proofs(backend, b.insts, proofs, b.tr, _rng(1024, 3)))
    assert got == [i not in bad for i in range(1024)]
    pick = sorted(set(np.random.Generator(np.random.PCG64(len(bad))).integers(0, 1024, size=4).tolist()) | set(bad[:2]))
    for i in pick:
        assert b.vk.verify_proof(b.insts[i], proofs[i], b.tr) == got[i], i
    if len(bad) in (1, 64):
        _, other = _launches_of(backend, lambda: b.vk.verify_proofs(
            backend, b.insts, [_tamper_eval(p) if i in ([5] if len(bad) == 64 else range(7, 1024, 16)) else p
                               for i, p in enumerate(b.proofs)], b.tr, _rng(1024, 3)))
        assert other == launches


def test_accumulator_with_failures_equals_the_reference(zk, backend, orc):
    """With tampered proofs in the batch the accumulator is still the reference's accumulate() byte for byte, and
    every status equals verify_proof's."""
    chips = importlib.import_module(zk.__name__ + ".chips")
    b = Batch(zk, backend, orc, [chips.merkle_sum_tree_job(9, levels=5, seed=s) for s in (1, 2)], 6)
    try:
        proofs = list(b.proofs)
        for i in (1, 4):
            proofs[i] = _tamper_eval(proofs[i])
        wide = _rng(6, 11)
        ok, (left, right) = b.vk.verify_proofs(backend, b.insts, proofs, b.tr, wide, accumulator=True)
        assert ok == [b.vk.verify_proof(b.insts[i], proofs[i], b.tr) for i in range(6)] == [i not in (1, 4) for i in range(6)]
        ovk = _oracle_vk(orc, b)
        duals = [VB.shplonk_dual(ovk, j.instances, p, j.transcript_repr) for j, p in zip(b.jobs, proofs)]
        want_l, want_r = VB.accumulate(duals, [VB.wide_to_fr(w) for w in wide])
        assert np.array_equal(left, _g1_mont(orc, want_l)) and np.array_equal(right, _g1_mont(orc, want_r))
    finally:
        b.close()
