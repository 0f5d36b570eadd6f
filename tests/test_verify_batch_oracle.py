"""CPU: the batch verifier's algebra on oracle proofs (tests/verify_batch_ref.py).  AccumulatorStrategy sums the
proofs' SHPLONK pairs with random weights; with the SRS secret s, the pairing check e(left, [s]_2) = e(right, [1]_2)
becomes s * left == right, so a batch of good proofs passes, and one tampered evaluation anywhere makes it fail."""
import importlib

import pytest

from oracle import prover as OP
from oracle import pyref as P
from tests import verify_batch_ref as VB

R = OP.R


@pytest.fixture(scope="module")
def batch(zk, orc):
    synth = importlib.import_module(zk.__name__ + ".circuits_synth")
    job = synth.small(5)
    s = orc.random_fr(1, 21)[0]
    g, gl = orc.params_setup(job.k, s)
    pk = OP.keygen_pk(job.cs, job.k, job.fixed, job.map_col, job.map_row)
    xs = orc.XorShiftWide()
    proofs = [OP.create_proof(g, gl, pk, job.advice, job.instances, xs.draw(OP.rng_draws_needed(job.cs, job.k)), job.transcript_repr)[0]
              for _ in range(4)]
    assert len(set(proofs)) == 4
    return orc.mont_to_ints(s)[0], g, pk, job, proofs


def _dual(b, proof):
    s, g, pk, job, _ = b
    return VB.shplonk_dual(pk, job.instances, proof, job.transcript_repr, params_g=g)


def _rs(orc, count, seed=3):
    return [VB.wide_to_fr(w) for w in orc.XorShiftWide(bytes(range(seed, seed + 16))).draw(count)]


def test_each_dual_opens(batch):
    s, g, pk, job, proofs = batch
    for p in proofs:
        left, right = _dual(batch, p)
        assert P.g1_mul(left, s) == right
        assert OP.verify_full(s, g, pk, job.instances, p, job.transcript_repr)


def test_accumulator_of_good_proofs_opens(batch, orc):
    s = batch[0]
    duals = [_dual(batch, p) for p in batch[4]]
    rs = _rs(orc, 4)
    left, right = VB.accumulate(duals, rs)
    assert left is not None and P.g1_mul(left, s) == right
    # written out: c_i = prod_{j > i} r_j
    cs = [1] * 4
    for i in range(2, -1, -1):
        cs[i] = cs[i + 1] * rs[i + 1] % R
    hand_l = hand_r = None
    for (l, r), c in zip(duals, cs):
        hand_l, hand_r = P.g1_add(hand_l, P.g1_mul(l, c)), P.g1_add(hand_r, P.g1_mul(r, c))
    assert (hand_l, hand_r) == (left, right)
    # r_0 only scales the empty accumulator; a different r_1 changes the accumulator, and it still opens
    assert VB.accumulate(duals, [rs[0] + 1] + rs[1:]) == (left, right)
    other = VB.accumulate(duals, [rs[0], rs[1] + 1] + rs[2:])
    assert other != (left, right) and P.g1_mul(other[0], s) == other[1]
    # a proof that adds nothing keeps the others' weights
    dropped = VB.accumulate([duals[0], (None, None), duals[2], duals[3]], rs)
    assert dropped == (P.g1_add(P.g1_add(P.g1_mul(duals[0][0], cs[0]), P.g1_mul(duals[2][0], cs[2])), duals[3][0]),
                       P.g1_add(P.g1_add(P.g1_mul(duals[0][1], cs[0]), P.g1_mul(duals[2][1], cs[2])), duals[3][1]))


@pytest.mark.parametrize("bad", [0, 2, 3])
def test_one_tampered_evaluation_breaks_the_batch(batch, orc, bad):
    s, proofs = batch[0], list(batch[4])
    t = bytearray(proofs[bad]); t[len(t) - 96] ^= 0x01             # the last evaluation (still canonical)
    proofs[bad] = bytes(t)
    duals = [_dual(batch, p) for p in proofs]
    assert P.g1_mul(duals[bad][0], s) != duals[bad][1]
    left, right = VB.accumulate(duals, _rs(orc, 4))
    assert P.g1_mul(left, s) != right
