"""GPU: b200zk_verify_proofs — many proofs of one verifying key checked with one pairing (AccumulatorStrategy), the
points decompressed and every proof's opening summed on the device.  Verdicts agree with verify_proof proof by proof,
the accumulator equals the reference restatement (tests/verify_batch_ref.py) byte for byte, and failing proofs are
located wherever they sit in the batch."""
import ctypes
import importlib

import numpy as np
import pytest

from oracle import prover as OP
from tests import verify_batch_ref as VB

pytestmark = pytest.mark.gpu

Q = 0x30644e72e131a029b85045b68181585d97816a916871ca8d3c208c16d87cfd47


def _synth(zk):
    return importlib.import_module(zk.__name__ + ".circuits_synth")


def _chips(zk):
    return importlib.import_module(zk.__name__ + ".chips")


def _mont_ints(orc, vals):
    return orc.ints_to_mont([v % OP.R for v in vals]) if len(vals) else np.zeros((0, 4), dtype=np.uint64)


class Batch:
    """count proofs of one key made by create_proofs (job i % len(jobs), rng stream i), and the key's vk"""

    def __init__(self, zk, backend, orc, jobs, count, seed_s=4321):
        self.jobs = [jobs[i % len(jobs)] for i in range(count)]
        self.s = orc.random_fr(1, seed_s)[0]
        j0 = jobs[0]
        self.params = zk.ParamsKZG.setup(backend, j0.k, self.s)
        self.pk = zk.ProvingKey(self.params, j0.cs, j0.k, j0.fixed, j0.map_col, j0.map_row)
        self.insts = [[_mont_ints(orc, c) for c in j.instances] for j in self.jobs]
        self.tr = orc.ints_to_mont([j0.transcript_repr])[0]
        xs = orc.XorShiftWide()
        self.wides = [xs.draw(self.pk.rng_draws) for _ in range(count)]
        self.proofs = self.pk.create_proofs([j.advice for j in self.jobs], self.insts, self.wides, self.tr)
        g, _ = self.params.read()
        self.g = g
        fixed_c, sigma_c = self.pk.vk_commitments()
        self.vk = zk.VerifyingKey(j0.cs, j0.k, fixed_c, sigma_c, g[0], zk.g2_mul(self.s))

    def close(self):
        self.pk.close()
        self.params.close()


def _rng(count, seed=7):
    return np.random.Generator(np.random.PCG64(seed)).integers(0, 1 << 63, size=(count, 8), dtype=np.uint64) * 2 + 1


def _tamper_eval(proof):
    t = bytearray(proof); t[len(t) - 96] ^= 0x01                   # the last evaluation: still canonical, passes stage 1
    return bytes(t)


def _reference_jobs(zk, which):
    fe = importlib.import_module(zk.__name__ + ".frontend")
    chips = _chips(zk)
    if which == "less_than":
        return [fe.synthesize_job(chips.LessThanCircuit(755), 10, [list(range(800))])]
    return [fe.synthesize_job(chips.SafeAccumulatorCircuit([1, 3], [0, 0, 14, 13]), 8, [[0, 0, 15, 1]])]


@pytest.mark.parametrize("name,k", [("small", 5), ("mst_shaped", 9), ("v3_shaped", 11), ("generic_shapes", 10),
                                    ("mst_real", 9), ("less_than", 10), ("safe_accumulator", 8)])
def test_accepts_batches_of_every_shape(zk, backend, orc, name, k):
    """Batches from create_proofs of the synthetic shapes, the real Merkle Sum Tree with four users' witnesses, LessThan
    (800 public inputs) and SafeAccumulator (16 quotient pieces): every proof accepted, as verify_proof accepts it."""
    if name == "mst_real":
        jobs = [_chips(zk).merkle_sum_tree_job(9, levels=5, seed=s) for s in (1, 2, 3, 4)]
    elif name in ("less_than", "safe_accumulator"):
        jobs = _reference_jobs(zk, name)
    elif name == "generic_shapes":
        jobs = [_synth(zk).generic_shapes(k, seed=4 + i) for i in range(3)]
    else:
        jobs = [getattr(_synth(zk), name)(k)]
    b = Batch(zk, backend, orc, jobs, 6)
    try:
        assert all(p is not None for p in b.proofs)
        assert all(b.vk.verify_proof(i, p, b.tr) for i, p in zip(b.insts, b.proofs))
        assert b.vk.verify_proofs(backend, b.insts, b.proofs, b.tr, _rng(6)) == [True] * 6
        assert b.vk.verify_proofs(backend, b.insts, b.proofs, b.tr) == [True] * 6         # os.urandom draws
    finally:
        b.close()


def _g1_mont(orc, pt):
    return np.zeros(8, dtype=np.uint64) if pt is None else np.asarray(orc.ints_to_mont([pt[0], pt[1]], which=1)).reshape(8)


def _oracle_vk(orc, b):
    j0 = b.jobs[0]
    return OP.verifying_key(j0.cs, j0.k, orc.affine_to_ints(b.vk.fixed), orc.affine_to_ints(b.vk.sigma))


@pytest.mark.parametrize("name", ["small_k5", "mst_k9"])
def test_accumulator_equals_the_reference(zk, backend, orc, name):
    """(left, right) is byte for byte the reference's accumulate() of its shplonk_dual()s with the same draws, and it
    opens: e(left, [s]_2) = e(right, [1]_2)."""
    jobs = [_synth(zk).small(5)] if name == "small_k5" else [_chips(zk).merkle_sum_tree_job(9, levels=5, seed=s) for s in (1, 2)]
    b = Batch(zk, backend, orc, jobs, 4)
    try:
        wide = _rng(4, 11)
        ok, (left, right) = b.vk.verify_proofs(backend, b.insts, b.proofs, b.tr, wide, accumulator=True)
        assert ok == [True] * 4
        ovk = _oracle_vk(orc, b)
        duals = [VB.shplonk_dual(ovk, j.instances, p, j.transcript_repr) for j, p in zip(b.jobs, b.proofs)]
        want_l, want_r = VB.accumulate(duals, [VB.wide_to_fr(w) for w in wide])
        assert np.array_equal(left, _g1_mont(orc, want_l)) and np.array_equal(right, _g1_mont(orc, want_r))
        assert zk.pairing_check([left, _g1_mont(orc, (want_r[0], Q - want_r[1]))], [b.vk.s_g2, b.vk.g2])
        assert VB.P.g1_mul(want_l, orc.mont_to_ints(b.s)[0]) == want_r
    finally:
        b.close()


def test_single_proof_agrees_with_verify_proof(zk, backend, orc):
    """count = 1 gives verify_proof's verdict on the golden proof and on every tampered variant test_verifier.py checks;
    the golden proofs at positions 1 and 3 of a batch of 4 are accepted."""
    tv = importlib.import_module("tests.test_verifier")
    z, vk, inst, proof = tv.load_golden(zk, "small_k5")
    tr = z["transcript_repr"]
    one = np.array(orc.ints_to_mont([1])).reshape(4)
    r_bytes = (OP.R).to_bytes(32, "little")
    variants = [proof, proof + b"\x00" * 32, proof[:-32], proof[:-1], b"", proof[:-96] + r_bytes + proof[-64:]]
    for el in range(len(proof) // 32):
        bad = bytearray(proof); bad[32 * el + 3] ^= 0x10
        variants.append(bytes(bad))
    wrong = [c.copy() for c in inst]
    wrong[0][-1] = one
    big = [np.tile(one, ((1 << vk.k), 1))]
    cases = [(inst, v, tr) for v in variants] + [(wrong, proof, tr), (inst, proof, one), (big, proof, tr)]
    for i, (ins, p, t) in enumerate(cases):
        assert vk.verify_proofs(backend, [ins], [p], t, _rng(1, i)) == [vk.verify_proof(ins, p, t)], i
    assert vk.verify_proof(inst, proof, tr)
    # golden vectors inside a batch: the other positions are proofs of the same key from other rng streams
    job = _synth(zk).small(5)
    params = zk.ParamsKZG.setup(backend, job.k, orc.random_fr(1, int(z["seed_s"]))[0])
    pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    try:
        xs = orc.XorShiftWide()
        xs.draw(pk.rng_draws)
        others = pk.create_proofs([job.advice] * 2, [inst] * 2, [xs.draw(pk.rng_draws) for _ in range(2)], tr)
        assert vk.verify_proofs(backend, [inst] * 4, [others[0], proof, others[1], proof], tr, _rng(4)) == [True] * 4
    finally:
        pk.close(); params.close()


@pytest.fixture(scope="module")
def small64(zk, backend, orc):
    b = Batch(zk, backend, orc, [_synth(zk).small(5)], 64)
    yield b
    b.close()


@pytest.mark.parametrize("bad", [[0], [31], [63], [5, 40], list(range(64))])
def test_localisation(zk, backend, orc, small64, bad):
    """A flipped evaluation or a wrong public input passes stage 1 and fails the pairing: the call returns EVERIFY with
    exactly those proofs rejected, wherever they sit in a batch of 64."""
    b = small64
    proofs, insts = list(b.proofs), [list(i) for i in b.insts]
    for n, i in enumerate(bad):
        if n % 2:
            col = insts[i][0].copy(); col[-1] = orc.ints_to_mont([12345])[0]; insts[i] = [col] + insts[i][1:]
        else:
            proofs[i] = _tamper_eval(proofs[i])
    got = b.vk.verify_proofs(backend, insts, proofs, b.tr, _rng(64, len(bad)))
    assert got == [i not in bad for i in range(64)]
    for i in bad[:2]:
        assert not b.vk.verify_proof(insts[i], proofs[i], b.tr)


def test_rng_changes_the_accumulator_not_the_verdicts(zk, backend, small64):
    b = small64
    proofs = list(b.proofs); proofs[9] = _tamper_eval(proofs[9])
    ok1, acc1 = b.vk.verify_proofs(backend, b.insts, proofs, b.tr, _rng(64, 1), accumulator=True)
    ok2, acc2 = b.vk.verify_proofs(backend, b.insts, proofs, b.tr, _rng(64, 2), accumulator=True)
    assert ok1 == ok2 == [i != 9 for i in range(64)]
    assert not np.array_equal(acc1[0], acc2[0]) and not np.array_equal(acc1[1], acc2[1])


def _off_curve_x():
    for x in range(1, 100):
        if pow((x ** 3 + 3) % Q, (Q - 1) // 2, Q) == Q - 1:
            return x
    raise AssertionError


def test_stage_one_rejections_inside_a_batch(zk, backend, orc):
    """A non-canonical scalar, an off-curve point, a sign bit on the identity, a truncated proof and an oversized instance
    each reject only their proof; the accumulator is the reference accumulator of the others with the same weights.
    Trailing bytes are accepted."""
    b = Batch(zk, backend, orc, [_synth(zk).small(5)], 8)
    try:
        p, insts = list(b.proofs), list(b.insts)
        p[0] = p[0] + b"\x07" * 40                                                            # trailing bytes: fine
        p[1] = p[1][:-96] + OP.R.to_bytes(32, "little") + p[1][-64:]                          # non-canonical scalar
        p[2] = _off_curve_x().to_bytes(32, "little") + p[2][32:]                               # x^3 + 3 has no root
        p[3] = bytes(31) + b"\x80" + p[3][32:]                                                 # identity with a sign bit
        p[5] = p[5][:-1]                                                                      # truncated
        one = np.array(orc.ints_to_mont([1])).reshape(4)
        insts[6] = [np.tile(one, ((1 << 5), 1))] + list(insts[6][1:])                          # instance too large
        rejected = {1, 2, 3, 5, 6}
        wide = _rng(8, 5)
        l0 = backend.launch_count()
        ok, (left, right) = b.vk.verify_proofs(backend, insts, p, b.tr, wide, accumulator=True)
        assert ok == [i not in rejected for i in range(8)]
        assert backend.launch_count() - l0 == 3
        for i in range(8):
            assert b.vk.verify_proof(insts[i], p[i], b.tr) == ok[i]
        ovk = _oracle_vk(orc, b)
        duals = [(None, None) if i in rejected else VB.shplonk_dual(ovk, b.jobs[i].instances, p[i], b.jobs[i].transcript_repr)
                 for i in range(8)]
        want_l, want_r = VB.accumulate(duals, [VB.wide_to_fr(w) for w in wide])
        assert np.array_equal(left, _g1_mont(orc, want_l)) and np.array_equal(right, _g1_mont(orc, want_r))
        # nothing survives stage 1: identity accumulator, every proof rejected
        ok, (left, right) = b.vk.verify_proofs(backend, [insts[i] for i in sorted(rejected)], [p[i] for i in sorted(rejected)],
                                               b.tr, _rng(5), accumulator=True)
        assert ok == [False] * 5 and not left.any() and not right.any()
    finally:
        b.close()


def _raw(zk, backend, vk, insts, proofs, tr, wide, count=None, blob=None, null_rng=False, null_proof=None):
    count = len(proofs) if count is None else count
    keep = [c if c.shape[0] else np.zeros((1, 4), dtype=np.uint64) for i in insts for c in i]
    lens = np.array([c.shape[0] for i in insts for c in i] + [0], dtype=np.uint32)
    bufs = [np.frombuffer(p, dtype=np.uint8) for p in proofs]
    ptrs = (ctypes.c_void_p * max(len(bufs), 1))(*[x.ctypes.data for x in bufs])
    if null_proof is not None:
        ptrs[null_proof] = None
    plens = np.array([x.shape[0] for x in bufs] + [0], dtype=np.uint64)
    blob = vk.blob if blob is None else blob
    status = np.full(max(len(proofs), 1), 7, dtype=np.int32)
    V = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rc = zk.lib().b200zk_verify_proofs(backend._ctx, V(blob), ctypes.c_size_t(blob.shape[0]), V(vk.fixed), V(vk.sigma), V(vk.g1), V(vk.g2),
                                       V(vk.s_g2), ctypes.c_uint32(count), (ctypes.c_void_p * len(keep))(*[c.ctypes.data for c in keep]),
                                       V(lens), V(np.ascontiguousarray(tr)), ptrs, V(plens), None if null_rng else V(wide), V(status), None)
    return rc, status


def test_bad_arguments(zk, backend, orc):
    """count = 0, a null rng, a null proof with a nonzero length and a blob that does not parse return EINVAL before any
    device work; the same ctx then verifies a batch, a pk on it proves the same bytes as before, and a rank of a sharded
    group verifies too."""
    b = Batch(zk, backend, orc, [_synth(zk).small(5)], 3)
    try:
        wide = _rng(3)
        l0 = backend.launch_count()
        assert _raw(zk, backend, b.vk, b.insts, b.proofs, b.tr, wide, count=0)[0] == zk.EINVAL
        assert _raw(zk, backend, b.vk, b.insts, b.proofs, b.tr, wide, null_rng=True)[0] == zk.EINVAL
        assert _raw(zk, backend, b.vk, b.insts, b.proofs, b.tr, wide, null_proof=1)[0] == zk.EINVAL
        blob = b.vk.blob.copy(); blob[0] ^= 1
        assert _raw(zk, backend, b.vk, b.insts, b.proofs, b.tr, wide, blob=blob)[0] == zk.EINVAL
        assert backend.launch_count() == l0
        with pytest.raises(zk.B200zkError):
            b.vk.verify_proofs(backend, [], [], b.tr)
        rc, status = _raw(zk, backend, b.vk, b.insts, b.proofs, b.tr, wide)
        assert rc == 0 and list(status) == [0, 0, 0]
        proofs = list(b.proofs); proofs[2] = _tamper_eval(proofs[2])
        rc, status = _raw(zk, backend, b.vk, b.insts, proofs, b.tr, wide)
        assert rc == zk.EVERIFY and list(status) == [0, 0, zk.EVERIFY]
        assert b.pk.create_proofs([j.advice for j in b.jobs], b.insts, b.wides, b.tr) == b.proofs
        assert b.pk.create_proof(b.jobs[1].advice, b.insts[1], b.wides[1], b.tr) == b.proofs[1]
        group = zk.Group([0, 0])
        try:
            assert b.vk.verify_proofs(group.backends[1], b.insts, proofs, b.tr, wide) == [True, True, False]
        finally:
            group.close()
    finally:
        b.close()


def test_scale_1024_mst_k9(zk, backend, orc):
    """1024 proofs of the Merkle Sum Tree at k = 9 with one tampered proof: exactly that one is reported, and randomly
    chosen proofs agree with verify_proof."""
    jobs = [_chips(zk).merkle_sum_tree_job(9, levels=5, seed=s) for s in (1, 2, 3, 4)]
    b = Batch(zk, backend, orc, jobs, 1024)
    try:
        proofs = list(b.proofs); proofs[777] = _tamper_eval(proofs[777])
        got = b.vk.verify_proofs(backend, b.insts, proofs, b.tr, _rng(1024, 3))
        assert got == [i != 777 for i in range(1024)]
        pick = sorted(set(np.random.Generator(np.random.PCG64(1)).integers(0, 1024, size=6).tolist()) | {777})
        for i in pick:
            assert b.vk.verify_proof(b.insts[i], proofs[i], b.tr) == got[i], i
    finally:
        b.close()
