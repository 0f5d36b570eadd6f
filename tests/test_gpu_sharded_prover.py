"""GPU: ONE create_proof sharded over G ranks (BASELINE config 5, SURVEY.md 8(e)) produces exactly the
bytes of the single-GPU proof — and therefore of the oracle, which tests/test_gpu_prover.py pins the
single-GPU prover to.  The ranks are the threads of a b200zk_group; on the single-GPU test tier they
all share device 0 (same SPMD code path, same exchanges, peer copies degenerate to device-to-device
copies), on a multi-GPU box B200ZK_TEST_DEVICES=0,1,... spreads them over real devices."""
import importlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _synth(zk):
    return importlib.import_module(zk.__name__ + ".circuits_synth")


def _devices(world):
    env = os.environ.get("B200ZK_TEST_DEVICES")
    devs = [int(x) for x in env.split(",")] if env else [0]
    return [devs[r % len(devs)] for r in range(world)]


def _single(zk, backend, orc, job, s):
    params = zk.ParamsKZG.setup(backend, job.k, s)
    pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    wide = orc.XorShiftWide().draw(pk.rng_draws)
    from oracle import prover as OP
    inst = [orc.ints_to_mont([v % OP.R for v in c]) if len(c) else np.zeros((0, 4), dtype=np.uint64) for c in job.instances]
    tr_repr = orc.ints_to_mont([job.transcript_repr])[0]
    proof = pk.create_proof(job.advice, inst, wide, tr_repr)
    pk.close(); params.close()
    return proof, wide, inst, tr_repr


def _proving_key(zk, params, job, lookup_early=None):
    """A ProvingKey built with B200ZK_LOOKUP_EARLY set to `lookup_early` (None: the library decides by free memory)."""
    if lookup_early is None:
        return zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    old = os.environ.get("B200ZK_LOOKUP_EARLY")
    os.environ["B200ZK_LOOKUP_EARLY"] = lookup_early
    try:
        return zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    finally:
        if old is None:
            del os.environ["B200ZK_LOOKUP_EARLY"]
        else:
            os.environ["B200ZK_LOOKUP_EARLY"] = old


def _sharded(zk, job, s, world, wide, inst, tr_repr, dev_inputs=False, lookup_early=None):
    group = zk.Group(_devices(world))
    try:
        params = [zk.ParamsKZG.setup(b, job.k, s) for b in group.backends]
        pks = [_proving_key(zk, p, job, lookup_early[r] if lookup_early else None) for r, p in enumerate(params)]
        if dev_inputs:
            adv = np.concatenate([np.ascontiguousarray(a).reshape(-1, 4) for a in job.advice])
            d_adv = [b.to_device(adv) for b in group.backends]
            d_wide = [b.to_device(wide) for b in group.backends]
            proof = group.create_proof_dev(pks, d_adv, inst, d_wide, tr_repr)
            for d in d_adv + d_wide:
                d.free()
        else:
            proof = group.create_proof(pks, job.advice, inst, wide, tr_repr)
        for pk in pks:
            pk.close()
        for p in params:
            p.close()
        return proof
    finally:
        group.close()


@pytest.mark.parametrize("name,k,worlds", [("small", 6, (2, 3)), ("mst_shaped", 9, (2, 4, 8)), ("v3_shaped", 8, (2, 5)),
                                           ("generic_shapes", 8, (3, 8))])
def test_sharded_proof_equals_single_gpu(zk, backend, orc, name, k, worlds):
    job = getattr(_synth(zk), name)(k)
    s = orc.random_fr(1, 4321)[0]
    want, wide, inst, tr_repr = _single(zk, backend, orc, job, s)
    for world in worlds:
        got = _sharded(zk, job, s, world, wide, inst, tr_repr)
        assert got == want, f"world {world}: sharded proof differs from the single-GPU proof"
    assert _sharded(zk, job, s, worlds[0], wide, inst, tr_repr, dev_inputs=True) == want


def _wide_job(zk, k, advice):
    """`advice` columns of bits at 2^k rows, every one queried by a single boolean gate (q * sum_i a_i (1 - a_i)); the
    instance column and advice column 0 in the permutation (two sets of one column)."""
    synth = _synth(zk)
    C = importlib.import_module(zk.__name__ + ".circuit")
    n = 1 << k
    rng = np.random.Generator(np.random.PCG64(11))
    cs = C.ConstraintSystem(advice, 1, 1)
    cs.enable_equality(C.ADVICE, 0)
    cs.enable_equality(C.INSTANCE, 0)
    poly = None
    for c in range(advice):
        a = cs.query_advice(c, 0)
        poly = a * (1 - a) if poly is None else poly + a * (1 - a)
    cs.create_gate([cs.query_fixed(0, 0) * poly])
    job = synth.Job(cs, k)
    usable = n - (cs.blinding_factors() + 1)
    job.fixed = [synth.mont_from_small((np.arange(n) < usable).astype(np.int64))]
    bits = rng.integers(0, 2, size=(advice, n), dtype=np.int64)
    job.advice = [synth.mont_from_small(b) for b in bits]
    job.instances = [[int(bits[0][r]) for r in range(2)]]
    asm = C.PermutationAssembly(len(cs.permutation), n)
    for r in range(2):
        asm.copy(1, r, 0, r)                                             # instance[0][r] == a_0[r]
    job.map_col, job.map_row = asm.map_col, asm.map_row
    return job


def test_sharded_wide_circuit(zk, backend, orc):
    """512 advice columns over 2 ranks: 256 commitments (16 KiB) per rank in one host exchange; the proof equals the
    single-GPU proof."""
    job = _wide_job(zk, 6, 512)
    s = orc.random_fr(1, 4321)[0]
    want, wide, inst, tr_repr = _single(zk, backend, orc, job, s)
    assert _sharded(zk, job, s, 2, wide, inst, tr_repr) == want


def test_sharded_ranks_with_different_arenas(zk, backend, orc):
    """Ranks whose proving keys differ in B200ZK_LOOKUP_EARLY carve different arenas (the early lookup cosets sit in the
    middle of it); the exchanges copy from each owner's own buffers, so the proof is still the single-GPU proof."""
    for name, k in (("small", 6), ("mst_shaped", 9)):
        job = getattr(_synth(zk), name)(k)
        s = orc.random_fr(1, 4321)[0]
        want, wide, inst, tr_repr = _single(zk, backend, orc, job, s)
        for early in (("1", "0"), ("0", "1", "0")):
            got = _sharded(zk, job, s, len(early), wide, inst, tr_repr, lookup_early=early)
            assert got == want, f"{name}: B200ZK_LOOKUP_EARLY per rank {early}"


def test_sharded_real_merkle_sum_tree_k11(zk, backend, orc):
    """The reference's MerkleSumTreeCircuit (8 lookups, 4 permutation sets, 5 quotient cosets, lookup terms on 4
    of them) at k = 11 over 2, 4 and 8 ranks: byte-identical to the single-GPU proof, which
    test_gpu_prover.py::test_real_merkle_sum_tree_k11 pins to the oracle."""
    chips = importlib.import_module(zk.__name__ + ".chips")
    job = chips.merkle_sum_tree_job(11, levels=9, seed=5)
    s = orc.random_fr(1, 4321)[0]
    want, wide, inst, tr_repr = _single(zk, backend, orc, job, s)
    for world in (2, 4, 8):
        assert _sharded(zk, job, s, world, wide, inst, tr_repr) == want, f"world {world}"


def test_sharded_lookup_failure_is_collective(zk, orc):
    """Error::ConstraintSystemFailure detected by the rank that owns the lookup reaches every rank (no hang)."""
    synth = _synth(zk)
    job = synth.small(6)
    byte_col = 5 + 3 + 2
    bad = np.array(job.advice[byte_col])
    bad[3] = orc.ints_to_mont([100000])[0]
    job.advice[byte_col] = bad
    s = orc.random_fr(1, 4321)[0]
    group = zk.Group(_devices(3))
    try:
        params = [zk.ParamsKZG.setup(b, job.k, s) for b in group.backends]
        pks = [zk.ProvingKey(p, job.cs, job.k, job.fixed, job.map_col, job.map_row) for p in params]
        wide = orc.XorShiftWide().draw(pks[0].rng_draws)
        from oracle import prover as OP
        inst = [orc.ints_to_mont([v % OP.R for v in c]) for c in job.instances]
        with pytest.raises(zk.B200zkError, match="-5"):
            group.create_proof(pks, job.advice, inst, wide, orc.ints_to_mont([job.transcript_repr])[0])
    finally:
        group.close()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_group_best_multiexp_and_best_fft(zk, backend, orc, world):
    """b200zk_group_msm / b200zk_group_fft: one best_multiexp by point range and one best_fft four-step (exchange fused into
    the column-step kernel) over the ranks of a group, host buffers in and out, against the oracle."""
    from oracle import pyref
    n = (1 << 14) + 37
    g, _ = orc.params_setup(15, orc.random_fr(1, 1234)[0], with_lagrange=False)
    coeffs = orc.random_fr(n, 77)
    want = orc.g1_batch_normalize(orc.best_multiexp(coeffs, g[:n]))[0]
    group = zk.Group(_devices(world))
    try:
        assert np.array_equal(group.best_multiexp(coeffs, g[:n])[:8], want)
        for k in (16, 17):
            a = orc.random_fr(1 << k, 90 + k)
            w = orc.ints_to_mont([pyref.omega_for_k(k)])[0]
            assert np.array_equal(group.best_fft(a, w, k), orc.best_fft(a, w, k)), f"k={k}"
        a = orc.random_fr(1 << 10, 5)                                      # below the four-step threshold: rank 0 alone
        w = orc.ints_to_mont([pyref.omega_for_k(10)])[0]
        assert np.array_equal(group.best_fft(a, w, 10), orc.best_fft(a, w, 10))
    finally:
        group.close()
