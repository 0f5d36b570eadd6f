"""GPU: b200zk_create_proofs — many witnesses of one proving key proved side by side on concurrent lanes of one device.
Every proof of a batch is byte for byte the proof create_proof returns for the same inputs, whatever the lane count,
the entry point (host or device inputs), the position in the batch, or a failing witness elsewhere in it."""
import ctypes
import hashlib
import importlib
import json
import os

import numpy as np
import pytest

from oracle import prover as OP

pytestmark = pytest.mark.gpu


def _synth(zk):
    return importlib.import_module(zk.__name__ + ".circuits_synth")


def _chips(zk):
    return importlib.import_module(zk.__name__ + ".chips")


def _mont_ints(orc, vals):
    return orc.ints_to_mont([v % OP.R for v in vals]) if len(vals) else np.zeros((0, 4), dtype=np.uint64)


def _key(zk, backend, orc, job, seed_s=4321):
    s = orc.random_fr(1, seed_s)[0]
    params = zk.ParamsKZG.setup(backend, job.k, s)
    pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    return s, params, pk


def _inputs(orc, jobs):
    return [[_mont_ints(orc, c) for c in j.instances] for j in jobs], orc.ints_to_mont([jobs[0].transcript_repr])[0]


def _streams(orc, pk, count):
    """count different rng streams: the halo2 test stream, then its continuation"""
    xs = orc.XorShiftWide()
    return [xs.draw(pk.rng_draws) for _ in range(count)]


def _same_key(jobs):
    j0 = jobs[0]
    for j in jobs[1:]:
        assert all(np.array_equal(a, b) for a, b in zip(j0.fixed, j.fixed))
        assert np.array_equal(j0.map_col, j.map_col) and np.array_equal(j0.map_row, j.map_row)
        assert j.transcript_repr == j0.transcript_repr


def _singles(pk, jobs, insts, wides, tr):
    return [pk.create_proof(j.advice, inst, w, tr) for j, inst, w in zip(jobs, insts, wides)]


def _dev_batch(backend, pk, jobs, insts, wides, tr):
    d_adv = [backend.to_device(np.concatenate([np.ascontiguousarray(a).reshape(-1, 4) for a in j.advice])) for j in jobs]
    d_rng = [backend.to_device(w) for w in wides]
    try:
        return pk.create_proofs_dev(d_adv, insts, d_rng, tr)
    finally:
        for d in d_adv + d_rng:
            d.free()


def _raw_batch(zk, pk, jobs, insts, wides, tr, count=None, cap=None, null_rng=False):
    """b200zk_create_proofs called directly: (return code, status, proofs buffer)"""
    count = len(jobs) if count is None else count
    adv = [np.ascontiguousarray(a, dtype=np.uint64).reshape(pk.n, 4) for j in jobs for a in j.advice]
    inst = [c if c.shape[0] else np.zeros((1, 4), dtype=np.uint64) for i in insts for c in i]
    lens = np.array([c.shape[0] for i in insts for c in i], dtype=np.uint32)
    out = np.zeros(max(len(jobs), 1) * pk.proof_size, dtype=np.uint8)
    status = np.full(max(len(jobs), 1), 7, dtype=np.int32)
    P = lambda arrs: (ctypes.c_void_p * max(len(arrs), 1))(*[a.ctypes.data for a in arrs])
    rng = P(wides)
    if null_rng:
        rng[len(wides) - 1] = None
    rc = zk.lib().b200zk_create_proofs(pk._h, ctypes.c_uint32(count), P(adv), P(inst), lens.ctypes.data_as(ctypes.c_void_p), rng,
                                       np.ascontiguousarray(tr).ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p),
                                       ctypes.c_size_t(out.nbytes if cap is None else cap), status.ctypes.data_as(ctypes.c_void_p))
    return rc, status, out


@pytest.mark.parametrize("name,k", [("small", 5), ("mst_shaped", 9), ("v3_shaped", 11), ("generic_shapes", 10)])
def test_synthetic_shapes(zk, backend, orc, name, k):
    """A batch of 5 (different witnesses where the shape keeps its fixed columns across seeds, different rng streams
    always) equals create_proof proof by proof, from host and device inputs; proof 2 also equals the oracle's proof, and
    every proof verifies."""
    make = getattr(_synth(zk), name)
    jobs = [make(k, seed=4 + i) for i in range(5)] if name == "generic_shapes" else [make(k)] * 5
    _same_key(jobs)
    s, params, pk = _key(zk, backend, orc, jobs[0])
    insts, tr = _inputs(orc, jobs)
    wides = _streams(orc, pk, 5)
    l0 = backend.launch_count()
    singles = _singles(pk, jobs, insts, wides, tr)
    l1 = backend.launch_count()
    assert len(set(singles)) == 5
    assert pk.create_proofs([j.advice for j in jobs], insts, wides, tr) == singles
    assert backend.launch_count() - l1 >= l1 - l0                  # every lane's launches are counted on the pk's ctx
    assert _dev_batch(backend, pk, jobs, insts, wides, tr) == singles
    g, gl = params.read()
    want, _ = OP.create_proof(g, gl, OP.keygen_pk(jobs[2].cs, k, jobs[2].fixed, jobs[2].map_col, jobs[2].map_row), jobs[2].advice,
                              jobs[2].instances, wides[2], jobs[2].transcript_repr)
    assert singles[2] == want
    fixed_c, sigma_c = pk.vk_commitments()
    vk = zk.VerifyingKey(jobs[0].cs, k, fixed_c, sigma_c, g[0], zk.g2_mul(s))
    assert all(vk.verify_proof(inst, p, tr) for inst, p in zip(insts, singles))
    pk.close(); params.close()


def _mst_jobs(zk):
    jobs = [_chips(zk).merkle_sum_tree_job(9, levels=5, seed=s) for s in (1, 2, 3, 4)]
    _same_key(jobs)
    return jobs


def test_real_mst_k9_lanes(zk, backend, orc):
    """The reference's Merkle Sum Tree circuit at k = 9: four different users' witnesses under one pk, 7 proofs (more
    proofs than lanes, and not a multiple of them) on 1, 2 and 4 lanes, host and device inputs."""
    base = _mst_jobs(zk)
    jobs = [base[i % 4] for i in range(7)]
    s, params, pk = _key(zk, backend, orc, jobs[0])
    insts, tr = _inputs(orc, jobs)
    wides = _streams(orc, pk, 7)
    singles = _singles(pk, jobs, insts, wides, tr)
    for lanes in (1, 2, 4):
        assert pk.reserve_lanes(lanes) == lanes
        assert pk.create_proofs([j.advice for j in jobs], insts, wides, tr) == singles, lanes
        assert _dev_batch(backend, pk, jobs, insts, wides, tr) == singles, lanes
    g, _ = params.read()
    fixed_c, sigma_c = pk.vk_commitments()
    vk = zk.VerifyingKey(jobs[0].cs, 9, fixed_c, sigma_c, g[0], zk.g2_mul(s))
    assert all(vk.verify_proof(inst, p, tr) for inst, p in zip(insts, singles))
    pk.close(); params.close()


@pytest.mark.parametrize("name", ["small_k5", "mst_k9"])
def test_golden_vectors_inside_a_batch(zk, backend, orc, name):
    """The committed golden vectors at positions 1 and 3 of a batch of 4 on 2 lanes give their committed proof bytes."""
    gold = importlib.import_module("tests.golden.make_golden")
    tv = importlib.import_module("tests.test_verifier")
    z, vk, inst, want = tv.load_golden(zk, name)
    job = _synth(zk).small(5) if name == "small_k5" else gold.mst_k9_job(zk)
    s = orc.random_fr(1, int(z["seed_s"]))[0]
    params = zk.ParamsKZG.setup(backend, job.k, s)
    pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    assert pk.reserve_lanes(2) == 2
    wides = _streams(orc, pk, 3)                                      # wides[0] is the golden stream
    order = [wides[1], wides[0], wides[2], wides[0]]
    got = pk.create_proofs([job.advice] * 4, [inst] * 4, order, z["transcript_repr"])
    assert got[1] == want and got[3] == want and hashlib.sha256(got[1]).hexdigest() == tv.SHA[name]
    assert got[0] != want and got[2] != want
    assert all(vk.verify_proof(inst, p, z["transcript_repr"]) for p in got)
    pk.close(); params.close()


def test_failing_witness_in_the_middle(zk, backend, orc):
    """Proof 3 has a lookup input that is not in the table: the call returns ESYNTH, status[3] is ESYNTH, and every
    other proof is its single-call proof."""
    job = _synth(zk).small(6)
    bad = _synth(zk).small(6)
    byte_col = 5 + 3 + 2
    col = np.array(bad.advice[byte_col]); col[3] = orc.ints_to_mont([100000])[0]; bad.advice[byte_col] = col
    jobs = [job, job, job, bad, job, job]
    s, params, pk = _key(zk, backend, orc, job)
    insts, tr = _inputs(orc, jobs)
    wides = _streams(orc, pk, 6)
    with pytest.raises(zk.B200zkError, match="-5"):
        pk.create_proof(bad.advice, insts[3], wides[3], tr)
    singles = [None if i == 3 else pk.create_proof(j.advice, inst, w, tr) for i, (j, inst, w) in enumerate(zip(jobs, insts, wides))]
    assert pk.reserve_lanes(3) == 3
    rc, status, out = _raw_batch(zk, pk, jobs, insts, wides, tr)
    assert rc == zk.ESYNTH and list(status) == [0, 0, 0, zk.ESYNTH, 0, 0]
    assert "proof 3" in zk.lib().b200zk_last_error(backend._ctx).decode()
    assert [None if st else bytes(out[i * pk.proof_size:(i + 1) * pk.proof_size]) for i, st in enumerate(status)] == singles
    assert pk.create_proofs([j.advice for j in jobs], insts, wides, tr) == singles
    assert _dev_batch(backend, pk, jobs, insts, wides, tr) == singles
    assert pk.create_proof(job.advice, insts[0], wides[0], tr) == singles[0]        # the pk stays usable
    pk.close(); params.close()


def test_lookup_cosets_early_and_late(zk, backend, orc, monkeypatch):
    """Proving keys built with the lookup cosets computed early and late give the same batch bytes."""
    jobs = [_synth(zk).mst_shaped(9)] * 3
    got = []
    for early in ("0", "1"):
        monkeypatch.setenv("B200ZK_LOOKUP_EARLY", early)
        s, params, pk = _key(zk, backend, orc, jobs[0])
        insts, tr = _inputs(orc, jobs)
        wides = _streams(orc, pk, 3)
        got.append(pk.create_proofs([j.advice for j in jobs], insts, wides, tr))
        assert got[-1][1] == pk.create_proof(jobs[1].advice, insts[1], wides[1], tr)
        pk.close(); params.close()
    assert got[0] == got[1] and len(set(got[0])) == 3


def test_lanes_that_cannot_get_memory(zk, backend, orc, monkeypatch):
    """A lane whose allocation fails is dropped: the batch runs on fewer lanes with the right bytes, and the failed
    allocation leaves no CUDA error behind for the proofs that run next on the calling thread.  B200ZK_LANE_ALLOC_LIMIT
    makes the lanes' allocations fail the way they fail on an exhausted device, without filling the GPU."""
    job = _chips(zk).merkle_sum_tree_job(9, levels=5, seed=1)
    s, params, pk = _key(zk, backend, orc, job)
    insts, tr = _inputs(orc, [job] * 6)
    wides = _streams(orc, pk, 6)
    singles = _singles(pk, [job] * 6, insts, wides, tr)
    monkeypatch.setenv("B200ZK_LANE_ALLOC_LIMIT", "1")
    assert pk.create_proofs([job.advice] * 6, insts, wides, tr) == singles        # the batch plans lanes, none can be made
    assert pk.reserve_lanes(4) == 1
    assert pk.create_proof(job.advice, insts[1], wides[1], tr) == singles[1]
    monkeypatch.delenv("B200ZK_LANE_ALLOC_LIMIT")
    assert pk.reserve_lanes(2) == 2
    monkeypatch.setenv("B200ZK_LANE_ALLOC_LIMIT", "1")                          # lane 1 holds more than that: lanes 2, 3 fail
    assert pk.reserve_lanes(4) == 2
    assert pk.create_proofs([job.advice] * 6, insts, wides, tr) == singles
    assert _dev_batch(backend, pk, [job] * 6, insts, wides, tr) == singles
    assert pk.create_proof(job.advice, insts[2], wides[2], tr) == singles[2]
    pk.close(); params.close()


def _debug_names(zk, pk):
    names = ["advice_values", "advice_polys", "lookups", "perm_polys", "h", "rnd", "tmp_n", "advice_cosets", "h_poly"]
    out = {}
    for nm in names:
        cnt = ctypes.c_size_t()
        buf = np.zeros((4, 4), dtype=np.uint64)
        assert zk.lib().b200zk_pk_debug_buffer(pk._h, nm.encode(), buf.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(4), ctypes.byref(cnt)) == 0, nm
        out[nm] = (cnt.value, buf.tobytes())
    return out


def test_single_batch_single(zk, backend, orc):
    """A batch between two single calls on one pk leaves the single calls' bytes, phase keys, trace labels and debug
    buffers as they were."""
    job = _synth(zk).mst_shaped(9)
    s, params, pk = _key(zk, backend, orc, job)
    insts, tr = _inputs(orc, [job] * 5)
    wides = _streams(orc, pk, 5)
    first = pk.create_proof(job.advice, insts[0], wides[0], tr)
    phase, labels, dbg = pk.last_phase_ms().keys(), [a for a, _ in pk.last_trace()], _debug_names(zk, pk)
    batch = pk.create_proofs([job.advice] * 5, insts, wides, tr)
    assert batch[0] == first
    assert pk.last_phase_ms().keys() == phase and [a for a, _ in pk.last_trace()] == labels
    again = pk.create_proof(job.advice, insts[0], wides[0], tr)
    assert again == first
    assert pk.last_phase_ms().keys() == phase and [a for a, _ in pk.last_trace()] == labels and _debug_names(zk, pk) == dbg
    pk.close(); params.close()


def test_bad_arguments(zk, backend, orc):
    """count == 0, a null rng stream, a buffer smaller than count * proof_size and a pk on a sharded rank's ctx are
    refused before any work; the pk proves correctly afterwards."""
    job = _synth(zk).small(5)
    s, params, pk = _key(zk, backend, orc, job)
    insts, tr = _inputs(orc, [job] * 2)
    wides = _streams(orc, pk, 2)
    singles = _singles(pk, [job] * 2, insts, wides, tr)
    l0 = backend.launch_count()
    assert _raw_batch(zk, pk, [job] * 2, insts, wides, tr, count=0)[0] == zk.EINVAL
    assert _raw_batch(zk, pk, [job] * 2, insts, wides, tr, null_rng=True)[0] == zk.EINVAL
    assert _raw_batch(zk, pk, [job] * 2, insts, wides, tr, cap=2 * pk.proof_size - 1)[0] == zk.EINVAL
    assert backend.launch_count() == l0
    with pytest.raises(zk.B200zkError):
        pk.create_proofs([job.advice] * 2, insts[:1], wides, tr)
    with pytest.raises(zk.B200zkError):
        pk.create_proofs([job.advice] * 2, insts, [wides[0], wides[1][:10]], tr)
    group = zk.Group([0, 0])
    try:
        gparams = zk.ParamsKZG.setup(group.backends[0], job.k, s)
        gpk = zk.ProvingKey(gparams, job.cs, job.k, job.fixed, job.map_col, job.map_row)
        with pytest.raises(zk.B200zkError, match="sharded"):
            gpk.create_proofs([job.advice] * 2, insts, wides, tr)
        with pytest.raises(zk.B200zkError, match="sharded"):
            gpk.reserve_lanes(2)
        gpk.close(); gparams.close()
    finally:
        group.close()
    rc, status, out = _raw_batch(zk, pk, [job] * 2, insts, wides, tr)
    assert rc == 0 and list(status) == [0, 0]
    assert [bytes(out[i * pk.proof_size:(i + 1) * pk.proof_size]) for i in range(2)] == singles
    assert pk.create_proof(job.advice, insts[1], wides[1], tr) == singles[1]
    pk.close(); params.close()


def test_full_size_mst_k20_two_lanes(zk, backend, orc):
    """The headline circuit at k = 20: a batch of 2 on 2 lanes gives, at proof 0, the committed digest of the oracle's
    proof (tests/golden/full_size_sha256.json), and at proof 1 the single-call proof of its own rng stream."""
    gold = importlib.import_module("tests.golden.make_full_size_digests")
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full_size_sha256.json")
    want = json.load(open(path)).get("mst_k20")
    if want is None:
        pytest.skip("no committed digest for mst_k20 (run tests/golden/make_full_size_digests.py mst_k20)")
    job = gold.build_job(zk, "mst_k20")
    params = zk.ParamsKZG.setup(backend, job.k, orc.random_fr(1, gold.SEED_S)[0])
    pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    try:                                                              # 9 GiB of key and 17 GiB per lane: never left to the collector
        insts, tr = _inputs(orc, [job] * 2)
        wides = _streams(orc, pk, 2)
        assert pk.reserve_lanes(2) == 2
        got = pk.create_proofs([job.advice] * 2, insts, wides, tr)
        assert len(got[0]) == want["proof_bytes"]
        assert hashlib.sha256(got[0]).hexdigest() == want["sha256"]
        assert got[1] == pk.create_proof(job.advice, insts[1], wides[1], tr)
    finally:
        pk.close(); params.close()
