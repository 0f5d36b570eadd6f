"""GPU: g_to_lagrange and ParamsKZG::downsize (csrc/g1_ntt.cuh, g_to_lagrange_run in csrc/setup.cu) against the
Lagrange basis of a direct setup, against the CPU restatement of upstream's g_to_lagrange for arbitrary bases, and
end to end through proofs made with downsized params."""
import hashlib
import importlib

import numpy as np
import pytest

from tests import g1_ntt_ref as H
from tests.test_lagrange_basis import edge_bases

pytestmark = pytest.mark.gpu


def _secret(orc, seed):
    return orc.random_fr(1, seed)[0]


@pytest.mark.parametrize("k", [1, 2, 5, 11, 12, 16, 20])
def test_g_to_lagrange_equals_setup_basis(zk, backend, orc, k):
    params = zk.ParamsKZG.setup(backend, k, _secret(orc, 500 + k))
    g, gl = params.read()
    params.close()
    assert np.array_equal(zk.g_to_lagrange(backend, g, k), gl)
    d_g, d_out = backend.to_device(g), backend.alloc(g.nbytes)
    try:
        backend.g_to_lagrange_dev(d_g, k, d_out)
        assert np.array_equal(d_out.download(g.shape), gl)
    finally:
        d_g.free(); d_out.free()


@pytest.mark.parametrize("k", [0, 4, 10, 13])
def test_g_to_lagrange_arbitrary_bases(zk, backend, orc, k):
    g = edge_bases(orc, k, 600 + k)
    want = H.g_to_lagrange(g, k)
    assert np.array_equal(zk.g_to_lagrange(backend, g, k), want)
    d_g = backend.to_device(g)
    try:
        backend.g_to_lagrange_dev(d_g, k, d_g)                             # out aliases g
        assert np.array_equal(d_g.download(g.shape), want)
    finally:
        d_g.free()


@pytest.mark.parametrize("K,k", [(8, 5), (12, 9), (22, 20), (9, 9)])
def test_downsize_equals_direct_setup(zk, backend, orc, K, k):
    s = _secret(orc, 700 + K)
    big = zk.ParamsKZG.setup(backend, K, s)
    before = big.read()
    poly = orc.random_fr(1 << K, 701)
    c_before = big.commit_lagrange(poly)
    small = big.downsize(k)
    direct = zk.ParamsKZG.setup(backend, k, s)
    try:
        for a, b in zip(small.read(), direct.read()):
            assert np.array_equal(a, b)
        for a, b in zip(big.read(), before):
            assert np.array_equal(a, b)
        assert np.array_equal(big.commit_lagrange(poly), c_before)
        g2, s_g2 = zk.g2_mul(np.array(zk._FR_ONE, dtype=np.uint64)), zk.g2_mul(s)
        assert small.to_bytes(g2, s_g2) == direct.to_bytes(g2, s_g2)
    finally:
        small.close(); direct.close(); big.close()


def test_downsize_gives_loaded_params_their_lagrange_basis(zk, backend, orc):
    job = importlib.import_module(zk.__name__ + ".circuits_synth").small(5)
    s = _secret(orc, 77)
    g, _ = orc.params_setup(job.k, s, with_lagrange=False)
    loaded = zk.ParamsKZG.load(backend, job.k, g, None)
    with pytest.raises(zk.B200zkError):
        zk.ProvingKey(loaded, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    params = loaded.downsize(job.k)
    pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    ref = zk.ParamsKZG.setup(backend, job.k, s)
    ref_pk = zk.ProvingKey(ref, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    try:
        for a, b in zip(pk.vk_commitments(), ref_pk.vk_commitments()):
            assert np.array_equal(a, b)
    finally:
        pk.close(); ref_pk.close(); params.close(); ref.close(); loaded.close()


@pytest.mark.parametrize("name", ["small_k5", "mst_k9"])
def test_golden_vectors_through_downsized_params(zk, backend, orc, name):
    """test_golden_vectors with params = setup(k + 3, s).downsize(k): the same commitments and proof bytes, the proof
    verifies, and a 2-rank group whose ranks downsize their own params gives the same bytes."""
    gold = importlib.import_module("tests.golden.make_golden")
    tv = importlib.import_module("tests.test_verifier")
    z, vk, inst, want = tv.load_golden(zk, name)
    job = importlib.import_module(zk.__name__ + ".circuits_synth").small(5) if name == "small_k5" else gold.mst_k9_job(zk)
    s = orc.random_fr(1, int(z["seed_s"]))[0]
    big = zk.ParamsKZG.setup(backend, job.k + 3, s)
    params = big.downsize(job.k)
    big.close()
    pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
    fixed_c, sigma_c = pk.vk_commitments()
    assert np.array_equal(fixed_c, z["fixed_commitments"]) and np.array_equal(sigma_c, z["sigma_commitments"])
    wide = orc.XorShiftWide().draw(pk.rng_draws)
    got = pk.create_proof(job.advice, inst, wide, z["transcript_repr"])
    assert got == want and hashlib.sha256(got).hexdigest() == tv.SHA[name]
    assert vk.verify_proof(inst, got, z["transcript_repr"])
    pk.close(); params.close()
    group = zk.Group([0, 0])
    try:
        bigs = [zk.ParamsKZG.setup(b, job.k + 3, s) for b in group.backends]
        gparams = [p.downsize(job.k) for p in bigs]
        gpks = [zk.ProvingKey(p, job.cs, job.k, job.fixed, job.map_col, job.map_row) for p in gparams]
        assert group.create_proof(gpks, job.advice, inst, wide, z["transcript_repr"]) == want
        for x in gpks + gparams + bigs:
            x.close()
    finally:
        group.close()


def test_invalid_arguments_raise_and_leave_the_context_usable(zk, backend, orc):
    s = _secret(orc, 900)
    params = zk.ParamsKZG.setup(backend, 6, s)
    try:
        with pytest.raises(zk.B200zkError, match="params_downsize"):
            params.downsize(7)
        with pytest.raises(zk.B200zkError, match="params_downsize"):
            params.downsize(29)
        with pytest.raises(zk.B200zkError, match="g_to_lagrange"):
            backend.g_to_lagrange_dev(None, 3, None)
        d = backend.alloc(64 << 3)
        try:
            with pytest.raises(zk.B200zkError, match="g_to_lagrange"):
                backend.g_to_lagrange_dev(d, 29, d)
        finally:
            d.free()
        with pytest.raises(zk.B200zkError):
            zk.ParamsKZG(backend, None, 6).downsize(3)
        g, gl = params.read()
        assert np.array_equal(zk.g_to_lagrange(backend, g, 6), gl)
        small = params.downsize(4)
        assert np.array_equal(small.read()[1], orc.params_setup(4, s)[1])
        small.close()
    finally:
        params.close()
