"""arithmetic::g_to_lagrange on the CPU: the restatement of upstream's FFT form (tests/g1_ntt_harness.cpp) against the
direct formula of ParamsKZG::setup, and the host-emulated per-thread bodies of csrc/g1_ntt.cuh against the restatement."""
import numpy as np
import pytest

from tests import g1_ntt_ref as H

R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001


def edge_bases(orc, k, seed):
    """2^k points: random multiples of the generator, plus (where they fit) the identity, a repeated point and a
    P / -P pair."""
    n = 1 << k
    sc = orc.random_fr(n, seed)
    ints = orc.mont_to_ints(sc)
    if n >= 4:
        ints[1] = ints[0]                       # repeated point
        ints[3] = (R_MOD - ints[2]) % R_MOD     # P, -P
    if n >= 8:
        ints[5] = 0                             # identity
    elif n >= 2:
        ints[n - 1] = 0
    g = orc.g1_fixed_base_mul(orc.ints_to_mont(ints))
    if n >= 2:
        assert not g[n - 1 if n < 8 else 5].any()
    return g


@pytest.mark.parametrize("k", range(1, 9))
def test_reference_fft_equals_setup_formula(orc, k):
    s = orc.random_fr(1, 100 + k)[0]
    g, gl = orc.params_setup(k, s)
    assert np.array_equal(H.g_to_lagrange(g, k), gl)


@pytest.mark.parametrize("k", range(0, 7))
def test_emulated_bodies_equal_reference(orc, k):
    g = edge_bases(orc, k, 200 + k)
    want = H.g_to_lagrange(g, k)
    assert orc.g1_on_curve(want)
    assert np.array_equal(H.g_to_lagrange_emu(g, k), want)


def test_emulated_transform_of_identities_and_k0(orc):
    assert not H.g_to_lagrange_emu(np.zeros((8, 8), dtype=np.uint64), 3).any()
    g = orc.g1_fixed_base_mul(orc.random_fr(1, 7))
    assert np.array_equal(H.g_to_lagrange_emu(g, 0), g)


def test_emulated_xyzz_mul_equals_reference(orc):
    ints = [0, 1, R_MOD - 1, R_MOD - 2] + [1 << j for j in (1, 3, 4, 7, 8, 63, 64, 127, 200, 253)]
    ints += orc.mont_to_ints(orc.random_fr(12, 31))
    ints += [0xF7F7F7F7F7F7F7F7F7F7F7F7F7F7F7F7, 0x88888888888888888888888888888888]      # signed-digit carries
    pts = orc.g1_fixed_base_mul(orc.random_fr(len(ints), 32))
    pts[5] = 0                                                                             # identity * s
    got = H.xyzz_mul(pts, orc.ints_to_raw(ints))
    mont = orc.ints_to_mont(ints)
    want = orc.g1_batch_normalize(np.stack([orc.g1_mul(orc.g1_from_affine(p), s) for p, s in zip(pts, mont)]))
    assert np.array_equal(got, want)
