"""ctypes binding over tests/g1_ntt_harness.cpp: the host-emulated G1 NTT bodies of csrc/g1_ntt.cuh and the CPU
restatement of halo2_proofs' arithmetic::g_to_lagrange.  The shared object is built with the host compiler into a
temporary directory (the tree may be read-only).  Points are (n, 8) uint64 G1Affine arrays in Montgomery form."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_HARNESS = os.path.join(ROOT, "tests", "g1_ntt_harness.cpp")
_ORACLE = os.path.join(ROOT, "oracle")
_CSRC = os.path.join(ROOT, "halo2-experiments_b200", "csrc")
_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    srcs = [_HARNESS, os.path.join(_ORACLE, "arith.cpp")]
    deps = srcs + sorted(os.path.join(d, x) for d in (_CSRC, _ORACLE) for x in os.listdir(d) if x.endswith((".cuh", ".hpp")))
    h = hashlib.sha256()
    for f in deps:
        h.update(open(f, "rb").read())
    so = os.path.join(tempfile.gettempdir(), f"g1_ntt_harness_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = so + f".{os.getpid()}"
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-w",
                               "-o", tmp] + srcs)
        os.replace(tmp, so)
    _lib = ctypes.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _pts(g):
    return np.ascontiguousarray(g, dtype=np.uint64).reshape(-1, 8)


def xyzz_mul(points, scalars_canonical):
    """s[i] * p[i] through the emulated xyzz_mul; scalars as (n, 4) canonical (non-Montgomery) limbs."""
    p = _pts(points)
    s = np.ascontiguousarray(scalars_canonical, dtype=np.uint64).reshape(-1, 4)
    assert s.shape[0] == p.shape[0]
    out = np.zeros_like(p)
    lib().g1h_xyzz_mul(_p(p), _p(s), _p(out), ctypes.c_size_t(p.shape[0]))
    return out


def g_to_lagrange_emu(g, k):
    """The device's g_to_lagrange, its per-thread bodies run on the host in launch order."""
    g = _pts(g)
    assert g.shape[0] == 1 << k
    out = np.zeros_like(g)
    lib().g1h_g_to_lagrange_emu(_p(g), ctypes.c_uint32(k), _p(out))
    return out


def g_to_lagrange(g, k, threads=0):
    """arithmetic::g_to_lagrange restated on the CPU (threads = 0: all cores)."""
    g = _pts(g)
    assert g.shape[0] == 1 << k
    out = np.zeros_like(g)
    lib().g1h_g_to_lagrange_ref(_p(g), ctypes.c_uint32(k), _p(out), ctypes.c_int(threads))
    return out
