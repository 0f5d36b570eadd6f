"""ctypes binding over tests/pairing_harness.cpp: the host-emulated pairing bodies of csrc/pairing.cuh next to the host
pairing of csrc/pairing.hpp.  The shared object is built with the host compiler into a temporary directory (the tree may
be read-only).  Fq values are 4 x u64 Montgomery limbs; an Fq2 is (n, 8) uint64, an Fq12 (n, 48), a line (n, 24), a
G1Affine (n, 8) and a G2Affine (n, 16)."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_HARNESS = os.path.join(ROOT, "tests", "pairing_harness.cpp")
_CSRC = os.path.join(ROOT, "halo2-experiments_b200", "csrc")
_lib = None

Q = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001


def lib():
    global _lib
    if _lib is not None:
        return _lib
    deps = [_HARNESS] + sorted(os.path.join(_CSRC, x) for x in os.listdir(_CSRC) if x.endswith((".cuh", ".hpp", ".inc")))
    h = hashlib.sha256()
    for f in deps:
        h.update(open(f, "rb").read())
    so = os.path.join(tempfile.gettempdir(), f"pairing_harness_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = so + f".{os.getpid()}"
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-w", "-o", tmp, _HARNESS])
        os.replace(tmp, so)
    _lib = ctypes.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def mont(v):
    """Montgomery limbs (4 x u64) of the integer v mod q."""
    m = (v << 256) % Q
    return [(m >> (64 * j)) & (2**64 - 1) for j in range(4)]


def limbs(v, n=4):
    return [(v >> (64 * j)) & (2**64 - 1) for j in range(n)]


def rand_fq(rng, n, words):
    """(n, 4 * words) uint64 of uniformly random Fq values (Montgomery form)."""
    return np.array([sum((mont(int.from_bytes(rng.bytes(40), "little") % Q) for _ in range(words)), []) for _ in range(n)],
                    dtype=np.uint64).reshape(n, 4 * words)


def fq2(op, a, b=None, which=0):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = a if b is None else np.ascontiguousarray(b, dtype=np.uint64)
    out = np.zeros_like(a)
    lib().ph_fq2(ctypes.c_int(op), _p(a), _p(b), _p(out), ctypes.c_size_t(a.shape[0]), ctypes.c_int(which))
    return out


FQ12_OPS = {"mul": 0, "sqr": 1, "inv": 2, "cyc_sqr": 3, "easy": 4, "final_exp": 5, "frob1": 6, "frob2": 7, "frob3": 8}


def fq12(op, a, b=None, which=0):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    b = a if b is None else np.ascontiguousarray(b, dtype=np.uint64)
    out = np.zeros_like(a)
    lib().ph_fq12(ctypes.c_int(FQ12_OPS[op]), _p(a), _p(b), _p(out), ctypes.c_size_t(a.shape[0]), ctypes.c_int(which))
    return out


def fq12_pow(a, e):
    """a^e on the host by square-and-multiply, e a non-negative integer."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    n = max(1, (e.bit_length() + 63) // 64)
    ev = np.array(limbs(e, n), dtype=np.uint64)
    out = np.zeros_like(a)
    lib().ph_fq12_pow(_p(a), _p(ev), ctypes.c_size_t(n), _p(out), ctypes.c_size_t(a.shape[0]))
    return out


def line(f, lines, p, which=0):
    f, lines, p = (np.ascontiguousarray(x, dtype=np.uint64) for x in (f, lines, p))
    out = np.zeros_like(f)
    lib().ph_line(_p(f), _p(lines), _p(p), _p(out), ctypes.c_size_t(f.shape[0]), ctypes.c_int(which))
    return out


def pairing(g1, g2, m, which=0):
    """(count, 48): prod_{i < m} e(g1[j m + i], g2[j m + i]) for every j, before the verdict."""
    g1 = np.ascontiguousarray(g1, dtype=np.uint64).reshape(-1, 8)
    g2 = np.ascontiguousarray(g2, dtype=np.uint64).reshape(-1, 16)
    count = g1.shape[0] // m
    out = np.zeros((count, 48), dtype=np.uint64)
    lib().ph_pairing(_p(g1), _p(g2), ctypes.c_uint32(m), ctypes.c_size_t(count), _p(out), ctypes.c_int(which))
    return out


def g1_mul(scalars):
    s = np.array([limbs(x % R) for x in scalars], dtype=np.uint64)
    out = np.zeros((len(scalars), 8), dtype=np.uint64)
    lib().ph_g1_mul(_p(s), _p(out), ctypes.c_size_t(len(scalars)))
    return out


def g2_mul(scalars):
    s = np.array([limbs(x % R) for x in scalars], dtype=np.uint64)
    out = np.zeros((len(scalars), 16), dtype=np.uint64)
    lib().ph_g2_mul(_p(s), _p(out), ctypes.c_size_t(len(scalars)))
    return out


def g1_neg(p):
    """-P for (n, 8) G1Affine (the identity stays)."""
    p = np.array(p, dtype=np.uint64).reshape(-1, 8).copy()
    for row in p:
        y = sum(int(row[4 + j]) << (64 * j) for j in range(4))
        row[4:] = limbs((Q - y) % Q)
    return p
