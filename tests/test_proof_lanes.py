"""CPU: the lane planner of b200zk_create_proofs (csrc/proof_lanes.hpp, compiled on the host through
tests/proof_lanes_harness.cpp): at least one lane, never more than the batch, the request or the memory share allows,
and B200ZK_PROOF_LANES replaces the request."""
import ctypes
import hashlib
import itertools
import os
import subprocess
import tempfile

import pytest

_HARNESS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "proof_lanes_harness.cpp")
_HEADER = os.path.join(os.path.dirname(_HARNESS), "..", "halo2-experiments_b200", "csrc", "proof_lanes.hpp")
GIB = 1 << 30


@pytest.fixture(scope="module")
def planner():
    """Built with the host compiler into a temporary directory (the tree may be read-only)."""
    h = hashlib.sha256()
    for f in (_HARNESS, _HEADER):
        h.update(open(f, "rb").read())
    so = os.path.join(tempfile.gettempdir(), f"proof_lanes_harness_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = so + f".{os.getpid()}"
        subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", tmp, _HARNESS])
        os.replace(tmp, so)
    lib = ctypes.CDLL(so)
    lib.plan_lanes_c.restype = ctypes.c_uint32
    lib.plan_lanes_c.argtypes = [ctypes.c_uint32, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint32]
    lib.lanes_default_cap.restype = ctypes.c_uint32
    lib.lanes_max.restype = ctypes.c_uint32
    return lib


def plan(lib, count, want=0, env=None, free=100 * GIB, per_lane=GIB, have=0):
    return lib.plan_lanes_c(count, want, None if env is None else env.encode(), free, per_lane, have)


def test_bounds_over_a_grid(planner):
    cap, mx = planner.lanes_default_cap(), planner.lanes_max()
    for count, want, free_gib, per_gib, have in itertools.product([0, 1, 2, 3, 7, 64, 1000], [0, 1, 2, 4, 8, 100], [0, 1, 3, 16, 170],
                                                                    [1, 2, 9], [0, 1, 3]):
        n = plan(planner, count, want, None, free_gib * GIB, per_gib * GIB, have)
        assert n >= 1
        if count:
            assert n <= count
        assert n <= (want or cap) and n <= mx
        assert n - 1 <= have + (free_gib * GIB // 2) // (per_gib * GIB)      # extra lanes: those that exist + half the free memory


def test_default_and_request(planner):
    cap = planner.lanes_default_cap()
    assert plan(planner, 64) == cap
    assert plan(planner, 0) == cap                 # a reservation without a batch
    assert plan(planner, 2) == 2
    assert plan(planner, 64, want=8) == 8
    assert plan(planner, 7, want=4) == 4
    assert plan(planner, 64, want=1) == 1


def test_memory_limits_but_never_below_one(planner):
    assert plan(planner, 64, want=8, free=6 * GIB, per_lane=GIB) == 4        # 3 extra lanes fit in half of 6 GiB
    assert plan(planner, 64, want=8, free=GIB, per_lane=2 * GIB) == 1
    assert plan(planner, 64, want=8, free=0, per_lane=GIB) == 1
    assert plan(planner, 64, want=8, free=0, per_lane=GIB, have=2) == 3      # lanes that exist already hold their memory


def test_environment_override_wins(planner):
    assert plan(planner, 64, want=2, env="6") == 6
    assert plan(planner, 64, env="1") == 1
    assert plan(planner, 3, want=2, env="6") == 3                # still no more than the batch
    assert plan(planner, 64, want=8, env="6", free=2 * GIB, per_lane=GIB) == 2     # nor than memory
    for bad in ["", "0", "-3", "four", "2x"]:
        assert plan(planner, 64, want=2, env=bad) == 2            # ignored
    assert plan(planner, 1000, env="100000", per_lane=1 << 20) == planner.lanes_max()
