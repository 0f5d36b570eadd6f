#!/usr/bin/env python
"""Time of b200zk_pairing_checks (many pairing-product checks on the device) and of verify_proofs, whose pairing checks it
now runs, next to one host b200zk_pairing_check.

    python tools/pairing_bench.py [--counts 1,16,256,4096,65536] [--work mst9,v3_14] [--reps 3] [--out FILE]

pairing_checks: 2-pair checks e(aP, bQ) e(-abP, Q), every eighth one false, tiled from a pool of 64 distinct checks
(two distinct G2 points per call, as verify_proofs and accumulator piles have).  verify_proofs: the workloads of
tools/verify_batch_bench.py at N = 1, 1 024 and 4 096, and at 1 024 with 1 and with 64 tampered proofs (a flipped
evaluation: it passes stage 1 and fails the pairing).  One warm-up call, then the median of --reps calls, a host clock
around each call (both calls synchronise their stream before they return).  The card's name and power limit are read
in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from proof_batch_bench import card, median  # noqa: E402
from verify_batch_bench import make_proofs  # noqa: E402


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return median(ts), out


def check_pool(n):
    from tests import pairing_ref as P
    rng = np.random.default_rng(1)
    q1, qb = P.g2_mul([1, 77])
    g1, g2, truth = [], [], []
    for j in range(n):
        a = int(rng.integers(1, 2**60))
        ok = j % 8 != 5
        g1 += [P.g1_mul([a])[0], P.g1_neg(P.g1_mul([a * 77 + (0 if ok else 1)]))[0]]
        g2 += [qb, q1]
        truth.append(ok)
    return np.array(g1), np.array(g2), truth


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--counts", default="1,16,256,4096,65536")
    ap.add_argument("--work", default="mst9,v3_14")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_pairing_bench.json"))
    a = ap.parse_args()
    from __graft_entry__ import load_package
    zk = load_package()
    backend = zk.Backend(0)
    res = {"card": card(), "cpu_count": os.cpu_count(), "reps": a.reps, "results": []}

    def emit(line):
        print(json.dumps(line), flush=True)
        res["results"].append(line)

    try:
        g1p, g2p, truth = check_pool(64)
        t, ok = timed(lambda: zk.pairing_check(g1p[:2], g2p[:2]), a.reps)
        assert ok == truth[0]
        emit({"call": "pairing_check (host)", "m": 2, "count": 1, "ms": 1e3 * t})
        for n in [int(x) for x in a.counts.split(",")]:
            idx = np.arange(n) % 64
            g1 = g1p.reshape(64, 2, 8)[idx].reshape(-1, 8)
            g2 = g2p.reshape(64, 2, 16)[idx].reshape(-1, 16)
            t, st = timed(lambda: zk.pairing_checks(backend, g1, g2, 2), a.reps)
            assert list(st == 0) == [truth[i] for i in idx]
            emit({"call": "pairing_checks", "m": 2, "count": n, "ms": 1e3 * t, "checks_per_s": n / t})
        for name in a.work.split(","):
            vk, insts, proofs, tr = make_proofs(zk, backend, name, 4096)
            for n in (1, 1024, 4096):
                t, ok = timed(lambda: vk.verify_proofs(backend, insts[:n], proofs[:n], tr), a.reps)
                assert all(ok)
                emit({"work": name, "call": "verify_proofs", "n": n, "ms": 1e3 * t, "proofs_per_s": n / t})
            for nbad in (1, 64):
                bad_idx = set(range(517, 1024, 8)[:nbad]) if nbad > 1 else {517}
                bad = [bytes(bytearray(p[:-96]) + bytes([p[-96] ^ 1]) + p[-95:]) if i in bad_idx else p for i, p in enumerate(proofs[:1024])]
                l0 = backend.launch_count()
                t, ok = timed(lambda: vk.verify_proofs(backend, insts[:1024], bad, tr), a.reps)
                launches = (backend.launch_count() - l0) // (a.reps + 1)
                assert ok == [i not in bad_idx for i in range(1024)]
                emit({"work": name, "call": f"verify_proofs, {nbad} tampered", "n": 1024, "ms": 1e3 * t, "launches": launches})
    finally:
        backend.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f)
        f.write("\n")
    print(json.dumps(res["card"]), "cpu_count", res["cpu_count"])


if __name__ == "__main__":
    main()
