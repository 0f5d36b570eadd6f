#!/usr/bin/env python
"""Throughput of b200zk_verify_proofs (many proofs of one verifying key, one pairing check: AccumulatorStrategy) against a
loop of b200zk_verify_proof on the same proofs.

    python tools/verify_batch_bench.py [--work mst9,v3_14] [--sizes 1,16,64,256,1024,4096] [--reps 3] [--out FILE]

Workloads: the reference's Merkle Sum Tree circuit at k = 9 (5 levels; four users' witnesses) and the Merkle tree v3 at
k = 14.  The proofs are made with create_proofs, each with its own rng stream, so every proof of a batch is distinct.
Timed: a loop of verify_proof over 16 proofs, and verify_proofs at each size; one warm-up call, then the median of
--reps calls, a host clock around each call (verify_proofs synchronises its stream before it returns).  The draws of
verify_proofs come from os.urandom, as a caller's would.  One more line per workload times a batch of 1024 with one
tampered proof (a flipped evaluation: it passes stage 1 and fails the pairing), i.e. the cost of locating it.
The card's name and power limit and the host's CPU count are read in the same run.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from proof_batch_bench import card, job_for, median, mont  # noqa: E402


def make_proofs(zk, backend, name, count):
    """(vk, instances per proof, proofs, transcript_repr): count proofs of one key, distinct rng streams"""
    import importlib

    import numpy as np
    chips = importlib.import_module(zk.__name__ + ".chips")
    if name == "mst9":
        jobs = [chips.merkle_sum_tree_job(9, levels=5, seed=s) for s in (1, 2, 3, 4)]
    else:
        jobs = [job_for(zk, name)[0]]
    j0 = jobs[0]
    s = mont([987654321])[0]
    params = zk.ParamsKZG.setup(backend, j0.k, s)
    pk = zk.ProvingKey(params, j0.cs, j0.k, j0.fixed, j0.map_col, j0.map_row)
    tr = mont([j0.transcript_repr])[0]
    insts_of = [[mont(c) if len(c) else np.zeros((0, 4), dtype=np.uint64) for c in j.instances] for j in jobs]
    rng = np.random.Generator(np.random.PCG64(99))
    proofs, insts = [], []
    for lo in range(0, count, 256):
        m = min(256, count - lo)
        idx = [(lo + i) % len(jobs) for i in range(m)]
        wides = [rng.integers(0, 1 << 63, size=(pk.rng_draws, 8), dtype=np.uint64) for _ in range(m)]
        proofs += pk.create_proofs([jobs[i].advice for i in idx], [insts_of[i] for i in idx], wides, tr)
        insts += [insts_of[i] for i in idx]
    g, _ = params.read()
    fixed_c, sigma_c = pk.vk_commitments()
    vk = zk.VerifyingKey(j0.cs, j0.k, fixed_c, sigma_c, g[0], zk.g2_mul(s))
    pk.close(); params.close()
    assert all(p is not None for p in proofs) and len(set(proofs)) == count
    return vk, insts, proofs, tr


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        ts.append(time.perf_counter() - t0)
    return median(ts), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--work", default="mst9,v3_14")
    ap.add_argument("--sizes", default="1,16,64,256,1024,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_verify_batch_bench.json"))
    a = ap.parse_args()
    from __graft_entry__ import load_package
    zk = load_package()
    backend = zk.Backend(0)
    sizes = [int(x) for x in a.sizes.split(",")]
    res = {"card": card(), "cpu_count": os.cpu_count(), "reps": a.reps, "results": []}
    try:
        for name in a.work.split(","):
            vk, insts, proofs, tr = make_proofs(zk, backend, name, max(sizes + [16, 1024]))
            t, ok = timed(lambda: [vk.verify_proof(insts[i], proofs[i], tr) for i in range(16)], a.reps)
            assert all(ok)
            line = {"work": name, "proof_bytes": len(proofs[0]), "call": "verify_proof loop", "n": 16, "ms": 1e3 * t, "proofs_per_s": 16 / t}
            print(json.dumps(line), flush=True)
            res["results"].append(line)
            for n in sizes:
                t, ok = timed(lambda: vk.verify_proofs(backend, insts[:n], proofs[:n], tr), a.reps)
                assert all(ok)
                line = {"work": name, "call": "verify_proofs", "n": n, "ms": 1e3 * t, "proofs_per_s": n / t}
                print(json.dumps(line), flush=True)
                res["results"].append(line)
            bad = list(proofs[:1024])
            t = bytearray(bad[517]); t[len(t) - 96] ^= 1; bad[517] = bytes(t)
            t, ok = timed(lambda: vk.verify_proofs(backend, insts[:1024], bad, tr), a.reps)
            assert ok == [i != 517 for i in range(1024)]
            line = {"work": name, "call": "verify_proofs, proof 517 tampered", "n": 1024, "ms": 1e3 * t, "proofs_per_s": 1024 / t}
            print(json.dumps(line), flush=True)
            res["results"].append(line)
    finally:
        backend.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f)
        f.write("\n")
    print(json.dumps(res["card"]), "cpu_count", res["cpu_count"])


if __name__ == "__main__":
    main()
