#!/usr/bin/env python
"""Timing of arithmetic::g_to_lagrange and ParamsKZG::downsize on the GPU, against the work model of the G1 NTT and
against the CPU restatement of upstream's g_to_lagrange (tests/g1_ntt_harness.cpp) on the host cores.

    python tools/lagrange_bench.py [--ks 16,20,22] [--reps 3] [--cpu-k 16] [--out FILE]

Prints one JSON object.  g_to_lagrange_dev times come from device events around the call after one warm-up call at
the same k; its input is the `g` of ParamsKZG::setup(k).  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FQ_MUL_PER_S = 67.7e9           # DESIGN.md §2: the Fq multiplier at the IMAD.WIDE issue limit of one B200
DBL, ADD = 9, 14                # Fq multiplications of xyzz_dbl and xyzz_add (csrc/curve.cuh)
XYZZ_MUL = DBL + 6 * ADD + 252 * DBL + 64 * ADD   # table 1p..8p, 63 x 4 doublings, at most 64 window additions


def model_muls(k):
    """Fq multiplications of g_to_lagrange_run at 2^k points: (n/2)k - (n-1) butterflies with a scalar
    multiplication, every butterfly's two additions, and the n^-1 scaling of every point."""
    n = 1 << k
    nontrivial = (n // 2) * k - (n - 1)
    return nontrivial * XYZZ_MUL + (n // 2) * k * 2 * ADD + n * XYZZ_MUL, nontrivial


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--ks", default="16,20,22")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--downsize", default="22,20", help="K,k: downsize a 2^K SRS to k, end to end")
    ap.add_argument("--cpu-k", type=int, default=16, help="k of the CPU g_to_lagrange (0: skip)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from __graft_entry__ import load_package
    from oracle import binding as orc
    from tests import g1_ntt_ref as H
    import numpy as np
    zk = load_package()
    be = zk.Backend(0)
    res = {"card": card(), "fq_mul_per_s_bound": FQ_MUL_PER_S, "g_to_lagrange_dev": [], "model_fq_muls_per_scalar_mul": XYZZ_MUL}
    s = orc.random_fr(1, 2024)[0]
    try:
        for k in [int(x) for x in args.ks.split(",") if x]:
            params = zk.ParamsKZG.setup(be, k, s)
            g, gl = params.read()
            params.close()
            d_g, d_out = be.to_device(g), be.alloc(g.nbytes)
            be.g_to_lagrange_dev(d_g, k, d_out)                             # warm-up: workspace, twiddle tables
            ms = []
            for _ in range(args.reps):
                be.event_record(0)
                be.g_to_lagrange_dev(d_g, k, d_out)
                be.event_record(1)
                be.sync()
                ms.append(be.event_elapsed_ms(0, 1))
            same = bool(np.array_equal(d_out.download(g.shape), gl))
            d_g.free(); d_out.free()
            muls, nontrivial = model_muls(k)
            best = min(ms)
            res["g_to_lagrange_dev"].append({
                "k": k, "ms": ms, "ms_best": best, "equals_setup_lagrange_basis": same,
                "nontrivial_butterflies": nontrivial, "model_fq_muls": muls,
                "model_bound_ms": muls / FQ_MUL_PER_S * 1e3, "fraction_of_bound": muls / FQ_MUL_PER_S / (best * 1e-3)})
        K, k = [int(x) for x in args.downsize.split(",")]
        big = zk.ParamsKZG.setup(be, K, s)
        be.sync()
        t0 = time.perf_counter()
        small = big.downsize(k)
        t1 = time.perf_counter()
        direct = zk.ParamsKZG.setup(be, k, s)
        same = all(np.array_equal(a, b) for a, b in zip(small.read(), direct.read()))
        small.close(); direct.close(); big.close()
        res["downsize"] = {"from_k": K, "to_k": k, "ms": (t1 - t0) * 1e3, "equals_direct_setup": same,
                           "includes": "device copy of g, g_to_lagrange, fixed-base tables of both bases"}
        if args.cpu_k:
            kc = args.cpu_k
            params = zk.ParamsKZG.setup(be, kc, s)
            g, gl = params.read()
            params.close()
            t0 = time.perf_counter()
            got = H.g_to_lagrange(g, kc)
            t1 = time.perf_counter()
            res["cpu_g_to_lagrange"] = {"k": kc, "threads": os.cpu_count(), "ms": (t1 - t0) * 1e3,
                                        "equals_setup_lagrange_basis": bool(np.array_equal(got, gl))}
            gpu = [r for r in res["g_to_lagrange_dev"] if r["k"] == kc]
            if gpu:
                res["cpu_g_to_lagrange"]["gpu_speedup"] = res["cpu_g_to_lagrange"]["ms"] / gpu[0]["ms_best"]
    finally:
        be.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
