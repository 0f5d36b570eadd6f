#!/usr/bin/env python
"""Throughput of b200zk_create_proofs (many proofs of one proving key on concurrent lanes of one GPU) against a loop of
create_proof_dev on the same key and inputs.

    python tools/proof_batch_bench.py [--work mst9,v3_14,mst14,mst20] [--lanes 1,2,4,8] [--reps 3] [--profile FILE] [--out FILE]

Workloads: the reference's Merkle Sum Tree circuit at k = 9 (5 levels) and k = 14 (16 levels) and the Merkle tree v3
at k = 14, batches of 64; the Merkle Sum Tree at k = 20 (16 levels), batches of 8.  Every proof of a batch has its
own rng stream (seeded numpy draws: any 512-bit value is a valid Fr::random input).  Inputs are device resident
(create_proofs_dev against a loop of create_proof_dev); one line per size also takes host inputs (create_proofs against
a loop of create_proof) on 4 lanes.  Each configuration runs one warm-up batch, then --reps timed batches; times are a
host clock around the call, which returns after its last proof has synchronised.  Reported per line:
  proofs_per_s        count / median batch time
  latency_ms_lane0    median over the timed batches of the wall time of the last proof lane 0 ran: one proof's latency
                      while the other lanes run theirs
  launches_per_proof  kernel launches of the batch (all lanes) / count
  lane_bytes          device memory one extra lane took (free memory before and after reserving the lanes)
Proof bytes of the batch are checked against the loop's.  --profile FILE: one batch of MST k = 9 on 4 lanes under
torch.profiler (CUDA activities); FILE gets a summary of its kernel timeline (busy time, overlap, gaps).
The card's name and power limit are read in the same run.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def job_for(zk, name):
    import numpy as np
    fe = importlib.import_module(zk.__name__ + ".frontend")
    chips = importlib.import_module(zk.__name__ + ".chips")
    if name == "mst9":
        return chips.merkle_sum_tree_job(9, levels=5), 64
    if name == "mst14":
        return chips.merkle_sum_tree_job(14), 64
    if name == "mst20":
        return chips.merkle_sum_tree_job(20), 8
    if name == "v3_14":
        rng = np.random.Generator(np.random.PCG64(14))
        elements = [int(x) for x in rng.integers(1, 1 << 62, size=13)]
        indices = [int(x) for x in rng.integers(0, 2, size=13)]
        root = chips.compute_merkle_root(99, elements, indices)
        return fe.synthesize_job(chips.MerkleTreeV3Circuit(99, elements, indices), 14, [[99, root]]), 64
    raise ValueError(name)


def mont(vals):
    """integers < r -> Montgomery limbs (R = 2^256 mod r), without the test oracle"""
    import numpy as np
    r = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001
    out = np.zeros((len(vals), 4), dtype=np.uint64)
    for i, v in enumerate(vals):
        m = (v % r) * (1 << 256) % r
        for j in range(4):
            out[i, j] = (m >> (64 * j)) & ((1 << 64) - 1)
    return out


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2] if len(xs) % 2 else 0.5 * (xs[len(xs) // 2 - 1] + xs[len(xs) // 2])


def free_bytes():
    import torch
    return torch.cuda.mem_get_info(0)[0]


def timeline(trace_path):
    """busy time (union of kernel intervals), summed kernel time, time with >= 2 kernels running, gaps, over the span"""
    ev = json.load(open(trace_path))
    ev = ev.get("traceEvents", ev)
    ks = sorted((e["ts"], e["ts"] + e["dur"]) for e in ev if e.get("cat") == "kernel" and "dur" in e)
    if not ks:
        return {"kernels": 0}
    pts = sorted([(a, 1) for a, _ in ks] + [(b, -1) for _, b in ks])
    busy = overlap = 0.0
    level, last = 0, pts[0][0]
    for t, d in pts:
        if level >= 1:
            busy += t - last
        if level >= 2:
            overlap += t - last
        level += d
        last = t
    span = ks[-1][1] - ks[0][0]
    durs = sorted(b - a for a, b in ks)
    return {"kernels": len(ks), "span_us": span, "busy_us": busy, "kernel_sum_us": sum(durs), "overlap_2plus_us": overlap,
            "idle_us": span - busy, "median_kernel_us": durs[len(durs) // 2], "mean_concurrency": sum(durs) / busy if busy else 0.0}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--work", default="mst9,v3_14,mst14,mst20")
    ap.add_argument("--lanes", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    from __graft_entry__ import load_package
    zk = load_package()
    be = zk.Backend(0)
    res = {"card": card(), "reps": args.reps, "lines": []}
    try:
        for name in [w for w in args.work.split(",") if w]:
            job, count = job_for(zk, name)
            params = zk.ParamsKZG.setup(be, job.k, mont([12345])[0])
            pk = zk.ProvingKey(params, job.cs, job.k, job.fixed, job.map_col, job.map_row)
            inst = [mont(c) for c in job.instances]
            tr = mont([job.transcript_repr])[0]
            rng = np.random.Generator(np.random.PCG64(7))
            wides = [rng.integers(0, 1 << 64, size=(pk.rng_draws, 8), dtype=np.uint64) for _ in range(count)]
            adv = np.concatenate([np.ascontiguousarray(a).reshape(-1, 4) for a in job.advice])
            d_adv = [be.to_device(adv) for _ in range(count)]
            d_rng = [be.to_device(w) for w in wides]
            insts = [inst] * count

            def timed(fn):
                t, lat, launches = [], [], 0
                want = fn()                                            # warm-up
                for _ in range(args.reps):
                    l0 = be.launch_count()
                    t0 = time.perf_counter()
                    got = fn()
                    t.append(time.perf_counter() - t0)
                    launches = be.launch_count() - l0
                    lat.append(dict(pk.last_trace()).get("end", 0.0))
                    assert got == want
                return median(t), median(lat), launches, want

            loop_s, loop_lat, loop_launches, ref = timed(lambda: [pk.create_proof_dev(a, inst, w, tr) for a, w in zip(d_adv, d_rng)])
            base = {"work": name, "k": job.k, "count": count, "inputs": "device", "mode": "loop", "lanes": 1,
                    "proofs_per_s": count / loop_s, "latency_ms_lane0": loop_lat, "launches_per_proof": loop_launches / count}
            res["lines"].append(base)
            print(json.dumps(base), flush=True)
            free1 = None
            for lanes in [int(x) for x in args.lanes.split(",") if x]:
                got_lanes = pk.reserve_lanes(lanes)
                if lanes == 1:
                    free1 = free_bytes()
                lane_bytes = (free1 - free_bytes()) / (got_lanes - 1) if got_lanes > 1 and free1 is not None else 0
                s, lat, launches, out = timed(lambda: pk.create_proofs_dev(d_adv, insts, d_rng, tr))
                assert out == ref, f"{name}: batch bytes differ from the loop's"
                line = {"work": name, "k": job.k, "count": count, "inputs": "device", "mode": "batch", "lanes": got_lanes,
                        "proofs_per_s": count / s, "speedup_vs_loop": loop_s / s, "latency_ms_lane0": lat,
                        "launches_per_proof": launches / count, "lane_bytes": lane_bytes}
                res["lines"].append(line)
                print(json.dumps(line), flush=True)
            # host inputs: 4 lanes against the host loop
            hadv = [job.advice] * count
            hl_s, hl_lat, _, href = timed(lambda: [pk.create_proof(job.advice, inst, w, tr) for w in wides])
            assert href == ref
            got_lanes = pk.reserve_lanes(4)
            hb_s, hb_lat, _, hout = timed(lambda: pk.create_proofs(hadv, insts, wides, tr))
            assert hout == ref
            line = {"work": name, "k": job.k, "count": count, "inputs": "host", "loop_proofs_per_s": count / hl_s, "lanes": got_lanes,
                    "batch_proofs_per_s": count / hb_s, "speedup_vs_loop": hl_s / hb_s, "latency_ms_lane0": hb_lat}
            res["lines"].append(line)
            print(json.dumps(line), flush=True)
            if args.profile and name == "mst9":
                import torch
                pk.reserve_lanes(4)
                pk.create_proofs_dev(d_adv, insts, d_rng, tr)
                trace = os.path.join(tempfile.gettempdir(), f"proof_batch_{os.getpid()}.json")
                out = {}
                for mode, fn in [("batch_4_lanes", lambda: pk.create_proofs_dev(d_adv, insts, d_rng, tr)),
                                 ("loop", lambda: [pk.create_proof_dev(a, inst, w, tr) for a, w in zip(d_adv, d_rng)])]:
                    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                        fn()
                    prof.export_chrome_trace(trace)
                    out[mode] = timeline(trace)
                    os.remove(trace)
                res["timeline_mst9"] = out
                with open(args.profile, "w") as f:
                    json.dump(out, f, indent=1)
            for d in d_adv + d_rng:
                d.free()
            pk.close(); params.close()
    finally:
        be.close()
    txt = json.dumps(res)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
