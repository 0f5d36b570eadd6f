#!/usr/bin/env python
"""bench.py — headline benchmark of the b200zk proving backend.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload prove|msm|ntt] [--k K] [--log-n L]
  python bench.py --impl reference ...     # CPU arm: the oracle's restatement of halo2's CPU
                                           # prover / best_multiexp / best_fft on this box's cores
  python bench.py --dump-outputs DIR ...   # also write what the last timed step computed to DIR/*.npy

Workloads (one "step" = one pass of the hot path over one batch of synthetic input):
  prove (default) : create_proof for the reference's Merkle Sum Tree circuit (chips.py: Poseidon
                    width 5, LtChip, u8 lookups; inclusion path of a 2^16-leaf tree, synthetic
                    values) padded to k = 20 — BASELINE.json's headline "create_proof ms (MST k=20)".
                    --circuit mst_dense is the same shape with every row in use (dense witness).
                    SRS and proving key resident in HBM.
  msm             : one best_multiexp over 2^L uniform scalars and 2^L SRS points
  ntt             : one best_fft over 2^L uniform Fr elements
Prints ONE JSON line: value = device-timed with inputs resident in HBM; e2e = the same call through
the host-buffer C-ABI entry point (pinned host witness / scalars -> H2D -> kernels -> D2H proof);
roofline for the dominant kernel; cpu_baseline on rank 0.  With N > 1 the default shards ONE proof over
the N GPUs (strong scaling: every rank holds SRS + pk and the same inputs, commits its columns, runs
its lookups, extends / evaluates its quotient cosets and multiplies its point range of the dense
commits; NCCL inside the library, see include/b200zk.h), checks the proof bytes against the
single-GPU proof of the same inputs outside the timed region ("verified"), and adds a "sharded"
block: one MSM 2^26 by point range and one NTT 2^26 four-step over the same N GPUs, each verified at
2^24.  --mode replicas gives the round-1 behaviour (one independent proof per GPU, weak scaling).
"""
import argparse
import atexit
import ctypes
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it (it may be read-only)

# measured on this pool's B200 with tools/imad_bench.cu (profiles/r01_imad_microbench.jsonl):
# IMAD.WIDE.U32 issues at 32 lanes/clk/SM -> 9.19e12 wide multiply-adds per second
IMAD_WIDE_PEAK = 9.19e12
MUL32_PER_FIELD_MUL = 136           # SURVEY.md §8(d): 8x8 product + 8x8 reduction + 8 (m = t0 * inv)


def msm_work_mul32(n):
    """SURVEY.md §8(d) accounting (c = 16, W = 16): (N*16*11 + 2*65536*16*16) * 136 mul32."""
    return (n * 16 * 11 + 2 * 65536 * 16 * 16) * MUL32_PER_FIELD_MUL


def ntt_digits(log_n):
    """Pass structure the library plans for a transform of 2^log_n (csrc/ntt_plan.hpp)."""
    if 10 <= log_n <= 21:
        P = (log_n + 7) // 8
    else:
        P = min(3, max(1, (log_n + 9) // 10))
    return [log_n // P + (1 if p < log_n % P else 0) for p in range(P)]


def ntt_passes(log_n):
    return len(ntt_digits(log_n))


def ntt_work_mul32(log_n):
    """Field multiplications one transform needs as executed: butterflies whose twiddle is not 1
    (stage with half-size 2^lh: a fraction 1 - 2^-lh of N/2) plus one inter-pass twiddle per element
    and pass boundary; 132 IMAD.WIDE-equivalents each (128 wide + 8 low IMAD at twice the rate)."""
    n = 1 << log_n
    d = ntt_digits(log_n)
    muls = sum(n / 2 * (1 - 2.0 ** -lh) for m in d for lh in range(m)) + n * (len(d) - 1)
    return muls * 132


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


def random_scalars(n, seed, out=None):
    """n Montgomery-form Fr elements, uniform below r's top limb (so every value is < r)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    a = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64) if out is None else out
    if out is not None:
        out[:] = rng.integers(0, 1 << 64, size=(n, 4), dtype=np.uint64)
    a[:, 3] %= np.uint64(0x30644e72e131a029)
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.path = device, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)         # a run that fails before stop() leaves no sampler behind
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "power_w_max": max(pw), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def dist_setup():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def max_over_ranks(dist, local, value):
    if dist is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64, device=torch.device("cuda", local))
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(dist, be):
    be.sync()
    if dist is not None:
        import torch
        dist.barrier()
        torch.cuda.synchronize()


def timed(be, dist, local, steps, fn):
    """CUDA events on the library's stream around `steps` calls, max over ranks -> total ms."""
    barrier(dist, be)
    be.event_record(0)
    for _ in range(steps):
        fn()
    be.event_record(1)
    be.sync()
    ms = be.event_elapsed_ms(0, 1)
    barrier(dist, be)
    return max_over_ranks(dist, local, ms)


CIRCUITS = {"mst": ("merkle_sum_tree_job", "the reference's MerkleSumTreeCircuit (Poseidon width 5, LtChip, 16-level path = tree of 2^16 leaves) padded to k={k}: 20 advice, 15 fixed, 8 u8 lookups, 16 permutation columns, degree 6; synthetic leaf / sibling values"),
            "v3": ("merkle_v3_job", "the reference's MerkleTreeV3Circuit (Poseidon width 3, 13-level path) at k={k}: 7 advice, 10 fixed, 10 permutation columns, degree 6"),
            "mst_dense": ("mst_shaped", "MST-shaped synthetic circuit k={k} with every row in use (dense witness, worst case for the commits): 20 advice, 8 u8 lookups, 16 permutation columns, degree 6"),
            "v3_dense": ("v3_shaped", "Merkle-v3-shaped synthetic circuit k={k} with every row in use: 9 advice, no lookups, 12 permutation columns, degree 6")}


def build_job(zk, circuit, k, seed):
    """Dense synthetic circuits come from circuits_synth, the reference's real circuits from chips."""
    mod = importlib.import_module(zk.__name__ + (".circuits_synth" if circuit.endswith("_dense") else ".chips"))
    return getattr(mod, CIRCUITS[circuit][0])(k, seed=seed)
WORKLOAD_TEXT = {
    "prove": "create_proof (KZG/SHPLONK/Blake2b), {circuit}; SRS + pk resident in HBM",
    "msm": "bn256 G1 MSM 2^{L} points (best_multiexp drop-in), uniform scalars, bases [s^i]G resident in HBM",
    "ntt": "bn256 Fr NTT 2^{L} (best_fft drop-in), uniform input",
}


# --------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    from __graft_entry__ import load_package
    zk = load_package()
    rank, world, local, dist = dist_setup()
    be = zk.Backend(local)
    peaks, peak_src = measured_peaks()
    line = {"n_gpus": world, "steps": args.steps, "warmup": args.warmup, "scaling": "weak", "vs_baseline": None,
            "data": "synthetic", "impl": "b200zk"}
    extra = {}
    sharded_proof = False
    restore = None                              # ntt: puts the seeded input back before the last timed step
    if args.workload == "prove":
        k = args.k
        n = 1 << k
        synth = importlib.import_module(zk.__name__ + ".circuits_synth")
        sharded_proof = world > 1 and args.mode == "sharded"
        if sharded_proof:
            rank_seed = 0                                         # every rank gets the same circuit, witness and rng stream
            line["scaling"] = "strong"
        else:
            rank_seed = rank
        job = build_job(zk, args.circuit, k, 1 + rank_seed)
        params = zk.ParamsKZG.setup(be, k, random_scalars(1, SRS_SEED)[0])
        pk = zk.ProvingKey(params, job.cs, k, job.fixed, job.map_col, job.map_row)
        A = job.cs.num_advice
        h_adv = be.pinned_empty((A * n, 4))
        for c in range(A):
            h_adv[c * n:(c + 1) * n] = job.advice[c]
        h_cols = [h_adv[c * n:(c + 1) * n] for c in range(A)]
        h_wide = be.pinned_empty((pk.rng_draws, 8))
        h_wide[:] = np.random.Generator(np.random.PCG64(RNG_SEED + rank_seed)).integers(0, 1 << 64, size=(pk.rng_draws, 8), dtype=np.uint64)
        d_adv, d_wide = be.to_device(h_adv), be.to_device(h_wide)
        lut = synth.mont_from_ints(job.instances[0] + [job.transcript_repr])
        inst, tr_repr = [lut[:-1]], lut[-1]
        single_proof = None
        if sharded_proof:
            # reference bytes: the single-GPU proof of the same inputs, made on this rank before its ctx joins the
            # communicator (outside every timed region)
            single_proof = pk.create_proof_dev(d_adv, inst, d_wide, tr_repr)
            uid = [zk.Backend.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            be.comm_init(world, rank, uid[0])

        def step_dev():
            return pk.create_proof_dev(d_adv, inst, d_wide, tr_repr)

        def step_e2e():
            return pk.create_proof(h_cols, inst, h_wide, tr_repr)

        def outputs(proof):
            return {"proof": np.frombuffer(proof, dtype=np.uint8)}

        unit, metric, hib = "ms", "create_proof_ms", False
        h2d, d2h = int(h_adv.nbytes + h_wide.nbytes), pk.proof_size
        dtype = "u32x8 Montgomery (bn256 Fr/Fq, IMAD pipe)"
        workload = WORKLOAD_TEXT["prove"].format(circuit=CIRCUITS[args.circuit][1].format(k=k))
    elif args.workload == "msm":
        # N > 1: ONE MSM of 2^L points sharded by point range (strong scaling): every rank holds
        # 2^L / N bases and scalars, partial sums are all-gathered (96 B per rank) and added.
        L = args.log_n
        shard_log = L - int(np.log2(world))
        n = 1 << shard_log
        params = zk.ParamsKZG.setup(be, shard_log, random_scalars(1, 4242 + rank)[0])
        h_scalars = be.pinned_empty((n, 4))
        random_scalars(n, 100 + rank, out=h_scalars)
        d_scalars = be.to_device(h_scalars)
        sharded = importlib.import_module(zk.__name__ + ".sharded")
        device = None
        if dist is not None:
            import torch
            device = torch.device("cuda", local)
        sc = sharded.ShardedCommit(sharded.GpuCommitEngine(zk, params), device)

        def step_dev():
            return sc.commit(d_scalars)

        def step_e2e():
            return sc.commit(h_scalars)

        def outputs(point):
            return {"msm": point}

        unit, metric, hib = "Mpts/s", "msm_mpts_per_s", True
        units_per_step = n / 1e6                                  # per rank; value multiplies by world
        if world > 1:
            line["scaling"] = "strong"
        h2d, d2h = n * 32, 96
        dtype = "u32x8 Montgomery (bn256 Fq/Fr, IMAD pipe)"
        workload = WORKLOAD_TEXT["msm"].format(L=L)
    else:
        L = args.log_n
        n = 1 << L
        dom = zk.EvaluationDomain(be, 2, L)
        h_a = be.pinned_empty((n, 4))
        random_scalars(n, 200 + rank, out=h_a)
        d_a = be.to_device(h_a)
        omega = dom.omega

        def step_dev():
            be.best_fft_dev(d_a, omega, L)

        def step_e2e():
            be._check(zk.lib().b200zk_fft(be._ctx, h_a.ctypes.data_as(ctypes.c_void_p), omega.ctypes.data_as(ctypes.c_void_p), L))

        def restore():
            d_a.upload(h_a)

        def outputs(_):
            return {"ntt": d_a.download((n, 4))}                   # transformed in place

        if world > 1:
            # ONE transform of 2^L elements sharded four-step (strong scaling): column blocks ->
            # column step -> NCCL all-to-all over NVLink -> row step (halo2-experiments_b200/sharded.py)
            import torch
            sharded = importlib.import_module(zk.__name__ + ".sharded")
            dev = torch.device("cuda", local)
            log_r = int(os.environ.get("B200ZK_FOURSTEP_LOG_R", min(7, L // 2)))   # R = 128: the column step is one warp-kernel pass
            # default: the exchange fused into the column-step kernel (NVLink peer stores, CUDA IPC);
            # B200ZK_NTT_NCCL=1 selects the NCCL all-to-all path
            fused = os.environ.get("B200ZK_NTT_NCCL", "0") != "1"
            fs = (sharded.FourStepNTTFused if fused else sharded.FourStepNTTDevice)(zk, be, L, log_r, rank, world, dev)
            extra["exchange"] = "fused into the column-step kernel (NVLink peer stores)" if fused else "NCCL all_to_all_single"
            blk_host = random_scalars((1 << L) // world, 300 + rank).reshape(1 << log_r, -1, 4)
            block = torch.from_numpy(blk_host.view(np.int64)).to(dev)
            omega_c = zk.EvaluationDomain(be, 2, L - log_r).omega
            pinned = torch.from_numpy(blk_host.view(np.int64)).pin_memory()
            pinned_np = pinned.numpy()

            def step_dev():
                return fs.forward(block, omega, omega_c)

            def restore():                                          # the NCCL path's column step overwrites the block
                block.copy_(pinned, non_blocking=False)

            def outputs(rows):                                      # this rank's output rows
                return {"ntt": rows.download((n, 4)) if fused else rows.cpu().numpy().view(np.uint64).reshape(n, 4)}

            def step_e2e():
                block.copy_(pinned, non_blocking=False)
                rows = fs.forward(block, omega, omega_c)
                if fused:
                    be._check(zk.lib().b200zk_download(be._ctx, pinned_np.ctypes.data_as(ctypes.c_void_p), rows.ptr, ctypes.c_size_t(pinned_np.nbytes)))
                else:
                    pinned.view(rows.shape).copy_(rows)

            n = (1 << L) // world                                   # per-rank elements; value multiplies by world
            line["scaling"] = "strong"

        unit, metric, hib = "GB/s", "ntt_gb_per_s", True
        units_per_step = 64.0 * n / 1e9
        h2d, d2h = n * 32, n * 32
        dtype = "u32x8 Montgomery (bn256 Fr, IMAD pipe)"
        workload = WORKLOAD_TEXT["ntt"].format(L=L)

    # ---- device-timed region: inputs resident in HBM --------------------------------
    for _ in range(max(args.warmup, 3)):
        step_dev()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = be.launch_count()
    result = [None]

    def step_kept():
        result[0] = None                        # no step's output is held while the next step runs
        result[0] = step_dev()

    if restore is None:
        ms = timed(be, dist, local, args.steps, step_kept)
    else:
        # the transform runs in place, so the last timed step starts again from the seeded input: what it computes
        # (and --dump-outputs writes) is the transform of that input; the copy stays outside both timed windows
        ms = timed(be, dist, local, args.steps - 1, step_kept)
        restore()
        ms += timed(be, dist, local, 1, step_kept)
    launches = (be.launch_count() - l0) // args.steps
    last = result[0]                            # what the last timed step computed: verified and dumped below
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, outputs(last))
    if args.workload == "prove":
        extra["phase_ms"] = pk.last_phase_ms()
        extra["timeline_ms"] = pk.last_trace()
        if dist is not None:
            tl = [None] * world
            dist.all_gather_object(tl, [round(v, 2) for _, v in extra["timeline_ms"]])
            extra["timeline_ms_all_ranks"] = {"labels": [a for a, _ in extra["timeline_ms"]], "ms": tl}
        extra["phase_note"] = "device time per phase; the advice-coset NTTs run on a side stream concurrently with the lookup / permutation phases, so the phases overlap and sum to more than the step"
    # ---- end-to-end region: host buffers through the C ABI ---------------------------
    for _ in range(2):
        step_e2e()
    barrier(dist, be)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    be.sync()
    e2e_ms = max_over_ranks(dist, local, (time.perf_counter() - t0) * 1e3) / args.steps
    clocks = sampler.stop() if rank == 0 else None
    if args.profile_step:                       # one extra step inside cudaProfilerStart/Stop for ncu
        be.profiler_range(True)
        step_dev()
        be.profiler_range(False)

    ms_per_step = ms / args.steps
    if args.workload == "prove":
        value, e2e_value = ms_per_step, e2e_ms
        extra["proofs_per_s_all_gpus"] = (1 if sharded_proof else world) / (ms_per_step / 1e3)
        if sharded_proof:
            import hashlib
            import torch
            e2e_proof = step_e2e()
            ok = int(last == single_proof and e2e_proof == single_proof)
            t = torch.tensor([ok], dtype=torch.int32, device=torch.device("cuda", local))
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            extra["verified"] = bool(t.item())
            extra["verification"] = {"what": "sharded proof bytes (device-resident and host-buffer entry points) == the single-GPU proof of the same circuit, "
                                             "witness, SRS and rng stream, compared on every rank (all-reduce MIN), outside the timed region",
                                     "proof_sha256_sharded": hashlib.sha256(last).hexdigest(), "proof_sha256_single_gpu": hashlib.sha256(single_proof).hexdigest(),
                                     "proof_bytes": len(last)}
            extra["parallelism"] = (f"one proof over {world} GPUs: advice / lookup / grand-product commits by column, lookups by argument, quotient by coset "
                                    f"({pk.degree - 1} cosets), dense commits (h pieces, random polynomial, SHPLONK) by point range, evaluations by query; "
                                    "polynomial exchange = grouped ncclBroadcast, commitments / partial sums = 64-byte all-gathers")
            h2d = h2d * world                                         # every rank uploads the witness over its own PCIe link
        elif rank == 0:
            # the proof of the timed region and the one of the host-buffer entry point, checked by the product's own verifier
            # (b200zk_verify_proof: transcript replay, SHPLONK, pairing) outside the timed region
            import hashlib
            e2e_proof = step_e2e()
            fixed_c, sigma_c = pk.vk_commitments()
            g, _ = params.read()
            vk = zk.VerifyingKey(job.cs, k, fixed_c, sigma_c, g[0], zk.g2_mul(random_scalars(1, SRS_SEED)[0]))
            extra["verified"] = bool(vk.verify_proof(inst, last, tr_repr) and vk.verify_proof(inst, e2e_proof, tr_repr))
            extra["verification"] = {"what": "b200zk_verify_proof accepts the proof of the last timed step and the proof of the host-buffer entry point "
                                             "(outside the timed region); byte identity with the CPU prover is in cpu_baseline.gpu_proof_bytes_identical",
                                     "proof_sha256": hashlib.sha256(last).hexdigest(), "proof_bytes": len(last)}
            del g
    else:
        value = units_per_step * world / (ms_per_step / 1e3)
        e2e_value = units_per_step * world / (e2e_ms / 1e3)
    line.update({"metric": metric, "unit": unit, "value": value, "ms_per_step": ms_per_step, "higher_is_better": hib, "dtype": dtype,
                 "config": {"workload": workload, "l2": "working set larger than L2 (126 MB); steps timed back to back"},
                 "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms},
                 "gpu_launches": int(launches), "clocks": clocks})

    # ---- roofline of the dominant kernel ------------------------------------------------
    imad_note = ("no HBM/tensor bound applies: 254-bit Montgomery arithmetic is IMAD-pipe bound; peak = measured IMAD.WIDE.U32 issue "
                 "rate on this B200 (tools/imad_bench.cu, profiles/r01_imad_microbench.jsonl)")
    if args.workload == "prove":
        # dominant kernel = the NTT pass kernel (per-coset size-n transforms of coeff_to_extended and
        # the iNTTs): time one size-n transform on device data with events
        omega = synth.mont_from_ints([pow(pow(7, (synth.R_MOD - 1) >> 28, synth.R_MOD), 1 << (28 - k), synth.R_MOD)])[0]
        d_vec = be.to_device(random_scalars(n, 5))
        for _ in range(3):
            be.best_fft_dev(d_vec, omega, k)
        reps = 20
        ms_ntt = timed(be, dist, local, reps, lambda: be.best_fft_dev(d_vec, omega, k)) / reps
        ph = extra["phase_ms"]
        ach = ntt_work_mul32(k) / (ms_ntt / 1e3)
        hbm = 64.0 * n / (ms_ntt / 1e3) / 1e9
        # the launch shape the proof mostly runs (5/6 of its NTT work): the q quotient cosets of one column as ONE
        # batched launch per pass — here q independent 2^k transforms through b200zk_fft_rows_dev
        q = pk.degree - 1
        d_rows = be.to_device(random_scalars(q * n, 7))
        rows_call = lambda: be._check(zk.lib().b200zk_fft_rows_dev(be._ctx, d_rows.ptr, ctypes.c_uint32(q), zk._p(zk._fr(omega, 1)), ctypes.c_uint32(k)))
        for _ in range(3):
            rows_call()
        ms_rows = timed(be, dist, local, reps, rows_call) / reps
        d_rows.free()
        ach_b = q * ntt_work_mul32(k) / (ms_rows / 1e3)
        hbm_b = 64.0 * n * q / (ms_rows / 1e3) / 1e9
        # The headline roofline is the launch the proof spends its NTT time in (q transforms per launch); the
        # single-transform figure — one best_fft call, a third of a wave short of filling the machine — is kept beside it.
        line["roofline"] = {"bound": "imad", "kernel": f"ntt pass kernel, {q} transforms of 2^{k} per launch (the quotient cosets of one column: "
                                                        f"{ntt_passes(k)} launches of {q} x 2^{k - 7} warp tiles)",
                            "achieved": ach_b / 1e12, "peak": IMAD_WIDE_PEAK / 1e12, "unit": "T IMAD.WIDE.U32/s", "frac": ach_b / IMAD_WIDE_PEAK,
                            # dram__bytes_read + write of the three pass launches of one batched coset extension inside the proof
                            # (5 transforms of 2^20 per launch), ncu --set full, profiles/r02_ncu_ntt_lazy_summary.txt: pass 1 also
                            # streams the 160 MB coset-power table, every pass its 64-byte twiddle records (one use each)
                            "traffic": ({"dram_bytes_per_launch": [672.2e6, 284.4e6, 293.9e6], "algorithmic_bytes_per_launch": 64 * n * 5,
                                         "source": "profiles/r02_ncu_ntt_lazy_summary.txt (5 x 2^20 per launch; cold-cache capture)",
                                         "single_2p20_dram_bytes_per_launch": [67.7e6, 34.1e6, 35.0e6],
                                         "single_source": "profiles/r01_ncu_ntt_warp_summary.txt"} if k == 20 else None),
                            "ms_per_launch_group": ms_rows, "share_of_step": ph["ntt"] / max(sum(ph.values()), 1e-9),
                            "hbm_view": {"achieved": hbm_b, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": hbm_b / peaks["hbm_gbs"],
                                         "algorithmic_bytes": 64 * n * q, "peak_source": peak_src},
                            "single": {"kernel": f"one 2^{k} transform = {ntt_passes(k)} launches (b200zk_fft_dev)", "ms_per_launch_group": ms_ntt,
                                       "achieved": ach / 1e12, "frac": ach / IMAD_WIDE_PEAK,
                                       "hbm_view": {"achieved": hbm, "frac": hbm / peaks["hbm_gbs"], "algorithmic_bytes": 64 * n}},
                            "note": imad_note + "; work = non-trivial butterfly and inter-pass twiddle multiplications x 132, the cost of a generic (CIOS) field multiplication "
                                    "— SURVEY 8(d)'s unit; the kernel's own constant-operand multiplier issues 99 wide + 16 low multiply-adds per product (DESIGN.md §4)"}
        # evaluate_h: multiplications per row as launched (b200zk_pk_quotient_muls) against the measured field-multiplication rate
        qm = pk.quotient_muls()
        if sharded_proof:                                         # rank 0 evaluates only its own cosets: the count below would not describe its kernels
            qm = None
        if qm is not None:
            muls = n * (qm["cosets"] * (qm["gates"] + qm["permutation"]) + qm["lookup_cosets"] * qm["lookups"])
            line["roofline_quotient"] = {"bound": "imad", "kernel": "expr_kernel + quot_perm_a/b + quot_lookup (evaluate_h on the quotient cosets)",
                                         "muls_per_row": qm, "field_muls": muls, "ms": ph["quotient"],
                                         "achieved": muls * 132 / (ph["quotient"] / 1e3) / 1e12 if ph["quotient"] else None, "peak": IMAD_WIDE_PEAK / 1e12,
                                         "unit": "T IMAD.WIDE.U32/s", "frac": muls * 132 / (ph["quotient"] / 1e3) / IMAD_WIDE_PEAK if ph["quotient"] else None,
                                         "share_of_step": ph["quotient"] / max(sum(ph.values()), 1e-9)}
        d_dense = be.to_device(random_scalars(n, 6))
        for _ in range(3):
            params.commit_dev(d_dense, n, lagrange=False)
        ms_msm = timed(be, dist, local, 5, lambda: params.commit_dev(d_dense, n, lagrange=False)) / 5
        line["roofline_msm"] = {"bound": "imad", "kernel": f"dense commit 2^{k} (msm_accumulate_task dominates)",
                                "achieved": msm_work_mul32(n) / (ms_msm / 1e3) / 1e12, "peak": IMAD_WIDE_PEAK / 1e12, "unit": "T IMAD.WIDE.U32/s",
                                "frac": msm_work_mul32(n) / (ms_msm / 1e3) / IMAD_WIDE_PEAK, "ms_per_launch_group": ms_msm,
                                "share_of_step": ph["msm"] / max(sum(ph.values()), 1e-9), "note": "work per SURVEY.md 8(d)"}
    elif args.workload == "msm":
        ach = msm_work_mul32(n) / (ms_per_step / 1e3)
        line["roofline"] = {"bound": "imad", "kernel": f"MSM 2^{int(np.log2(n))} (msm_accumulate dominates)", "achieved": ach / 1e12,
                            "peak": IMAD_WIDE_PEAK / 1e12, "unit": "T IMAD.WIDE.U32/s", "frac": ach / IMAD_WIDE_PEAK, "traffic": None,
                            "ms_per_launch_group": ms_per_step, "share_of_step": 1.0, "note": imad_note + "; work per SURVEY.md 8(d)"}
    else:
        ach = 64.0 * n / (ms_per_step / 1e3) / 1e9
        line["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                            "traffic": None, "peak_source": peak_src,
                            "note": "254-bit butterflies are IMAD-bound on B200 (see DESIGN.md): 64N bytes vs ~15N field muls"}
    line.update(extra)
    if args.workload == "prove" and not args.no_sharded_sweep:
        # BASELINE's "MSM Mpts/s & NTT GB/s at 1/2/4/8 B200": one MSM by point range and one NTT four-step over the
        # same N GPUs, in the same line.  The proving key is released first (2^26 points are 4 GiB per basis).
        pk.close(); params.close(); d_adv.free(); d_wide.free()
        try:
            line["sharded"] = sharded_sweep(zk, be, dist, rank, world, local, args)
        except Exception as e:                                      # the headline number stands on its own
            line["sharded"] = {"error": f"{type(e).__name__}: {e}"}
    if rank == 0:
        if not args.no_cpu_baseline:
            # prove: rank 0's circuit, witness, SRS secret and rng stream are the CPU arm's, so the two proofs must be the same bytes
            line["cpu_baseline"] = cpu_baseline(args, gpu_proof=last if args.workload == "prove" else None)
        emit(line)
    barrier(dist, be)
    be.close()
    if dist is not None:
        dist.destroy_process_group()


def sharded_sweep(zk, be, dist, rank, world, local, args):
    """One best_multiexp of 2^L points sharded by point range (partial sums all-gathered, 96 B per rank) and one
    best_fft of 2^L elements sharded four-step with the exchange fused into the column-step kernel (NVLink peer
    stores), over the `world` GPUs of this run; L = --sweep-log-n (26).  Both are verified at 2^--sweep-verify-log-n
    (24) outside the timed regions: the sharded MSM against ONE generic-path best_multiexp over the concatenated
    bases and scalars on rank 0, the sharded NTT rows against Horner evaluations of the full input on every rank."""
    import torch
    sharded = importlib.import_module(zk.__name__ + ".sharded")
    dev = torch.device("cuda", local) if dist is not None else None
    lw = int(np.log2(world))
    out = {"n_gpus": world}

    def msm_at(L, reps):
        shard_log = L - lw
        ns = 1 << shard_log
        params = zk.ParamsKZG.setup(be, shard_log, random_scalars(1, 4242 + rank)[0])
        h_sc = random_scalars(ns, 100 + rank)
        d_sc = be.to_device(h_sc)
        sc = sharded.ShardedCommit(sharded.GpuCommitEngine(zk, params), dev)
        res = sc.commit(d_sc)
        ms = None
        if reps:
            for _ in range(2):
                sc.commit(d_sc)
            ms = timed(be, dist, local, reps, lambda: sc.commit(d_sc)) / reps
        return params, d_sc, res, ms

    # ---- MSM: verify at Lv, time at L
    Lv, L = args.sweep_verify_log_n, args.sweep_log_n
    params, d_sc, res, _ = msm_at(Lv, 0)
    ok = True
    if rank == 0:
        ns = 1 << (Lv - lw)
        bases = [params.read(lagrange=False)[0]]
        for r in range(1, world):
            pr = zk.ParamsKZG.setup(be, Lv - lw, random_scalars(1, 4242 + r)[0])
            bases.append(pr.read(lagrange=False)[0])
            pr.close()
        d_b = be.to_device(np.concatenate(bases))
        d_s = be.to_device(np.concatenate([random_scalars(ns, 100 + r) for r in range(world)]))
        one = be.best_multiexp_dev(d_s, d_b, ns * world)           # generic path: no fixed-base table, explicit bases
        d_b.free(); d_s.free()
        ok = bool(np.array_equal(one, res))
    params.close(); d_sc.free()
    params, d_sc, res, ms = msm_at(L, 3)
    params.close(); d_sc.free()
    out["msm"] = {"log_n": L, "mpts_per_s": (1 << L) / 1e6 / (ms / 1e3), "ms": ms,
                  "path": "ParamsKZG commit over each rank's point range (fixed-base window tables when they fit in HBM, else the generic Pippenger), "
                          "partial sums combined by a 96-byte all-gather + host additions",
                  "verified": ok, "verified_how": f"2^{Lv} points: sharded result == one generic-path best_multiexp over the concatenation (rank 0)"}

    # ---- NTT: verify at Lv, time at L
    def ntt_at(L, reps, check):
        log_r = int(os.environ.get("B200ZK_FOURSTEP_LOG_R", min(7, L // 2)))       # R = 128: the column step is one warp-kernel pass
        R, C = 1 << log_r, 1 << (L - log_r)
        omega = zk.EvaluationDomain(be, 2, L).omega
        if world == 1:
            h_a = random_scalars(1 << L, 300)
            d_a = be.to_device(h_a)
            good = True
            if check:
                d_in = be.to_device(h_a)
                be.best_fft_dev(d_a, omega, L)
                got = d_a.download((1 << L, 4))
                wpow = zk.EvaluationDomain(be, 2, L)
                for kk in (0, 1, 12345, (1 << L) - 1):
                    x = wpow.rotate_omega(np.array(zk._FR_ONE, dtype=np.uint64), kk)
                    good = good and bool(np.array_equal(be.eval_polynomial_dev(d_in, 1 << L, x), got[kk]))
                d_in.free()
            ms = None
            if reps:
                for _ in range(2):
                    be.best_fft_dev(d_a, omega, L)
                ms = timed(be, dist, local, reps, lambda: be.best_fft_dev(d_a, omega, L)) / reps
            d_a.free()
            return good, ms
        cg, rg = C // world, R // world
        fs = sharded.FourStepNTTFused(zk, be, L, log_r, rank, world, dev)
        omega_c = zk.EvaluationDomain(be, 2, L - log_r).omega
        good = True
        if check:
            full = random_scalars(1 << L, 300)                       # the same input on every rank
            mine = np.ascontiguousarray(full.reshape(R, C, 4)[:, rank * cg:(rank + 1) * cg])
            block = torch.from_numpy(mine.view(np.int64)).to(dev)
            rows = fs.forward(block, omega, omega_c).download((rg, C, 4))   # [k_r local][k_c] = X[k_r + R k_c]
            d_in = be.to_device(full)
            dom = zk.EvaluationDomain(be, 2, L)
            for (a, b) in ((0, 0), (rg - 1, C - 1), (rg // 2, 4321 % C), (1 % rg, C // 2)):
                kk = (rank * rg + a) + R * b
                x = dom.rotate_omega(np.array(zk._FR_ONE, dtype=np.uint64), kk)
                good = good and bool(np.array_equal(be.eval_polynomial_dev(d_in, 1 << L, x), rows[a, b]))
            d_in.free()
        else:
            mine = random_scalars((1 << L) // world, 300 + rank).reshape(R, cg, 4)
            block = torch.from_numpy(mine.view(np.int64)).to(dev)
        ms = None
        if reps:
            for _ in range(2):
                fs.forward(block, omega, omega_c)
            ms = timed(be, dist, local, reps, lambda: fs.forward(block, omega, omega_c)) / reps
        fs.close()
        del block
        return good, ms

    good, _ = ntt_at(Lv, 0, True)
    _, ms = ntt_at(L, 5, False)
    if dist is not None:
        t = torch.tensor([int(good)], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        good = bool(t.item())
    out["ntt"] = {"log_n": L, "gb_per_s": 64.0 * (1 << L) / 1e9 / (ms / 1e3), "ms": ms,
                  "path": "single-GPU best_fft" if world == 1 else "four-step, column step fused with the exchange (NVLink peer stores), then row step",
                  "verified": good, "verified_how": f"2^{Lv} elements: output rows == Horner evaluation of the full input at 4 indices per rank"}
    return out


# --------------------------------------------------------------------------- CPU legs
SRS_SEED, RNG_SEED = 4242, 99         # both arms: SRS secret = random_scalars(1, SRS_SEED)[0], rng stream = PCG64(RNG_SEED)


def cpu_sample(args):
    """(callable, units, description) for the CPU restatement.  prove: the SAME configuration as the GPU arm
    — same circuit, witness (seed 1), size k, SRS secret and rng stream — through oracle/prover.cpp, the threaded
    C++ restatement of halo2's CPU prover; no extrapolation.  msm / ntt: a bounded sample size."""
    from __graft_entry__ import load_package
    from oracle import binding as orc
    from oracle import pyref
    if args.workload == "prove":
        zk = load_package()
        ks = args.k if args.cpu_k is None else min(args.k, args.cpu_k)
        job = build_job(zk, args.circuit, ks, 1)
        g, gl = orc.params_setup(ks, random_scalars(1, SRS_SEED)[0])
        pk = orc.CppProvingKey(job.cs, ks, job.fixed, job.map_col, job.map_row)
        wide = np.random.Generator(np.random.PCG64(RNG_SEED)).integers(0, 1 << 64, size=(pk.rng_draws, 8), dtype=np.uint64)
        fn = lambda: pk.create_proof(g, gl, job.advice, job.instances, wide, job.transcript_repr)
        return fn, None, (f"oracle/prover.cpp create_proof — threaded C++ restatement of halo2 v2023_02_02's CPU prover (best_multiexp, best_fft, "
                          f"evaluate_h on the 2^extended_k domain) — on the same circuit, witness, SRS and rng stream at k={ks}"), ks
    Ls = min(args.log_n, args.cpu_log_n)
    ns = 1 << Ls
    if args.workload == "msm":
        bases, _ = orc.params_setup(Ls, orc.random_fr(1, 4242)[0], with_lagrange=False)
        sc = random_scalars(ns, 7)
        return (lambda: orc.best_multiexp(sc, bases)), ns / 1e6, f"best_multiexp restatement on 2^{Ls} points", Ls
    a = random_scalars(ns, 8)
    w = orc.ints_to_mont([pyref.omega_for_k(Ls)])[0]
    return (lambda: orc.best_fft(a, w, Ls)), 64.0 * ns / 1e9, f"best_fft restatement on 2^{Ls} elements", Ls


def cpu_baseline(args, gpu_proof=None):
    """One pass of the CPU restatement on rank 0 (prove: one complete proof at the benchmarked size, whose bytes are
    also compared with the GPU proof of the same inputs)."""
    import hashlib
    from oracle import binding as orc
    fn, units, desc, size = cpu_sample(args)
    t0 = time.perf_counter()
    res = fn()
    dt = time.perf_counter() - t0
    cores = orc.get_threads()
    if args.workload == "prove":
        out = {"value": dt * 1e3, "unit": "ms", "cores": cores, "kind": "port", "k": size, "same_config": size == args.k,
               "sample": f"{desc}: one complete proof, {dt:.1f} s, no scaling"}
        if gpu_proof is not None and size == args.k:
            out["proof_sha256"] = hashlib.sha256(res).hexdigest()
            out["gpu_proof_bytes_identical"] = bool(res == gpu_proof)
        return out
    return {"value": units / dt, "unit": "Mpts/s" if args.workload == "msm" else "GB/s", "cores": cores, "kind": "port",
            "sample": f"{desc}, {dt:.2f} s"}


def run_reference(args):
    """--impl reference: halo2's CPU algorithm (oracle restatement; the Rust crate cannot be built here) on this
    box's host cores, same metric and config.  prove: every step is one complete create_proof at the benchmarked k
    (about a minute on 16 cores); the run times exactly --steps of them; nothing is extrapolated."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import binding as orc
    fn, units, desc, size = cpu_sample(args)
    cores = orc.get_threads()
    for _ in range(min(args.warmup, 1)):
        fn()
    times = []
    while len(times) < args.steps:
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    if args.workload == "prove":
        v, unit, metric, hib = dt * 1e3, "ms", "create_proof_ms", False
        workload = WORKLOAD_TEXT["prove"].format(circuit=CIRCUITS[args.circuit][1].format(k=size))
        sample = f"{desc}: {len(times)} complete proof(s) timed, mean {dt:.1f} s, no scaling"
    else:
        v = units / dt
        unit, metric, hib = ("Mpts/s", "msm_mpts_per_s", True) if args.workload == "msm" else ("GB/s", "ntt_gb_per_s", True)
        workload = WORKLOAD_TEXT[args.workload].format(L=size)
        sample = f"{desc} per step"
    emit({"impl": "reference", "metric": metric, "unit": unit, "value": v, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
          "steps": args.steps, "steps_timed": len(times), "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": hib,
          "scaling": "strong" if int(os.environ.get("WORLD_SIZE", "1")) > 1 and args.workload == "prove" else "weak", "vs_baseline": None,
          "dtype": "u64x4 Montgomery (CPU)", "data": "synthetic",
          "config": {"workload": workload, "same_config_as_gpu_arm": size == (args.k if args.workload == "prove" else args.log_n)},
          "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
          "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


DUMP_ROWS, DUMP_SEED = 1 << 16, 1234


def write_outputs(path, arrays):
    """--dump-outputs: every array as path/<name>.npy in float64, so that two builds can be compared output for output.
    Integers are stored exactly (a 64-bit limb as its two 32-bit halves, low half first).  An output of more than
    DUMP_ROWS rows is replaced by the same seeded sample of its rows in every run; their indices go to <name>_rows.npy."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        if a.dtype == np.uint64:
            a = a.view(np.uint32)
        if a.shape[0] > DUMP_ROWS:
            rows = np.sort(np.random.Generator(np.random.PCG64(DUMP_SEED)).choice(a.shape[0], DUMP_ROWS, replace=False))
            a = a[rows]
            np.save(os.path.join(path, name + "_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


_JSON_OUT = None


def emit(line):
    """The one JSON line of the contract, on the process's real stdout."""
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # stdout carries exactly one JSON line: libraries that write to fd 1 (NCCL prints its version banner there
    # under torchrun) are sent to stderr, the line itself goes to a duplicate of the original descriptor
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200zk", choices=["b200zk", "reference"])
    ap.add_argument("--workload", default="prove", choices=["prove", "msm", "ntt"])
    ap.add_argument("--k", type=int, default=20, help="prove: circuit size")
    ap.add_argument("--circuit", default="mst", choices=sorted(CIRCUITS), help="prove: circuit shape")
    ap.add_argument("--cpu-k", type=int, default=None, help="prove: size of the CPU arm's proof (default: the benchmarked k; smaller only for quick local runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--log-n", type=int, default=24, help="msm / ntt size")
    ap.add_argument("--cpu-log-n", type=int, default=None, help="msm / ntt: size of the bounded CPU sample")
    ap.add_argument("--profile-step", action="store_true", help="bracket one extra step with cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--mode", default="sharded", choices=["sharded", "replicas"], help="prove with N > 1: one proof over N GPUs (default) or N independent proofs")
    ap.add_argument("--no-sharded-sweep", action="store_true", help="prove: skip the MSM / NTT 2^26 block")
    ap.add_argument("--sweep-log-n", type=int, default=26)
    ap.add_argument("--sweep-verify-log-n", type=int, default=24)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (rank 0: the proof, the MSM point or the NTT output) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path")
    if args.cpu_log_n is None:
        args.cpu_log_n = 20 if args.workload == "msm" else 22
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
