#!/usr/bin/env python
"""bench.py - proofs/sec at 2^16 gates (BASELINE.json metric) for the B200-native prover backend.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA prover
  python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's proofs as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic input: `--inflight` independent
2^16-gate proofs issued concurrently (one host thread + CUDA stream each) on every rank.  Ranks
hold independent proofs (SURVEY.md section 8e: replicas, no data-path collective), so scaling is
weak.  `value` = proofs/s with the witness tables already resident in HBM; `e2e` = the same through
the host-pointer C ABI call (pb200_prove), i.e. including the pinned-host -> device copy of every
proof's witnesses and the device -> host read of the proof; `e2e_with_synthesis` additionally re-runs
the circuit on the host for every proof (the composer's witness-only mode), which is what the
reference's Prover::prove(rng, circuit) does first (src/compiler/prover.rs:425).  The roofline block
describes the dominant kernel (MSM bucket accumulation), timed live with CUDA events on its launching
stream.  `extra` carries the other BASELINE.json configs: one 2^20-gate proof (configs[2], N = 1) and the
point-sharded MSM sweep 2^16..2^24 with its one NCCL all-gather (configs[3], every N).
"""
import argparse
import math
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

R_MOD = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
LOG_GATES = 16
N_GATES = (1 << LOG_GATES) - 6          # fills the 2^16 domain, commit key trimmed to 2^16 + 7 points
SRS_POINTS = (1 << LOG_GATES) + 7
SRS_X, SRS_G = 0x1234567, 0x7654321     # synthetic "toxic waste" (seeded; a real SRS comes from a ceremony)
LABEL = b"bench-2^16"
# per G1 mixed addition (XYZZ madd = 8M + 2S in Fp) the SASS of k_msm_accumulate issues 276 IMAD.WIDE per product,
# 210 per squaring (symmetric partial products once) and 420 for the fused pair R(Q - X3) - Y1 PPP (two products,
# one Montgomery reduction): 6 products + 2 squarings + 1 fused pair
IMAD_PER_ADD = 6 * 276 + 2 * 210 + 420
FP_PRODUCTS_PER_ADD = IMAD_PER_ADD / 276.0  # in units of one carry-chained Fp product
IMAD_PER_BUTTERFLY = 137


def mont(v: int) -> bytes:
    return ((v << 256) % R_MOD).to_bytes(32, "little")


def blinders_for(i: int) -> bytes:
    import random

    rng = random.Random(0xB200_0000 + i)
    return b"".join(mont(rng.randrange(R_MOD)) for _ in range(14))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory: str, outputs: dict):
    """Writes every list of proofs in `outputs` as directory/<name>.npy: float32 [proofs, 1008], one byte of
    Proof::to_bytes per element (exact in float32).  The inputs are seeded, so two builds run with the same
    arguments can be compared output for output.  Past 64 MiB in all, each array keeps its first rows."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    rows = DUMP_LIMIT_BYTES // (4 * sum(len(proofs[0]) for proofs in outputs.values()))
    for name, proofs in outputs.items():
        a = np.frombuffer(b"".join(proofs[:rows]), dtype=np.uint8).reshape(-1, len(proofs[0]))
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float32))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:]):
                    if val.strip().lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.2)

    def result(self):
        busy = sorted(self.samples)[len(self.samples) // 2:] if self.samples else []
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def host_cpu_state():
    """CPU bandwidth state of this container (cgroup v2 cpu.max / cpu.stat, v1 fallbacks): quota in CPUs and the
    cumulative throttling counters - proving is host-driven (one thread per proof in flight), so a throttled
    container shows up as lost proofs/s, not as a slow GPU."""
    st = {"quota_cpus": None, "nr_throttled": None, "throttled_usec": None, "usable_cpus": len(os.sched_getaffinity(0))}
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        st["quota_cpus"] = None if q == "max" else int(q) / int(per)
        for ln in open("/sys/fs/cgroup/cpu.stat"):
            k, v = ln.split()
            if k in ("nr_throttled", "throttled_usec"):
                st[k] = int(v)
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            st["quota_cpus"] = q / per if q > 0 else None
            for ln in open("/sys/fs/cgroup/cpu/cpu.stat"):
                k, v = ln.split()
                if k == "nr_throttled":
                    st[k] = int(v)
                if k == "throttled_time":
                    st["throttled_usec"] = int(v) // 1000
        except (OSError, ValueError):
            pass
    return st


def finish_dist(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()


def build_workload(circuit: str):
    """Returns (arrays, description).  "bench" is the reference's own benchmark circuit
    (benches/plonk.rs BenchCircuit<2^16>: 64129 gates of every gadget family), built by the native
    composer of libplonk_b200; "synthetic" is a random arithmetic-gate circuit filling the domain."""
    if circuit == "bench":
        from plonk_b200.gadgets import bench_circuit

        arrays = bench_circuit(1 << LOG_GATES).arrays()
        what = f"reference BenchCircuit<2^16> (benches/plonk.rs: {arrays.constraints} gates of all gadget families"
    else:
        from plonk_b200.composer import synthetic_circuit

        arrays = synthetic_circuit(N_GATES, seed=16).arrays()
        what = f"2^16-gate synthetic arithmetic circuit ({arrays.constraints} constraints"
    return arrays, what + ", domain 2^16, quotient domain 2^19)"


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from plonk_b200 import Prover
    from plonk_b200._lib import check, lib

    L = lib()
    check(L.pb200_init(local))
    arrays, workload = build_workload(args.circuit)
    srs_raw = ctypes.create_string_buffer(SRS_POINTS * 96)
    check(L.pb200_srs_setup_from_secret(mont(SRS_X), mont(SRS_G), SRS_POINTS, srs_raw))
    prover = Prover(LABEL, arrays.constraints, arrays.selectors, arrays.wires, arrays.n_witnesses, srs_raw.raw)
    inflight = args.inflight
    n_wit = arrays.n_witnesses
    # pinned host staging buffers (one per in-flight slot) and device-resident copies
    host_wit = [torch.empty(n_wit * 32, dtype=torch.uint8).pin_memory() for _ in range(inflight)]
    for t in host_wit:
        t.copy_(torch.frombuffer(bytearray(arrays.witnesses), dtype=torch.uint8))
    dev_wit = [t.cuda() for t in host_wit]
    proofs = [ctypes.create_string_buffer(1008) for _ in range(inflight)]
    pool = ThreadPoolExecutor(inflight)
    pi_idx, pi_vals, n_pi = arrays.pi_idx, arrays.pi_vals, arrays.n_pi

    def synthesize(slot):
        """Prover::prove's first step (prover.rs:425): run the circuit again for its witness values; the table
        lands straight in the slot's pinned staging buffer."""
        h = ctypes.c_void_p()
        check(L.pb200_composer_new(ctypes.byref(h)))
        try:
            check(L.pb200_composer_set_witness_only(h, 1))
            check(L.pb200_composer_bench_circuit(h, 1 << LOG_GATES))
            assert L.pb200_composer_witnesses(h) == n_wit
            check(L.pb200_composer_export(h, None, None, host_wit[slot].data_ptr(), None, None))
        finally:
            L.pb200_composer_free(h)

    def one(slot, step, resident):
        bl = blinders_for(step * inflight + slot)
        if resident == "synth":
            synthesize(slot)
            check(L.pb200_prove(prover._h, host_wit[slot].data_ptr(), n_wit, pi_idx, pi_vals, n_pi, bl, proofs[slot]))
        elif resident:
            check(L.pb200_prove_dev(prover._h, dev_wit[slot].data_ptr(), n_wit, pi_idx, pi_vals, n_pi, bl, proofs[slot], None))
        else:
            check(L.pb200_prove(prover._h, host_wit[slot].data_ptr(), n_wit, pi_idx, pi_vals, n_pi, bl, proofs[slot]))

    def run_steps(k, resident, base=0):
        # k steps = k proofs on each of the `inflight` slots; the slots run back to back without a
        # barrier between steps (independent proofs: nothing to wait for)
        def worker(slot):
            for s in range(k):
                one(slot, base + s, resident)

        list(pool.map(worker, range(inflight)))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(k, resident):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_steps(k, resident, base=1000)
        torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    run_steps(args.warmup, True)
    run_steps(max(1, args.warmup // 2), False)
    sampler = ClockSampler(local)
    use_sampler = rank == 0 and not os.environ.get("PB200_NO_SAMPLER")  # one nvidia-smi poller per box is enough
    if use_sampler:
        sampler.start()
    host = {"before": host_cpu_state()}
    launches0 = L.pb200_launch_count()
    cpu0 = time.process_time()
    ms_res = timed(args.steps, True)
    host["cpu_s_value"] = time.process_time() - cpu0
    host["after_value"] = host_cpu_state()
    launches = L.pb200_launch_count() - launches0
    # the proofs of each timed region's last step, one per slot (later regions overwrite the buffers)
    outputs = {"proofs": [p.raw for p in proofs]}
    cpu0 = time.process_time()
    ms_e2e = timed(args.steps, False)
    host["cpu_s_e2e"] = time.process_time() - cpu0
    host["after_e2e"] = host_cpu_state()
    outputs["proofs_e2e"] = [p.raw for p in proofs]
    ms_synth = None
    if args.circuit == "bench":
        run_steps(1, "synth")
        t_cpu0 = time.process_time()
        ms_synth = timed(args.steps, "synth")
        cpu_s_synth = time.process_time() - t_cpu0
        outputs["proofs_e2e_with_synthesis"] = [p.raw for p in proofs]
    # Dominant kernel (MSM bucket accumulation), timed with CUDA events on its launching stream while
    # proofs run one at a time, so the event pairs bracket the kernel alone (with several proofs in
    # flight the kernels of different streams overlap and a per-kernel duration is not meaningful).
    barrier()
    t_single0 = time.time()
    for s in range(3):
        one(0, 5000 + s, True)
    torch.cuda.synchronize()
    single_ms = (time.time() - t_single0) * 1e3 / 3  # a proof that is alone (latency-oriented launch shapes)
    # the same three proofs in the launch shape of the timed region (one lane per bucket in the dense MSMs), with the
    # in-library CUDA-event timing of the accumulation phase switched on
    check(L.pb200_throughput_mode(1))
    check(L.pb200_profile_enable(1))
    barrier()
    t_prof0 = time.time()
    for s in range(3):
        one(0, 6000 + s, True)
    torch.cuda.synchronize()
    prof_ms = (time.time() - t_prof0) * 1e3 / 3
    check(L.pb200_throughput_mode(0))
    acc_ms, acc_adds, acc_launches, acc_points = ctypes.c_double(), ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
    check(L.pb200_profile_read(ctypes.byref(acc_ms), ctypes.byref(acc_adds), ctypes.byref(acc_launches), ctypes.byref(acc_points)))
    sp_ms, sp_adds, sp_launches, sp_points = ctypes.c_double(), ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
    check(L.pb200_profile_read_sparse(ctypes.byref(sp_ms), ctypes.byref(sp_adds), ctypes.byref(sp_launches), ctypes.byref(sp_points)))
    check(L.pb200_profile_enable(0))
    sampler.stop_flag = True
    if use_sampler:
        sampler.join()
    host["after_synthesis"] = host_cpu_state()

    total_proofs = args.steps * inflight * world
    value = total_proofs / (ms_res * 1e-3)
    e2e_value = total_proofs / (ms_e2e * 1e-3)
    # BASELINE.json configs[3]: every rank takes part in the point-sharded MSM sweep (one NCCL all-gather per MSM)
    sweep = None if args.no_msm_sweep else msm_sweep(L, torch, rank, world, local, args)
    if rank != 0:
        finish_dist(world)
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    # dominant kernel: MSM bucket accumulation.  Both hot kernels are integer-multiply bound at 256/381-bit
    # precision (SURVEY.md section 8d: ~20 MAC per algorithmic byte against a machine balance of ~2.8), so the
    # binding roofline is the ALU one; the HBM fraction is reported beside it.
    hbm_peak, peak_src = measured_peaks()
    imad, fp_peak = ctypes.c_double(), ctypes.c_double()
    check(L.pb200_imad_peak(ctypes.byref(imad)))
    check(L.pb200_fp_product_peak(ctypes.byref(fp_peak)))
    acc_s = acc_ms.value * 1e-3
    adds_per_s = acc_adds.value / acc_s if acc_s else 0.0
    algo_bytes = 128.0 * acc_points.value  # SURVEY 8(d): 96 B affine base + 32 B scalar per MSM point
    alu_peak = imad.value / IMAD_PER_ADD
    alu_frac = adds_per_s / alu_peak if alu_peak else 0.0
    hbm_achieved = algo_bytes / acc_s / 1e9 if acc_s else 0.0
    traffic, traffic_src = measured_traffic()
    roof = {
        "kernel": "k_msm_accumulate (+ k_msm_heavy_chunks / k_msm_heavy_combine for over-long buckets)", "bound": "alu",
        "achieved": adds_per_s, "peak": alu_peak, "unit": "G1 adds/s", "frac": max(alu_frac, hbm_achieved / hbm_peak),
        "peak_source": "pb200_imad_peak, measured in this run: register-only IMAD.WIDE.U32 issue rate / "
                       f"{IMAD_PER_ADD} IMAD.WIDE per XYZZ mixed addition (SASS count)",
        "imad_wide_per_s_measured": imad.value,
        "hbm": {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak, "peak_source": peak_src,
                "algorithmic_bytes": "128 B per MSM point (96 B affine base + 32 B scalar, each once)"},
        "traffic": traffic, "traffic_source": traffic_src,
        "launches": acc_launches.value, "avg_launch_ms": acc_ms.value / max(1, acc_launches.value),
        "adds_per_launch": acc_adds.value / max(1, acc_launches.value),
        "share_of_step": (acc_ms.value / 3) / prof_ms if prof_ms else None,
        "launches_counted": "the dense MSMs of a proof (z, the four quotient parts, the two openings: 3 launches per proof); the wire-value "
                            "commitments are sparse (~1 non-zero digit per scalar) and reported under sparse_msm",
        "sparse_msm": {"launches": sp_launches.value, "avg_launch_ms": sp_ms.value / max(1, sp_launches.value),
                       "adds_per_launch": sp_adds.value / max(1, sp_launches.value), "points_per_launch": sp_points.value / max(1, sp_launches.value),
                       "share_of_step": (sp_ms.value / 3) / prof_ms if prof_ms else None},
        "measured": "3 proofs issued one at a time after the timed region (exclusive kernel durations, CUDA events on the launching stream), "
                    "in the launch shape of the timed region (pb200_throughput_mode(1): one lane per bucket in the dense MSMs; a proof "
                    "that is really alone splits buckets over lanes for latency - single_stream_ms_per_proof is measured that way)",
        "ms_per_proof_in_this_shape": prof_ms,
        "single_stream_ms_per_proof": single_ms,
        "carry_chain_ceiling": {"fp_products_per_s": fp_peak.value, "adds_per_s": fp_peak.value / FP_PRODUCTS_PER_ADD,
                                "frac": adds_per_s * FP_PRODUCTS_PER_ADD / fp_peak.value if fp_peak.value else None,
                                "source": "pb200_fp_product_peak, measured in this run: dependent chains of carry-chained Fp products "
                                          "(IMAD.WIDE.U32.X issues at half the rate of the carry-free form); "
                                          f"{FP_PRODUCTS_PER_ADD:.2f} Fp-product equivalents per mixed addition"},
    }
    ntt = ntt_microbench(L, torch, imad.value)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(2)
    extra = {"host": host}
    if ms_synth is not None:
        host_threads = len(os.sched_getaffinity(0))
        extra["e2e_with_synthesis"] = {
            "value": total_proofs / (ms_synth * 1e-3), "unit": "proofs/s",
            "what": "every proof first re-runs the circuit on the host (native composer, witness-only mode: BenchCircuit<2^16>, "
                    "as Prover::prove(rng, circuit) does, prover.rs:425), then pb200_prove with host witnesses",
            "host_threads": inflight, "host_threads_available": host_threads,
            "host_cpu_s_per_proof": cpu_s_synth / (args.steps * inflight),
            "frac_of_value": (total_proofs / (ms_synth * 1e-3)) / value}
    line = {
        "metric": "proofs/sec @ 2^16 gates", "value": value, "unit": "proofs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 limbs (Fr 256-bit / Fp 384-bit Montgomery)", "data": "synthetic",
        "config": {"workload": workload + "; Proof bytes == CPU restatement of the reference (tests/test_gpu_prover.py)",
                   "proofs_per_step_per_gpu": inflight, "parallelism": f"replicas x{world}, no collective",
                   "l2": "per-proof working set ~0.7 GB (prover key 240 MB + MSM tables 100 MB + scratch) > 126 MB L2; no flush needed"},
        "e2e": {"value": e2e_value, "unit": "proofs/s", "h2d_bytes_per_step": inflight * (n_wit * 32 + n_pi * 32 + 14 * 32),
                "d2h_bytes_per_step": inflight * (11 * 96 + 15 * 32)},
        "gpu_launches": int(launches), "clocks": sampler.result(), "roofline": roof, "ntt": ntt, "extra": extra,
    }
    if cpu:
        line["cpu_baseline"] = cpu
    if sweep is not None:
        extra["msm_sweep"] = sweep
    if world == 1 and not args.no_proof20:
        del prover, dev_wit  # make room: the 2^20-gate prover key is ~5 GB, its commit-key tables ~2.6 GB
        torch.cuda.empty_cache()
        extra.update(proof_2_20(L, torch))
    print(json.dumps(line), flush=True)
    finish_dist(world)


def msm_sweep(L, torch, rank, world, local, args):
    """BASELINE.json configs[3] / SURVEY.md section 8e-ii: one G1 MSM of 2^16 .. 2^24 points whose points are
    partitioned across the ranks.  Every rank makes its slice of a seeded key [x^i]g on its own GPU, holds the
    full scalar vector in HBM and reads its slice; plonk_b200.dist.ShardedCommitKey runs the slice MSM and the
    device-resident ncclAllGather of the digit sums (pb200_msm_g1_allgather_dev) - or, below its size threshold,
    the whole MSM on a replicated key with no collective.  The scalars are s_i = u[i mod 4096] + v[i div 4096] for
    random u, v (distinct, full-range), so the result is checked against [g p(x)]G from a closed form.
    Timed with CUDA events on the launching stream, max over ranks, best of `iters`."""
    import random

    import torch.distributed as dist

    from plonk_b200 import dist as pd
    from plonk_b200._lib import check

    comm = pd.NcclComm() if world > 1 else None
    x, gs = SRS_X, SRS_G
    threshold = 1 << 18
    stream = torch.cuda.Stream()
    rows = []
    # replica of the first `threshold` points, for MSMs too small to be worth an exchange
    rep_raw = ctypes.create_string_buffer(96 * threshold)
    check(L.pb200_srs_setup_from_secret(mont(x), mont(gs), threshold, rep_raw))
    for log_n in [int(v) for v in args.msm_sizes.split(",") if v]:
        n = 1 << log_n
        first, count = pd.shard_range(n, rank, world)
        slice_raw = ctypes.create_string_buffer(96 * max(count, 1))
        if count:  # [x^(first+i)] g = [x^i] ([x^first] g)
            check(L.pb200_srs_setup_from_secret(mont(x), mont(gs * pow(x, first, R_MOD) % R_MOD), count, slice_raw))
        key = pd.ShardedCommitKey(slice_raw.raw[: 96 * count], n, comm, threshold=threshold, replica_raw=rep_raw.raw[: 96 * min(n, threshold)])
        del slice_raw
        # scalars s_i = u[i mod 4096] + v[i div 4096] (mod r) with random u, v: pairwise distinct full-range values
        # (uniform window digits), and p(x) = U(x) (x^n - 1)/(x^4096 - 1) + V(x^4096) (x^4096 - 1)/(x - 1) in closed form
        rng = random.Random(4096 + log_n)  # the same on every rank
        m = 4096
        u = [rng.randrange(R_MOD) for _ in range(m)]
        v = [rng.randrange(R_MOD) for _ in range(n // m)]
        sc = fr_outer_sum(torch, u, v)
        times = []
        total = None
        for it in range(args.msm_iters + 1):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            total = key.commit_dev(sc.data_ptr(), n, stream.cuda_stream)  # returns after its one synchronisation + host tail
            e1.record(stream)
            stream.synchronize()
            ms = pd.max_over_ranks(e0.elapsed_time(e1), torch.device("cuda", local))
            if it:
                times.append(ms)
        # [g p(x)] G as a one-point "key"
        xm = pow(x, m, R_MOD)
        ux = 0
        for c in reversed(u):
            ux = (ux * x + c) % R_MOD
        vx = 0
        for c in reversed(v):
            vx = (vx * xm + c) % R_MOD
        geo_n = (pow(x, n, R_MOD) - 1) * pow(xm - 1, -1, R_MOD) % R_MOD
        geo_m = (xm - 1) * pow(x - 1, -1, R_MOD) % R_MOD
        px = (ux * geo_n + vx * geo_m) % R_MOD
        want = ctypes.create_string_buffer(96)
        check(L.pb200_srs_setup_from_secret(mont(1), mont(gs * px % R_MOD), 1, want))
        ok = want.raw == total
        best = min(times)
        rows.append({"log_n": log_n, "gpus": world, "ms": best, "points_per_s": n / best * 1e3, "window_bits": key.window,
                     "collective": "ncclAllGather of digit sums (device-resident)" if key.uses_collective(n) else "none (replicated key below the threshold)",
                     "checked": bool(ok)})
        key.free()
        del sc
        torch.cuda.empty_cache()
        if not ok:
            raise SystemExit(f"sharded MSM 2^{log_n} differs from [p(x)]g on rank {rank}")
    if comm is not None:
        comm.destroy()
    return {"sizes": rows, "single_gpu_threshold_points": threshold,
            "scalars": "s_i = u[i mod 4096] + v[i div 4096] mod r, u and v uniform: distinct full-range scalars whose polynomial has a closed form"}


def fr_outer_sum(torch, u, v):
    """[len(v) * len(u), 4] int64 tensor on the GPU: Montgomery forms of (u[j] + v[k]) mod r at index k * len(u) + j.
    Montgomery form is linear, so it is a 256-bit modular addition of the two tables: 32-bit limbs in int64 lanes."""
    def limbs(vals):
        raw = b"".join(mont(x) for x in vals)
        t = torch.frombuffer(bytearray(raw), dtype=torch.int32).view(len(vals), 8).cuda().to(torch.int64)
        return t & 0xFFFFFFFF

    U, V = limbs(u), limbs(v)
    r_l = torch.tensor([(R_MOD >> (32 * i)) & 0xFFFFFFFF for i in range(8)], dtype=torch.int64, device="cuda")
    s = (V[:, None, :] + U[None, :, :]).reshape(-1, 8)  # limb sums < 2^33
    carry = torch.zeros(s.shape[0], dtype=torch.int64, device="cuda")
    for i in range(8):
        t = s[:, i] + carry
        s[:, i] = t & 0xFFFFFFFF
        carry = t >> 32
    # s < 2r < 2^256: subtract r where s >= r
    d = s.clone()
    borrow = torch.zeros_like(carry)
    for i in range(8):
        t = d[:, i] - r_l[i] - borrow
        borrow = (t < 0).to(torch.int64)
        d[:, i] = t & 0xFFFFFFFF
    ge = (carry > 0) | (borrow == 0)
    out = torch.where(ge[:, None], d, s)
    return (out[:, 0::2] | (out[:, 1::2] << 32)).contiguous()


def proof_2_20(L, torch):
    """BASELINE.json configs[2]: one proof of the reference's BenchCircuit at 2^20 gates (quotient on the 4n coset
    2^22, 2^20 + 7-point commit key) - byte parity at this size is tests/test_gpu_prover.py::test_gpu_prover_2_20_gates."""
    from plonk_b200 import Prover
    from plonk_b200._lib import check
    from plonk_b200.gadgets import bench_circuit

    log_gates = 20
    t0 = time.time()
    arrays = bench_circuit(1 << log_gates).arrays()
    n_srs = (1 << log_gates) + 7
    srs_raw = ctypes.create_string_buffer(n_srs * 96)
    check(L.pb200_srs_setup_from_secret(mont(SRS_X), mont(SRS_G), n_srs, srs_raw))
    prover = Prover(b"bench-2^20", arrays.constraints, arrays.selectors, arrays.wires, arrays.n_witnesses, srs_raw.raw)
    setup_s = time.time() - t0
    wit = torch.frombuffer(bytearray(arrays.witnesses), dtype=torch.uint8).cuda()
    out = ctypes.create_string_buffer(1008)
    stream = torch.cuda.Stream()
    times = []
    for it in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        check(L.pb200_prove_dev(prover._h, wit.data_ptr(), arrays.n_witnesses, arrays.pi_idx, arrays.pi_vals, arrays.n_pi, blinders_for(it), out, stream.cuda_stream))
        e1.record(stream)
        stream.synchronize()
        if it:
            times.append(e0.elapsed_time(e1))
    return {"proof_2^20_ms": min(times), "proof_2^20": {"gates": arrays.constraints, "circuit": "reference BenchCircuit<2^20>", "ms_all": times,
                                                        "compile_and_key_setup_s": setup_s, "proofs_in_flight": 1}}


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_msm_accumulate launch, from the text export of the
    ncu --set full capture of THIS build's kernel (profiles/ncu_r02_accumulate.json, written by tools/ncu_export.py);
    None when no capture of the current kernel is committed."""
    p = os.path.join(ROOT, "profiles", "ncu_r02_accumulate.json")
    try:
        d = json.load(open(p))
        return float(d["dram_bytes_read"]) + float(d["dram_bytes_write"]), f"profiles/ncu_r02_accumulate.json ({d.get('kernel', '?')}, {d.get('launch', '?')})"
    except (OSError, KeyError, ValueError):
        return None, "no committed capture of this build's kernel"


def ntt_microbench(L, torch, imad_peak):
    from plonk_b200._lib import check

    s = torch.cuda.Stream()
    out = {}
    with torch.cuda.stream(s):
        for log_n, batch in ((16, 4), (19, 5)):
            n = 1 << log_n
            x = torch.randint(0, 2**62, (batch * n, 4), dtype=torch.int64, device="cuda")
            y = torch.empty_like(x)
            f = lambda: check(L.pb200_ntt_dev(x.data_ptr(), n, y.data_ptr(), log_n, 0, 1, batch, n, n, s.cuda_stream))
            for _ in range(3):
                f()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.synchronize()
            e0.record(s)
            for _ in range(10):
                f()
            e1.record(s)
            s.synchronize()
            ms = e0.elapsed_time(e1) / 10
            bf = batch * (n // 2) * log_n / (ms * 1e-3)
            out[f"coset_ntt_2^{log_n}_batch{batch}"] = {"ms": ms, "butterflies_per_s": bf, "algorithmic_GBps": 64 * n * batch / ms / 1e6,
                                                         "alu_frac": bf / (imad_peak / IMAD_PER_BUTTERFLY)}
    return out


def cpu_kernel_rates(cref, srs, threads):
    """The two kernels on their own on the CPU, same sizes as the GPU microbenchmarks (SURVEY.md section 8d)."""
    import random

    rng = random.Random(19)
    n19 = 1 << (LOG_GATES + 3)
    vec = b"".join(mont(rng.randrange(R_MOD)) for _ in range(1 << 12)) * (n19 >> 12)
    t0 = time.time()
    for _ in range(2):
        cref.ntt(vec, LOG_GATES + 3, 0, 1, threads)
    ntt_s = (time.time() - t0) / 2
    scalars = vec[: SRS_POINTS * 32]
    t0 = time.time()
    cref.msm(srs, scalars, threads)
    msm_s = time.time() - t0
    window = int(math.log(SRS_POINTS)) + 2  # msm_variable_base's window rule (SURVEY.md section 8 row a8)
    return {"coset_ntt_2^19": {"ms": ntt_s * 1e3, "butterflies_per_s": (n19 // 2) * (LOG_GATES + 3) / ntt_s},
            "msm_2^16": {"ms": msm_s * 1e3, "points_per_s": SRS_POINTS / msm_s,
                         "bucket_adds_per_s": SRS_POINTS * math.ceil(255 / window) / msm_s, "window_bits": window}}


def cpu_baseline(n_proofs):
    """Restated reference (oracle/cref.cpp) on a bounded sample of the same workload.  It runs as the reference arm
    itself - `bench.py --impl reference` in a child process - so that the number is the one the arm reports: inside
    this process, next to torch's OpenMP runtime and the proving threads, the same code measured 2.3 x slower."""
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(n_proofs), "--warmup", "1", "--cpu-kernels"],
                         capture_output=True, text=True, timeout=900, env={k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "RANK", "WORLD_SIZE", "LOCAL_RANK")})
    line = json.loads(out.stdout.strip().splitlines()[-1])
    return line["cpu_baseline"]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import cref

    if args.circuit == "bench":
        # the reference arm runs none of the product's code: the circuit comes from the oracle's own composer
        # (byte-identical to the native one, tests/test_gadgets.py)
        from oracle import gadgets as oracle_gadgets

        comp = oracle_gadgets.GadgetComposer.initialized()
        oracle_gadgets.bench_circuit(comp, 1 << LOG_GATES)
        arrays = cref.CircuitArrays(comp)
        workload = (f"reference BenchCircuit<2^16> (benches/plonk.rs: {arrays.constraints} gates of all gadget families, "
                    "domain 2^16, quotient domain 2^19)")
    else:
        arrays, workload = build_workload(args.circuit)

    threads = cref.best_threads()
    srs = cref.srs_from_secret(SRS_POINTS, SRS_X, SRS_G, threads)
    prover = cref.CrefProver(LABEL, arrays, srs, threads)
    for i in range(args.warmup):
        prover.prove(blinders_for(i), arrays)
    t0 = time.time()
    for i in range(args.steps):
        proof = prover.prove(blinders_for(1000 + i), arrays)
    dt = time.time() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"proofs": [proof]})
    value = args.steps / dt
    sample = (f"each step = 1 proof of the 2^16-gate workload ({args.steps} timed after {args.warmup} warm-up); {cref.thread_policy()}; "
              "C++/OpenMP restatement (the Rust reference cannot be built here)")
    cpu = {"value": value, "unit": "proofs/s", "cores": threads, "kind": "port", "sample": sample}
    if args.cpu_kernels:
        cpu.update(cpu_kernel_rates(cref, srs, threads))
    print(json.dumps({
        "impl": "reference", "metric": "proofs/sec @ 2^16 gates", "value": value, "unit": "proofs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (CPU)", "data": "synthetic",
        "config": {"workload": workload, "proofs_per_step": 1},
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--inflight", type=int, default=int(os.environ.get("PB200_INFLIGHT", "12")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-kernels", action="store_true", help="(reference arm) also time one coset NTT 2^19 and one MSM 2^16 on the CPU")
    ap.add_argument("--no-msm-sweep", action="store_true", help="skip extra.msm_sweep (BASELINE.json configs[3])")
    ap.add_argument("--msm-sizes", default="16,18,20,22,24", help="log2 point counts of the sharded-MSM sweep")
    ap.add_argument("--msm-iters", type=int, default=3)
    ap.add_argument("--no-proof20", action="store_true", help="skip extra.proof_2^20_ms (BASELINE.json configs[2], N = 1 only)")
    ap.add_argument("--circuit", default="bench", choices=["bench", "synthetic"],
                    help="bench = the reference's BenchCircuit<2^16> (default); synthetic = random arithmetic gates")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the proofs of each timed region's last step as DIR/<name>.npy (float32 bytes)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        args.steps = args.steps if args.steps is not None else 3
        args.warmup = args.warmup if args.warmup is not None else 1
        run_reference(args)
    else:
        args.steps = args.steps if args.steps is not None else 20
        args.warmup = max(3, args.warmup if args.warmup is not None else 3)
        run_ours(args)


if __name__ == "__main__":
    main()
