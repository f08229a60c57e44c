#!/usr/bin/env python3
"""Benchmark of the phase-1 hot path (BASELINE.json metric: phase-1 contribute points/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--curve C] [--dump-outputs DIR]

One *step* = Phase1::computation over ONE chunk of the configuration BASELINE.json names for a
single B200: BLS12-377, 2^20 powers, chunk size 2^16 (262 145 points: 196 608 G1 + 65 537 G2),
synthetic accumulator (a previous contribution applied to the all-generator accumulator).

  value      points/s with the chunk already resident in HBM (sso_p1_contribute_dev), CUDA events
  e2e        points/s through the reference-facing host-buffer call with K chunks in flight
             (sso_p1_contribute_many_buf): per chunk H2D of the 31 MB challenge, compute, Blake2b hash-chain
             link, D2H of the 15 MB response; e2e.single_call = one chunk per call (sso_p1_contribute_buf)
  roofline   integer-pipe roofline of the dominant kernel (declared multiply-accumulates / event time
             / measured mad.wide.u32 peak), plus the per-kernel breakdown
  cpu_baseline  the oracle's C++ restatement of the reference algorithm on the host cores (bounded sample)

N > 1 (torchrun): every rank contributes its own chunk (chunks are independent: no data-path
collective, weak scaling); time = max over ranks.  --impl reference times the CPU restatement only.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the tree as it found it (it may be read-only)

CURVE_BITS = {"bls12_377": (12, 253), "bw6_761": (24, 377), "mnt4_753": (24, 753), "mnt6_753": (24, 753)}
G2_DEG = {"bls12_377": 2, "bw6_761": 1, "mnt4_753": 2, "mnt6_753": 3}
A_ZERO = {"bls12_377": True, "bw6_761": True, "mnt4_753": False, "mnt6_753": False}


def macs_per_fq_mul(limbs: int) -> int:
    return 2 * limbs * limbs + limbs            # SURVEY.md §8d: CIOS on L 32-bit limbs


GLV_KBITS = {"bls12_377": 129, "bw6_761": 191}
# dram__bytes_read.sum + dram__bytes_write.sum of one k_batch_exp_chunk launch on the bench workload, from the committed
# `ncu --set full` capture (profiles/r1_ncu_batch_exp_chunk_summary.csv): 3.64 GB read + 1.95 GB written.  The algorithmic
# bytes are 31.5 MB in + 38 MB of Jacobian intermediates out; the rest is the per-thread stack (window tables, by-reference
# point arguments, spills: 4.8 KB/thread x 37.9 k resident threads = 181 MB, more than the 126 MB L2).  207 GB/s: 3 % of HBM.
def ncu_dram_bytes_per_launch(curve: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, read from the committed summary of
    the newest `ncu --set full` capture of this curve under profiles/ (r<N>_ncu_batch_exp_chunk_summary[_curve].csv);
    None when no capture is committed.  -> (bytes, file name)"""
    import glob
    import re
    best = None
    for fn in glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_batch_exp_chunk_summary*.csv")):
        m = re.match(r"r(\d+)_ncu_batch_exp_chunk_summary(?:_(\w+))?\.csv", os.path.basename(fn))
        if not m or (m.group(2) or "bls12_377") != curve:
            continue
        if best is None or int(m.group(1)) > best[0]:
            best = (int(m.group(1)), fn)
    if best is None:
        return None, None
    tot = 0.0
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for line in open(best[1]):
        parts = line.strip().split(",")
        if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(parts[2]) * scale.get(parts[1], 1.0)
    return (tot or None), os.path.relpath(best[1], ROOT)


COOP_G2_DEFAULT = {"bls12_377": False, "bw6_761": False, "mnt4_753": True, "mnt6_753": True}      # csrc/curves.cuh::COOP_DEFAULT


def coop_g2(curve: str) -> bool:
    """Does the G2 half of a chunk run through the warp-cooperative bodies (csrc/coop.cuh)?  SSO_COOP_G2 = 0 / 1 forces it."""
    e = os.environ.get("SSO_COOP_G2", "")
    return COOP_G2_DEFAULT[curve] if not e else e[0] != "0"


def declared_work_per_point(curve: str, group: int):
    """Closed-form count of base-field multiplications and squarings (m, s) of the batch_exp kernel per point (DESIGN.md §4):
      read the point into Montgomery form            2 deg
      window table 1P..8P                            4 dbl + 3 madd
      affine table (all but the one-thread MNT6 G2)  6 F-mul (Z products) + 13 F-mul + 7 (1 S + 3 M) (normalisation)
                                                     + 3 F-mul (share of the per-block inversion tree)
      window loop, signed 4-bit digits               4 (NW - 1) dbl + additions on 15/16 of the windows:
         plain ladder (MNT4/6)   NW = ceil((bits+2)/4)   one addition per window
         GLV (BLS12-377 G1, BW6) NW = ceil((KBITS+2)/4)  two additions per window + one multiplication by beta (deg Fq-muls)
         2-way psi (MNT4/6 G2)   NW = 95                 two additions per window + the psi-image of the table entry
         4-way psi decomposition (BLS12-377 G2)  NW = 17  four additions per window + (4 + 2 + 2) Fq-muls for psi, psi^2, psi^3
      additions are mixed (madd) with the affine table, full Jacobian additions otherwise.
    Point formulas with unreduced operands (csrc/ec.cuh SSO_LAZY_EC): where the field's squaring is no cheaper than its
    multiplication (24-limb prime fields, Fq3) the doubling is 3 M + 4 S (a = 0) / 3 M + 6 S (a != 0) and the mixed addition
    8 M + 3 S — the same totals as the 2 M + 5 S / 1 M + 8 S / 7 M + 4 S counted below, and there M and S cost the same.
    Base-field cost of an extension operation: Fq2 mul = 3 M, Fq2 sqr = 2 M (complex squaring); Fq3 mul = sqr = 6 M;
    only prime-field squarings use the dedicated squaring (fewer multiply-accumulates, macs_per_fq_sqr).
    The warp-cooperative Fq2 body executes FOUR base multiplications per Fq2 product (two per lane); the declared work keeps
    Karatsuba's three — the roofline fraction is quoted on the algorithmic count, not on what the layout executes."""
    _, bits = CURVE_BITS[curve]
    deg = G2_DEG[curve] if group == 1 else 1
    M, S = {1: ((1, 0), (0, 1)), 2: ((3, 0), (2, 0)), 3: ((6, 0), (6, 0))}[deg]

    def comb(*terms):
        m = sum(k * t[0] for k, t in terms)
        sq = sum(k * t[1] for k, t in terms)
        return (m, sq)

    dbl = comb((2, M), (5, S)) if A_ZERO[curve] else comb((1, M), (8, S))
    madd = comb((7, M), (4, S))
    add = comb((11, M), (5, S))
    base = (1, 0)
    # MNT6-753 G2: Jacobian table in the one-thread-per-element body, affine table in the warp-cooperative body (the default)
    affine = not (curve == "mnt6_753" and group == 1) or coop_g2(curve)
    terms = [(2 * deg, base), (4, dbl), (3, madd)]
    if affine:
        terms += [(6 + 13 + 21 + 3, M), (7, S)]
    step = madd if affine else add
    if curve == "bls12_377" and group == 1:
        nw = 17
        terms += [(4 * (nw - 1), dbl), (4 * nw * 15.0 / 16.0, step), (nw * (15.0 / 16.0) * 8, base)]
    elif curve in GLV_KBITS:
        nw = (GLV_KBITS[curve] + 2 + 3) // 4
        terms += [(4 * (nw - 1), dbl), (2 * nw * 15.0 / 16.0, step), (nw * (15.0 / 16.0) * deg, base)]
    elif curve in ("mnt4_753", "mnt6_753") and group == 1:
        # 2-way psi decomposition (k = k0 + k1 |t - 1|, 378-bit halves): two additions per window, the second on the psi-image of
        # the table entry: Fq2 (affine table) 2 mul_base = 4 Fq-muls; Fq3 (Jacobian table) Frobenius of X, Y, Z (2 each) + 2 mul_base (3 each) = 12
        nw = (378 + 2 + 3) // 4
        terms += [(4 * (nw - 1), dbl), (2 * nw * 15.0 / 16.0, step), (nw * (15.0 / 16.0) * (4 if deg == 2 else 12), base)]
    else:
        nw = (bits + 2 + 3) // 4
        terms += [(4 * (nw - 1), dbl), (nw * 15.0 / 16.0, step)]
    return comb(*terms)


VECTOR_NAMES = ("tau_powers_g1", "tau_powers_g2", "alpha_tau_powers_g1", "beta_tau_powers_g1", "beta_g2")
VECTOR_GROUPS = (0, 1, 0, 0, 1)
DUMP_BUDGET = 64 * 10 ** 6


def accumulator_vectors(buf, sz, es, compressed):
    """Splits an accumulator or a contribution (64-byte hash slot first) into its five point vectors:
    [(name, uint8 array of shape (points, point bytes))]."""
    counts = (sz["g1_count"], sz["other_count"], sz["other_count"], sz["other_count"], 1)
    out, off = [], 64
    for name, cnt, g in zip(VECTOR_NAMES, counts, VECTOR_GROUPS):
        pb = es[("g1" if g == 0 else "g2") + ("_c" if compressed else "_u")]
        out.append((name, buf[off:off + cnt * pb].reshape(cnt, pb)))
        off += cnt * pb
    return out


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes every (name, uint8 array of shape (rows, bytes per row)) as out_dir/<name>.npy in float32, one
    byte per element, so that two builds can be compared output for output.  When the arrays together would exceed
    DUMP_BUDGET bytes, each keeps the same fraction of its rows (at least one), chosen with a fixed seed, and the kept row
    indices go to out_dir/<name>_rows.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    full = sum(a.size * 4 for _, a in arrays)
    sampled = full > DUMP_BUDGET - 4096 * len(arrays)
    frac = (DUMP_BUDGET - 8192 * len(arrays)) / sum(a.size * 4 + a.shape[0] * 8 for _, a in arrays) if sampled else 1.0
    rng = np.random.default_rng(20)
    for name, a in arrays:
        if sampled:
            rows = np.sort(rng.choice(a.shape[0], max(1, int(a.shape[0] * frac)), replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def macs_per_fq_sqr(limbs: int) -> int:
    """csrc/fp.cuh: the point formulas use the dedicated squaring up to 12 limbs (SSO_SQR_EC_MAX_L), mul(a, a) above"""
    if limbs > 12:
        return macs_per_fq_mul(limbs)
    return limbs * (limbs + 1) // 2 + limbs * limbs + limbs      # mont_sqr


def declared_fq_muls_per_point(curve: str, group: int) -> float:
    m, sq = declared_work_per_point(curve, group)
    return m + sq


def declared_macs_per_point(curve: str, group: int) -> float:
    limbs, _ = CURVE_BITS[curve]
    m, sq = declared_work_per_point(curve, group)
    return m * macs_per_fq_mul(limbs) + sq * macs_per_fq_sqr(limbs)


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.05)
        except Exception as e:  # NVML missing: report nothing rather than fail the bench
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def cpu_reference_run(curve: str, power: int, chunk_log: int, steps: int, warmup: int, target_s: float):
    """Times the C++ restatement of the reference algorithm (oracle/c) on the host cores on a bounded
    sample of the workload: a chunk of the same curve and vector mix with fewer points."""
    from oracle import cport, phase1, synth
    from oracle.params import Phase1Params
    threads = cport.hw_threads()
    # calibrate on 2^6-point vectors, then size the sample for ~target_s per step
    def one(clog):
        o = Phase1Params.new_chunk(curve, 1, 1 << clog, clog + 4, 1 << clog)
        ch = phase1.new_challenge(o)
        k1 = phase1.PrivateKey(*synth.scalars_from_seed(o.curve, synth.SEED_PREV))
        t0 = time.perf_counter()
        cport.contribute_with_key(o, ch, k1, bytes(o.public_key_size), threads=threads)
        return time.perf_counter() - t0, o.g1_count + 3 * o.other_count + 1
    t, n = one(8)
    rate = n / t
    clog = 8
    while clog < chunk_log and (4 << (clog + 1)) / rate < target_s:
        clog += 1
    times = []
    for it in range(warmup + steps):
        t, n = one(clog)
        if it >= warmup:
            times.append(t)
    mean = sum(times) / len(times)
    return {"value": n / mean, "unit": "points/s", "cores": threads, "kind": "port",
            "caveats": "a C++ restatement of the reference algorithm, not the Rust binary (no toolchain in the image): unsigned __int128 limbs "
                       "without the x86 assembly of ark-ff-asm, per-point double-and-add without the BatchInversion mode of batch_exp; "
                       "a stated baseline, not the target",
            "sample": "%s chunk of 2^%d elements per vector (%d points) per step, %d steps; C++ restatement of "
                      "per-index pow + double-and-add + batch normalisation (oracle/c/oracle.cpp), std::thread over points"
                      % (curve, clog, n, len(times))}, mean


def run_phase2(args, rank, world, local_rank):
    """--workload phase2 (BASELINE config 4): the delta^-1 scaling of a Groth16 H or L query of n G1 points
    (phase2_cli::contribute -> batch_mul, reference src/bin/contribute.rs:827-838), synthetic vectors of the sizes the
    Nimiq circuits have (2^19 .. 2^22, reference e2e/nimiq_e2e.sh:61-71).  value: device-resident points/s (sso_batch_mul_dev);
    e2e: sso_p2_scale_queries_buf from pinned host buffers.  Every rank scales its own vector (no collective)."""
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import snark_setup_operator_b200 as sso
    from snark_setup_operator_b200 import phase2 as p2
    from snark_setup_operator_b200.phase1 import curve_sizes
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = local_rank
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    name = args.curve
    es = curve_sizes(name)
    limbs, bits = CURVE_BITS[name]
    n = 1 << args.query_log
    tau = int.from_bytes(bytes(range(1, 33)), "little") >> 8
    delta_inv = int.from_bytes(bytes(range(7, 7 + 128)), "little") >> (1024 - (bits - 1))
    # a vector of distinct subgroup points: tau^i * G
    d_gen = torch.frombuffer(bytearray(n * es["g1_u"]), dtype=torch.uint8).cuda()
    pchunk = sso.Phase1Parameters.new_chunk(name, 0, 1, 1, 1)
    d_one = torch.empty(pchunk.accumulator_size, dtype=torch.uint8, device="cuda")
    sso.new_challenge_dev(pchunk, d_one, device=dev)
    d_gen.view(n, es["g1_u"])[:] = d_one[64:64 + es["g1_u"]]
    d_in = torch.empty(n * es["g1_u"], dtype=torch.uint8, device="cuda")
    d_c = torch.empty(n * es["g1_c"], dtype=torch.uint8, device="cuda")
    sso.batch_exp(name, 0, d_gen, n, 1 + rank, tau, None, d_c, device=dev)
    sso.reencode(name, 0, d_c, n, d_in, check=sso.CHECK_NO, subgroup_check=False, device=dev)
    del d_gen, d_c
    d_out = torch.empty(n * es["g1_u"], dtype=torch.uint8, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    h_in = torch.empty(n * es["g1_u"], dtype=torch.uint8).pin_memory()
    h_in.copy_(d_in)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(fn, k):
        tot = 0.0
        for _ in range(k):
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); e1.synchronize()
            tot += e0.elapsed_time(e1)
        return tot

    step = lambda: sso.batch_mul(name, 0, d_in, n, delta_inv, d_out, in_compressed=False, out_compressed=False, check=sso.CHECK_NO, device=dev)
    run_steps(step, args.warmup)
    sso.profile_reset()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    ms = run_steps(step, args.steps)
    barrier()
    last_out = d_out.cpu().numpy() if args.dump_outputs and rank == 0 else None
    launches = sum(v["launches"] for v in sso.profile_read().values()) // max(1, args.steps)
    sso.profile_reset(); sso.profile_enable(2)
    run_steps(step, args.steps)
    sso.profile_enable(False)
    prof = sso.profile_read()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    h_out = torch.empty(n * es["g1_u"], dtype=torch.uint8).pin_memory()
    e2e_fn = lambda: p2.scale_queries(name, h_in, n, delta_inv, device=dev, out=h_out)
    run_steps(e2e_fn, 1)
    ms_e2e = run_steps(e2e_fn, args.steps)
    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        peak = sso.imad_peak(0, dev)
        k = prof["batch_exp_g1"]
        macs = k["elems"] * declared_macs_per_point(name, 0)
        achieved = macs / (k["ms"] * 1e-3) if k["ms"] > 0 else None
        ms_step, ms_e2e_step = t[0].item() / args.steps, t[1].item() / args.steps
        line = {"metric": "phase2_scale_points_per_s", "value": world * n / (ms_step * 1e-3), "unit": "points/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u32 limbs (Montgomery, integer pipe)", "data": "synthetic",
                "config": {"workload": "phase-2 %s: delta^-1 scaling of a query vector of 2^%d G1 points (uncompressed in and out)" % (name, args.query_log),
                           "curve": name, "points": n, "l2": "flushed between timed steps (256 MiB write)"},
                "e2e": {"value": world * n / (ms_e2e_step * 1e-3), "unit": "points/s", "ms_per_step": ms_e2e_step,
                        "h2d_bytes_per_step": n * es["g1_u"], "d2h_bytes_per_step": n * es["g1_u"], "call": "sso_p2_scale_queries_buf"},
                "gpu_launches": launches,
                "roofline": {"bound": "imad", "kernel": "k_batch_exp<G1> (one shared scalar)", "achieved": achieved / 1e12 if achieved else None,
                             "peak": peak / 1e12, "unit": "TMAC/s", "frac": achieved / peak if achieved else None, "traffic": None,
                             "fq_muls_per_point": round(declared_fq_muls_per_point(name, 0), 1),
                             "kernels": {kk: {"launches": v["launches"], "ms_total": round(v["ms"], 3)} for kk, v in prof.items() if v["launches"]}},
                "clocks": sampler.summary()}
        if last_out is not None:
            dump_outputs(args.dump_outputs, [("scaled_query_g1", last_out.reshape(n, es["g1_u"]))])
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()


def run_verify_transcript(args, rank, world, local_rank):
    """--workload verify_transcript: one pass of what the operator's verify_transcript binary drives through the crate
    boundary for a phase-1 ceremony with one contribution per chunk (reference src/bin/verify_transcript.rs:293-569, 602-607,
    675-696, 745-776, 811-822), on files in tmpfs:
      chunk loop   per chunk: regenerate the round-0 challenge and compare its hash, transform_pok_and_correctness of the
                   contribution — chunks dealt round-robin over the ranks, no collective
      combine      cooperative: every rank decodes its share of the pieces into the shared combined file
      beacon       phase1_cli::contribute on the combined accumulator, Full mode, cooperative (pieces of batch_size)
      verify       transform_pok_and_correctness of the beacon contribution, Full mode, cooperative; the partial MSM results of
                   the ranks meet in ONE NCCL all-gather
      ratios       transform_ratios on the final accumulator, cooperative, ONE NCCL all-gather
    value = seconds per pass (max over ranks); setup (new_challenge + the contributions being verified) is not timed."""
    import hashlib
    import shutil
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import torch
    import snark_setup_operator_b200 as sso
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = local_rank
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        sso.dist_init_from_torch(dev)
    name, power, cs, batch = args.curve, args.power, 1 << args.chunk_log, 1 << args.batch_log
    base = [None]
    if rank == 0:
        root = "/dev/shm" if os.path.isdir("/dev/shm") else None
        base[0] = tempfile.mkdtemp(prefix="sso_bench_", dir=root)
    if dist is not None:
        dist.broadcast_object_list(base, src=0)
    base = base[0]
    f = lambda n: os.path.join(base, n)
    p0 = sso.Phase1Parameters.new_chunk(name, 0, cs, power, batch)
    pf = sso.Phase1Parameters.new_full(name, power, batch)
    sz0 = p0.sizes()
    nchunks = sz0["num_chunks"]
    full = pf.sizes()
    npts = full["g1_count"] + 3 * full["other_count"] + 1
    seed = bytes(range(32))
    beacon = hashlib.blake2s(b"bench beacon").digest()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def chunk_params(k):
        return sso.Phase1Parameters.new_chunk(name, k, cs, power, batch)

    # ---- setup: round 0 and one contribution per chunk (the transcript being verified)
    t_setup = time.perf_counter()
    for k in range(rank, nchunks, world):
        sso.new_challenge(f("ch%d" % k), f("ch%d.hash" % k), chunk_params(k), device=dev)
        sso.contribute(f("ch%d" % k), f("ch%d.h2" % k), f("resp%d" % k), f("resp%d.hash" % k), sso.CHECK_NONZERO, 0, chunk_params(k), seed, device=dev)
    barrier()
    if rank == 0:
        open(f("list"), "w").write("\n".join(f("resp%d" % k) for k in range(nchunks)))
    barrier()
    t_setup = time.perf_counter() - t_setup
    outputs = ["combined", "combined.hash", "beacon", "beacon.hash", "c.vhash", "b.vhash", "final", "final.hash"]

    def clean():
        for k in range(rank, nchunks, world):
            for n in ("regen%d", "regen%d.hash", "ch%d.vhash", "resp%d.vhash", "new%d", "new%d.hash"):
                if os.path.exists(f(n % k)):
                    os.remove(f(n % k))
        if rank == 0:
            for n in outputs:
                if os.path.exists(f(n)):
                    os.remove(f(n))
        barrier()

    phases = ("chunks", "combine", "beacon", "verify", "ratios")

    def one_pass():
        t = {}
        barrier()
        t0 = time.perf_counter()
        def one_chunk(k):
            pk = chunk_params(k)
            sso.new_challenge(f("regen%d" % k), f("regen%d.hash" % k), pk, device=dev)                    # verify_transcript.rs:316-361
            assert open(f("regen%d.hash" % k), "rb").read() == open(f("ch%d.hash" % k), "rb").read()
            sso.transform_pok_and_correctness(f("ch%d" % k), f("ch%d.vhash" % k), sso.CHECK_NO, f("resp%d" % k), f("resp%d.vhash" % k),
                                              sso.CHECK_NONZERO, f("new%d" % k), f("new%d.hash" % k), 0, True, pk, device=dev)
        # the chunk loop as a work queue: three chunks in flight per rank (the serial tails of one chunk — pairings, MSM folds —
        # overlap the decompression of the next); the hash-chain order across rounds stays with the caller
        with ThreadPoolExecutor(args.lanes) as ex:
            list(ex.map(one_chunk, range(rank, nchunks, world)))
        barrier()
        t["chunks"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sso.combine(f("list"), f("combined"), p0, device=dev)
        barrier()
        t["combine"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sso.contribute(f("combined"), f("combined.hash"), f("beacon"), f("beacon.hash"), sso.CHECK_NONZERO, 0, pf, beacon, device=dev)
        barrier()
        t["beacon"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sso.transform_pok_and_correctness(f("combined"), f("c.vhash"), sso.CHECK_NO, f("beacon"), f("b.vhash"), sso.CHECK_NONZERO, f("final"),
                                          f("final.hash"), 0, True, pf, device=dev)
        barrier()
        t["verify"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        sso.transform_ratios(f("final"), sso.CHECK_NO, pf, device=dev)
        barrier()
        t["ratios"] = time.perf_counter() - t0
        return t

    sampler = ClockSampler(local_rank)
    try:
        for _ in range(max(1, args.warmup)):
            clean()
            one_pass()
        sampler.start()
        totals = {k: 0.0 for k in phases}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev_ms = 0.0
        for _ in range(args.steps):
            clean()
            e0.record()
            t = one_pass()
            e1.record()
            e1.synchronize()
            ev_ms += e0.elapsed_time(e1)
            for k in phases:
                totals[k] += t[k]
        sampler.stop_flag = True
        if sampler.is_alive():
            sampler.join(timeout=2)
        vals = torch.tensor([totals[k] for k in phases] + [ev_ms / 1e3], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        stats = sso.dist_stats()
        final_hash = open(f("final.hash"), "rb").read().hex() if rank == 0 else None
        if args.dump_outputs and rank == 0:
            import numpy as np
            final = np.fromfile(f("final"), dtype=np.uint8)
            dumped = [("final_hash", np.frombuffer(bytes.fromhex(final_hash), dtype=np.uint8).reshape(1, 64))]
            dump_outputs(args.dump_outputs, dumped + accumulator_vectors(final, full, sso.phase1.curve_sizes(name), False))
    finally:
        barrier()
        if rank == 0:
            shutil.rmtree(base, ignore_errors=True)
    if rank == 0:
        per = {k: vals[i].item() / args.steps for i, k in enumerate(phases)}
        total_s = vals[len(phases)].item() / args.steps
        es = sso.phase1.curve_sizes(name)
        line = {"metric": "verify_transcript_s", "value": total_s, "unit": "s", "n_gpus": world, "steps": args.steps, "warmup": max(1, args.warmup),
                "ms_per_step": total_s * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
                "dtype": "u32 limbs (Montgomery, integer pipe)", "data": "synthetic",
                "config": {"workload": "verify_transcript of a phase-1 %s 2^%d-power ceremony, %d chunks of 2^%d, one contribution per chunk, beacon "
                                       "applied, batch_size 2^%d; files in tmpfs" % (name, power, nchunks, args.chunk_log, args.batch_log),
                           "curve": name, "power": power, "chunk_size": cs, "batch_size": batch, "points": npts, "chunks_in_flight_per_rank": args.lanes,
                           "accumulator_bytes": full["accumulator_size"],
                           "sharding": "chunks round-robin over ranks; Full-mode calls cooperative in batch_size pieces; partial MSM results: one "
                                       "NCCL all-gather per Full-mode verification and per transform_ratios"},
                "phases_s": per, "points_per_s": npts / total_s, "setup_s": t_setup,
                "nccl": {"ranks": stats["world"] if stats["initialised"] else 1, "all_gathers_total": stats["all_gathers"], "version": stats["nccl_version"]},
                "final_hash": final_hash, "clocks": sampler.summary(), "point_bytes": es}
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if dist is not None:
        sso.dist_finalize()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--curve", default="bls12_377")
    ap.add_argument("--power", type=int, default=20)
    ap.add_argument("--chunk-log", type=int, default=16)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="contribute", choices=["contribute", "verify_transcript", "phase2"])
    ap.add_argument("--query-log", type=int, default=20, help="phase2 workload: log2 of the query length")
    ap.add_argument("--batch-log", type=int, default=None, help="log2 of Phase1Parameters::batch_size (default: the chunk size)")
    ap.add_argument("--lanes", type=int, default=3, help="verify_transcript workload: chunks in flight per rank")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (rank 0) as DIR/<name>.npy, float32, "
                         "at most 64 MB in all; the inputs are the same from run to run, so two builds can be compared")
    args = ap.parse_args()
    if args.batch_log is None:
        args.batch_log = args.chunk_log
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = "phase-1 %s 2^%d powers, chunk 2^%d: single-chunk contribute" % (args.curve, args.power, args.chunk_log)
    config = {"workload": workload, "curve": args.curve, "power": args.power, "chunk_size": 1 << args.chunk_log,
              "sharding": "one chunk per rank, no data-path collective", "l2": "flushed between timed steps (256 MiB write)"}

    if args.workload == "verify_transcript" and args.impl == "ours":
        return run_verify_transcript(args, rank, world, local_rank)
    if args.workload == "phase2" and args.impl == "ours":
        return run_phase2(args, rank, world, local_rank)
    if args.impl == "reference":
        if rank != 0:
            return
        cb, mean = cpu_reference_run(args.curve, args.power, args.chunk_log, max(1, args.steps), max(0, args.warmup), 6.0)
        line = {"impl": "reference", "metric": "phase1_contribute_points_per_s", "value": cb["value"], "unit": "points/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (Montgomery)",
                "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # the contract is ONE JSON line on stdout: libraries that chat on fd 1 (NCCL prints its version banner there)
    # are sent to stderr, and the line is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    import torch
    import snark_setup_operator_b200 as sso
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = local_rank
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # ---- synthetic input, built on the device by the product itself (validated by tests/): the
    # all-generator accumulator, one contribution with the "previous contributor" scalars, decompressed.
    chunk_index = 1 + rank                      # every rank owns a different (full) chunk
    cs = 1 << args.chunk_log
    p = sso.Phase1Parameters.new_chunk(args.curve, chunk_index, cs, args.power, cs)
    sz = p.sizes()
    acc, contrib = sz["accumulator_size"], sz["contribution_size"]
    npts = sz["g1_count"] + 3 * sz["other_count"] + 1
    from snark_setup_operator_b200.phase1 import curve_sizes
    es = curve_sizes(args.curve)

    def scalars(seed_byte):
        # deterministic non-trivial scalars without the oracle: Blake2b of a seed, reduced by truncation
        import hashlib
        out = []
        for i in range(3):
            h = b"".join(hashlib.blake2b(bytes([seed_byte, i, j]), digest_size=64).digest() for j in range(2))
            out.append(int.from_bytes(h, "little") >> (1024 - (CURVE_BITS[args.curve][1] - 1)))
        return out

    prev, mine = scalars(0x5E), scalars(0x01)
    d_gen = torch.empty(acc, dtype=torch.uint8, device="cuda")
    sso.new_challenge_dev(p, d_gen, device=dev)
    d_resp = torch.zeros(contrib, dtype=torch.uint8, device="cuda")
    sso.contribute_dev(p, d_gen, d_resp, *prev, check=sso.CHECK_NO, device=dev)
    d_ch = torch.empty(acc, dtype=torch.uint8, device="cuda")
    d_ch[:64] = d_gen[:64]
    for g, (_, src), (_, dst) in zip(VECTOR_GROUPS, accumulator_vectors(d_resp, sz, es, True), accumulator_vectors(d_ch, sz, es, False)):
        if src.shape[0]:
            sso.reencode(args.curve, g, src, src.shape[0], dst, check=sso.CHECK_NO, subgroup_check=False, device=dev)
    del d_gen
    h_ch = torch.empty(acc, dtype=torch.uint8).pin_memory()
    h_ch.copy_(d_ch)
    h_resp = torch.empty(contrib, dtype=torch.uint8).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    pubkey = bytes(sz["public_key_size"])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(fn, n, timed):
        """Each step is bracketed by CUDA events on the current stream; the library call is synchronous
        (returns when its internal streams drained), so the bracket covers the whole step."""
        total = 0.0
        for _ in range(n):
            flush.zero_()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            total += e0.elapsed_time(e1)
        return total

    step_dev = lambda: sso.contribute_dev(p, d_ch, d_resp, *mine, check=sso.CHECK_NONZERO, device=dev)
    step_e2e = lambda: sso.contribute_buf(p, h_ch, h_resp, *mine, pubkey=pubkey, check=sso.CHECK_NONZERO, device=dev)

    # ---- device-resident timing (value)
    run_steps(step_dev, args.warmup, False)
    sso.profile_reset()
    sampler = ClockSampler(local_rank)
    if not os.environ.get("SSO_BENCH_NOSAMPLER"):
        sampler.start()
    barrier()
    ms_total = run_steps(step_dev, args.steps, True)
    barrier()
    last_resp = d_resp.cpu().numpy() if args.dump_outputs and rank == 0 else None
    launches_total = sum(v["launches"] for v in sso.profile_read().values())
    # ---- roofline pass: the same steps with every kernel timed by CUDA events on its launching stream and
    # the two streams of a call serialised, so that each kernel's time is its time alone on the GPU
    sso.profile_reset()
    sso.profile_enable(2)
    run_steps(step_dev, args.steps, True)
    sso.profile_enable(False)
    prof = sso.profile_read()
    # the NVML sampler covers the device-resident timed region and the roofline pass; it is stopped before the end-to-end
    # passes because its queries contend with the CUDA calls of the host worker threads (measured: 27.7 ms per chunk without,
    # outliers of 34-40 ms with the sampler polling)
    sampler.stop_flag = True
    if sampler.is_alive():
        sampler.join(timeout=2)
    quick = bool(os.environ.get("SSO_BENCH_QUICK"))       # kernel A/B runs: device-resident value + roofline pass only
    ms_e2e_total = ms_e2e_single_total = ms_e2e_seeded_total = ms_e2e_seeded_many_total = float("nan")
    e2e_same = None
    if not quick:
        # ---- end-to-end timing through the host-buffer entry point
        # (a) one chunk per call: the latency of a single reference-facing call (hash of the 31 MB challenge on one core inside)
        run_steps(step_e2e, 1, False)
        barrier()
        ms_e2e_single_total = run_steps(step_e2e, args.steps, True)
        barrier()
        h_resp_single = h_resp.clone()
        # (a') the whole of phase1_cli::contribute on host buffers: key generation from the seed, proofs of knowledge, computation
        step_seeded = lambda: sso.contribute_seeded_buf(p, h_ch, h_resp, bytes(range(32)), check=sso.CHECK_NONZERO, device=dev)
        run_steps(step_seeded, 1, False)
        ms_e2e_seeded_total = run_steps(step_seeded, args.steps, True)
        barrier()
        # (b) the headline: the same K steps with several chunks in flight (sso_p1_contribute_many_buf, the reference's
        # Process lane): every step still copies its own challenge from pinned host memory and reads its own response back
        n_resp = min(args.steps, 64)
        h_resps = [torch.empty(contrib, dtype=torch.uint8).pin_memory() for _ in range(n_resp)]

        def many(n):
            done = 0
            while done < n:
                k = min(n_resp, n - done)
                sso.contribute_many_buf([p] * k, [h_ch] * k, h_resps[:k], *mine, pubkey=pubkey, check=sso.CHECK_NONZERO, device=dev)
                done += k

        many(min(3, args.steps))
        flush.zero_()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        many(args.steps)
        e1.record()
        e1.synchronize()
        ms_e2e_total = e0.elapsed_time(e1)
        barrier()
        e2e_same = all(torch.equal(h_resps[i], h_resp_single) for i in range(n_resp))
        # (b') the same with the full call (key generation + proofs of knowledge per chunk), six host workers
        def many_seeded(n):
            done = 0
            while done < n:
                k = min(n_resp, n - done)
                sso.contribute_seeded_many_buf([p] * k, [h_ch] * k, h_resps[:k], bytes(range(32)), check=sso.CHECK_NONZERO, host_threads=6,
                                               device=dev)
                done += k

        many_seeded(min(4, args.steps))
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        many_seeded(args.steps)
        e1.record()
        e1.synchronize()
        ms_e2e_seeded_many_total = e0.elapsed_time(e1)
        barrier()
    # (c) the call the operator makes: phase1_cli::contribute on FILES (tmpfs), one call per process-lane slot
    # (--max-in-process-lane threads, reference src/bin/contribute.rs:118-123, 809-823): mmap of the challenge, key generation,
    # proofs of knowledge, computation, Blake2b of challenge and response, response + 2 hash files written and renamed
    file_call = None
    if not quick:
        import shutil
        import tempfile
        from concurrent.futures import ThreadPoolExecutor
        tdir = tempfile.mkdtemp(prefix="sso_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        try:
            ch_fn = os.path.join(tdir, "challenge")
            with open(ch_fn, "wb") as fh:
                fh.write(h_ch.numpy().tobytes())

            def one_file(i):
                out = [os.path.join(tdir, "%s_%d" % (n, i)) for n in ("challenge.hash", "response", "response.hash")]
                for o in out:
                    if os.path.exists(o):
                        os.remove(o)
                sso.contribute(ch_fn, out[0], out[1], out[2], sso.CHECK_NONZERO, 0, p, bytes(range(32)), device=dev)

            one_file(0)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(args.steps):
                one_file(0)
            t_single = (time.perf_counter() - t0) / args.steps
            lanes = 8
            with ThreadPoolExecutor(lanes) as ex:
                list(ex.map(one_file, range(lanes)))
                n_calls = max(lanes, 2 * args.steps)
                t0 = time.perf_counter()
                list(ex.map(one_file, range(lanes, lanes + n_calls)))          # distinct outputs per call (lanes run concurrently)
                t_lanes = (time.perf_counter() - t0) / n_calls
            file_call = {"single_call": {"value": npts / t_single, "ms_per_step": t_single * 1e3},
                         "lanes": {"value": npts / t_lanes, "ms_per_step": t_lanes * 1e3, "process_lanes": lanes},
                         "unit": "points/s (this rank)",
                         "call": "sso_p1_contribute_file on tmpfs: everything phase1_cli::contribute does, files in and out"}
        finally:
            shutil.rmtree(tdir, ignore_errors=True)
    sampler.stop_flag = True
    if sampler.is_alive():
        sampler.join(timeout=2)
    # ---- chunk verification (BASELINE metric, second half: "chunk verify s"): transform_pok_and_correctness on host
    # buffers — hash chain, 3 proofs of knowledge, decompression + subgroup checks, RLC power-ratio MSMs, pairings
    verify = None
    if rank == 0 and not os.environ.get("SSO_BENCH_NOVERIFY"):
        seed = bytes(range(32))
        sso.contribute_seeded_buf(p, h_ch, h_resp, seed, check=sso.CHECK_NO, device=dev)
        h_new = torch.empty(acc, dtype=torch.uint8).pin_memory()
        vt = []
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sso.verify_chunk_buf(p, h_ch, h_resp, h_new, ratio_check=True, device=dev)
            vt.append(time.perf_counter() - t0)
        # the chunk loop of verify_transcript as a work queue: six chunks in flight on three host workers
        n_v = 6
        h_news = [h_new] + [torch.empty(acc, dtype=torch.uint8).pin_memory() for _ in range(n_v - 1)]
        sso.verify_chunk_many_buf([p] * 3, [h_ch] * 3, [h_resp] * 3, h_news[:3], ratio_check=True, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sso.verify_chunk_many_buf([p] * n_v, [h_ch] * n_v, [h_resp] * n_v, h_news, ratio_check=True, device=dev)
        v_many = (time.perf_counter() - t0) / n_v
        verify = {"s_per_chunk": min(vt[1:]), "runs_s": [round(x, 4) for x in vt], "s_per_chunk_in_flight": v_many,
                  "in_flight": "sso_p1_verify_chunk_many_buf, %d chunks, 3 host workers" % n_v,
                  "what": "sso_p1_verify_chunk_buf: hash chain, PoK pairings, decompress + direct subgroup checks of %d points, "
                          "RLC power-ratio MSMs, same_ratio pairings; host buffers" % npts}

    t = torch.tensor([ms_total, ms_e2e_total, ms_e2e_single_total, ms_e2e_seeded_total, ms_e2e_seeded_many_total], dtype=torch.float64,
                     device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t[0].item() / args.steps
    ms_e2e = t[1].item() / args.steps
    ms_e2e_single = t[2].item() / args.steps
    ms_e2e_seeded = t[3].item() / args.steps
    ms_e2e_seeded_many = t[4].item() / args.steps
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    limbs, _ = CURVE_BITS[args.curve]
    mac = macs_per_fq_mul(limbs)
    peak = sso.imad_peak(0, dev)                 # independent mad.wide.u32 chains: the integer-MAC ceiling of the chip
    peak_chain = sso.imad_peak(1, dev)           # mad.lo.cc/madc.hi.cc carry chains: what carry-propagating limbs can reach
    kernels = []
    n_g1 = sz["g1_count"] + 2 * sz["other_count"]
    n_g2 = sz["other_count"] + 1
    fm1, fm2 = declared_fq_muls_per_point(args.curve, 0), declared_fq_muls_per_point(args.curve, 1)
    k = prof["batch_exp_chunk"]
    if k["launches"] and k["ms"] > 0:
        macs = k["launches"] * (n_g1 * declared_macs_per_point(args.curve, 0) + n_g2 * declared_macs_per_point(args.curve, 1))   # both groups run in the one launch
        achieved = macs / (k["ms"] * 1e-3)
        kernels.append({"kernel": "k_batch_exp_chunk", "launches": k["launches"], "ms_total": round(k["ms"], 3),
                        "points": k["elems"], "fq_muls_per_point": {"g1": round(fm1, 1), "g2": round(fm2, 1)},
                        "achieved_tmacs": achieved / 1e12, "frac": achieved / peak})
    for kind, grp in (("batch_exp_g1", 0), ("batch_exp_g2", 1)):
        k = prof[kind]
        if k["launches"] and k["ms"] > 0:
            fm = declared_fq_muls_per_point(args.curve, grp)
            achieved = k["elems"] * declared_macs_per_point(args.curve, grp) / (k["ms"] * 1e-3)
            kernels.append({"kernel": "k_" + kind, "launches": k["launches"], "ms_total": round(k["ms"], 3),
                            "points": k["elems"], "fq_muls_per_point": round(fm, 1), "achieved_tmacs": achieved / 1e12,
                            "frac": achieved / peak})
    for kind in ("normalize_chunk", "normalize_g1", "normalize_g2", "tau_tables"):
        k = prof[kind]
        if k["launches"]:
            kernels.append({"kernel": "k_" + kind, "launches": k["launches"], "ms_total": round(k["ms"], 3), "points": k["elems"]})
    dom = max((k for k in kernels if "frac" in k), key=lambda k: k["ms_total"], default={"kernel": None, "achieved_tmacs": None, "frac": None})
    launches = launches_total // max(1, args.steps)
    line = {
        "metric": "phase1_contribute_points_per_s", "value": world * npts / (ms_step * 1e-3), "unit": "points/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (Montgomery, integer pipe)", "data": "synthetic",
        "config": config,
        # headline e2e: the call the operator makes — phase1_cli::contribute on files, one call per process-lane slot; the host-buffer
        # entries below it explain where the time goes (in_memory = the same chunks from pinned buffers with scalars given)
        "e2e": {"value": (world * file_call["lanes"]["value"]) if file_call else world * npts / (ms_e2e * 1e-3), "unit": "points/s",
                "h2d_bytes_per_step": acc, "d2h_bytes_per_step": contrib - 64 - sz["public_key_size"],
                "ms_per_step": file_call["lanes"]["ms_per_step"] if file_call else ms_e2e,
                "call": ("sso_p1_contribute_file on tmpfs, %d process lanes per GPU: file read into page-locked staging, key generation from the "
                         "seed, proofs of knowledge, H2D + kernels + D2H, Blake2b of challenge and response, response and two hash files written "
                         "and renamed" % file_call["lanes"]["process_lanes"]) if file_call else "sso_p1_contribute_many_buf",
                "in_memory": {"value": world * npts / (ms_e2e * 1e-3), "ms_per_step": ms_e2e,
                              "call": "sso_p1_contribute_many_buf: K chunks from pinned host buffers, 3 host workers, each chunk = H2D + kernels + "
                                      "Blake2b(challenge) + D2H; responses identical to the single-chunk call: %s" % e2e_same},
                "single_call": {"value": world * npts / (ms_e2e_single * 1e-3), "ms_per_step": ms_e2e_single,
                                "call": "sso_p1_contribute_buf, one chunk per call (Blake2b of the challenge on one host core is the floor)"},
                "seeded_call": {"value": world * npts / (ms_e2e_seeded * 1e-3), "ms_per_step": ms_e2e_seeded,
                                "call": "sso_p1_contribute_seeded_buf, one chunk per call: key generation from the seed, proofs of "
                                        "knowledge (hash_to_g2), computation — all of phase1_cli::contribute but the file I/O"},
                "seeded_in_flight": {"value": world * npts / (ms_e2e_seeded_many * 1e-3), "ms_per_step": ms_e2e_seeded_many,
                                     "call": "sso_p1_contribute_seeded_many_buf: the full call with K chunks in flight, 6 host workers"},
                "file_call": file_call},
        "gpu_launches": launches,
        "roofline": {"bound": "imad",
                     "kernel": dom["kernel"], "achieved": dom["achieved_tmacs"], "peak": peak / 1e12, "unit": "TMAC/s",
                     "frac": dom["frac"], "traffic": ncu_dram_bytes_per_launch(args.curve)[0],
                     "peak_source": "measured live: mad.wide.u32 probe kernel (sso_imad_peak variant 0)",
                     "peak_carry_chain": peak_chain / 1e12, "frac_of_carry_chain_peak": (dom["frac"] * peak / peak_chain) if dom["frac"] else None,
                     "traffic_source": "%s (dram__bytes_read.sum + dram__bytes_write.sum, one launch)" % ncu_dram_bytes_per_launch(args.curve)[1],
                     "algorithmic_bytes": acc + contrib - 64 - sz["public_key_size"],
                     "macs_per_fq_mul": mac, "macs_per_fq_sqr": macs_per_fq_sqr(limbs), "kernels": kernels},
        "clocks": sampler.summary(),
        "points_per_step": npts,
        "verify": verify,
    }
    line["config"]["g2_body"] = "warp-cooperative (coop.cuh)" if coop_g2(args.curve) else "one thread per element"

    if not args.no_cpu_baseline:
        cb, _ = cpu_reference_run(args.curve, args.power, args.chunk_log, 1, 0, 12.0)
        line["cpu_baseline"] = cb
    if last_resp is not None:
        dump_outputs(args.dump_outputs, accumulator_vectors(last_resp, sz, es, True))
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
