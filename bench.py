#!/usr/bin/env python3
"""bench.py -- one PCD step's proving work (ECCyclePCD::prove, /root/reference/src/ec_cycle_pcd/mod.rs:92-181) on B200,
through libpcdgpu.so.

One "step" = what the SNARK backend sees for one PCD node, in the order the reference issues it: the default-circuit
proof on the helper curve (made while MainCircuit synthesises, data_structures.rs:135-143), the MAIN proof
(MNT4-298, mod.rs:171), the default-circuit proof on the main curve (HelpCircuit synthesis, data_structures.rs:343-350)
and the HELPER proof (MNT6-298, G2 over Fq3, mod.rs:179) -- four Groth16 proofs, strictly one after the other (the
helper circuit's witness contains the main proof).  Synthetic satisfiable R1CS of PCD-like size (SURVEY.md 8d): main
domain 2^18, helper 2^16, default circuits 2^10; keys with known trapdoors, resident on the GPU with window tables
(the default-circuit keys are the same on every call -- the reference builds them from a fixed-seed rng -- so a
resident-key cache serves them).  Constraint synthesis and the CRH (CPU work above the SNARK seam) are not part of it.
With N > 1 every GPU proves its own chain (independent PCD nodes: no data-path collective, weak scaling); the line
also carries the figures BASELINE.json names beside it: G1 MSM at 2^20 points (Mpts/s), the largest radix-2 NTT (GB/s),
a 2^20 Groth16 proof, GM17, a 64-node PCD tree, and -- N > 1 -- one MSM and one proof sharded over the GPUs through the
library's own NCCL exchange.  Every timed figure is first checked against the CPU oracle (outside the timed regions).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

`--dump-outputs DIR`: after the timed steps, the four proofs of the last one go to DIR/<proof>.npy (see dump_outputs).

`--impl reference`: the CPU arm.  The reference (Rust, un-vendored arkworks crates) cannot be built here, so this times
oracle/c (the C++ restatement of the same algorithms in the shape arkworks runs them: 5x64 CIOS, arkworks' Pippenger
with one task per window, per-stage parallel FFT) on all host threads, on the SAME four proofs at the SAME sizes.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODMUL_IMADS = 210            # 10-limb Montgomery product (SURVEY.md 8d)
MADD_MODMULS = {1: 10, 2: 28, 3: 58}  # XYZZ mixed add 8M + 2S in Fq / Fq2 (M=3,S=2) / Fq3 (M=6,S=5)
METRIC = "pcd_step_proofs_per_sec"
UNIT = "PCD steps/s"
PROF_NAMES = ["msm_digits_sort", "msm_accumulate_g1", "msm_accumulate_g2_fq2", "msm_reduce", "msm_horner", "ntt", "spmv_qap",
              "assemble", "msm_accumulate_g2_fq3", "msm_accumulate_small", "msm_accumulate_tail"]
PROF_TAIL = 10  # part fold + heavy-bucket kernels behind the accumulate kernel of a large MSM
PROF_ACC = {1: 1, 2: 2, 8: 3}  # accumulation classes of the large MSMs -> extension degree of the coordinates


def workload_config(args):
    """identical in both arms (the driver compares them)"""
    return {"workload": "pcd_step_groth16: default(mnt6,2^%d) -> main(mnt4,2^%d) -> default(mnt4,2^%d) -> helper(mnt6,2^%d)"
                        % (args.pcd_tiny_log_n, args.pcd_main_log_n, args.pcd_tiny_log_n, args.pcd_help_log_n),
            "proofs_per_step": 4,
            "main": {"pairing": "MNT4-298", "domain": "2^%d" % args.pcd_main_log_n},
            "helper": {"pairing": "MNT6-298", "domain": "2^%d" % args.pcd_help_log_n},
            "default_circuits": {"domain": "2^%d" % args.pcd_tiny_log_n, "pairings": ["MNT6-298", "MNT4-298"]}}


def step_plan(args):
    """(label, pairing, log_n) of the four proofs, in the reference's order"""
    return [("default_help", 1, args.pcd_tiny_log_n), ("main", 0, args.pcd_main_log_n),
            ("default_main", 0, args.pcd_tiny_log_n), ("helper", 1, args.pcd_help_log_n)]


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle():
    """the CPU oracle (test infrastructure): the checker of the gates and the thing timed by the CPU arms -- never part
    of a GPU-timed region"""
    for p in (os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import c_oracle as co
    return co


def limbs(v):
    return np.array([(v >> (64 * i)) & 0xFFFFFFFFFFFFFFFF for i in range(5)], dtype=np.uint64)


# ---------------------------------------------------------------------------------------------------
# CPU arm (oracle/c): the same four proofs at the same sizes
# ---------------------------------------------------------------------------------------------------
class NoGpu:
    """Key builder for the CPU arm.  The key's points are 4096 random group elements tiled over the queries: Pippenger's
    running time does not depend on which points it adds, and 5 x 2^18 distinct scalar multiplications on the CPU would
    take longer than the whole run.  Sizes, scalars, matrices and assignment are the real ones."""

    def __init__(self, co):
        self.co = co

    def fixed_base_mul(self, curve, g, k):
        k = np.ascontiguousarray(k, dtype=np.uint64).reshape(-1, 5)
        if k.shape[0] <= 4096:
            return self.co.fixed_base_mul(curve, g, k)
        base = self.co.fixed_base_mul(curve, g, k[:4096])
        reps = (k.shape[0] + 4095) // 4096
        return np.tile(base, (reps, 1))[:k.shape[0]].copy()


def cpu_step_setup(args, log=None):
    from pcd_b200 import synthetic
    co = oracle()
    insts = []
    for label, pairing, lg in step_plan(args):
        t0 = time.time()
        insts.append((label, synthetic.make_groth16_instance(NoGpu(co), pairing, lg, seed=77 + pairing + 10 * lg)))
        if log:
            log("CPU arm: %s instance (2^%d) built in %.1f s" % (label, lg, time.time() - t0))
    return co, insts


def cpu_step_once(co, insts, threads, rs):
    t0 = time.perf_counter()
    for (label, inst), (r, s) in zip(insts, rs):
        co.groth16_prove(inst["pairing"], inst["pk"], inst["A"], inst["B"], inst["C"], inst["m"], inst["num_inputs"],
                         inst["num_witness"], inst["z"], r, s, threads=threads)
    return time.perf_counter() - t0


def draw_rs(rng, p):
    v = lambda: limbs(int.from_bytes(rng.bytes(40), "little") % p)
    return v(), v()


def run_reference(args, rank, world):
    if rank != 0:
        return
    log = lambda m: print("[bench reference] %s" % m, file=sys.stderr, flush=True)
    co, insts = cpu_step_setup(args, log)
    threads = co.hw_threads()
    rng = np.random.Generator(np.random.Philox(99))
    draw = lambda: [draw_rs(rng, inst["p"]) for _, inst in insts]
    for _ in range(args.warmup):
        cpu_step_once(co, insts, threads, draw())
    t = 0.0
    for _ in range(args.steps):
        t += cpu_step_once(co, insts, threads, draw())
    value = args.steps / t
    cfg = workload_config(args)
    cfg["cpu_impl"] = "oracle/c (C++ restatement of arkworks' prover; the Rust reference cannot be built here)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (5x64-bit limbs)",
        "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d full PCD steps (4 proofs each, the stated sizes), oracle/c on all host threads; key "
                                   "points tiled from 4096 distinct ones" % args.steps},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
class PcdStep:
    """the four resident (key, matrices, assignment) sets of one PCD step and the calls that prove them in order"""

    def __init__(self, ctx, dev, args, seed_base=77, log=None):
        import torch

        import pcd_b200
        from pcd_b200 import synthetic
        self.ctx, self.parts = ctx, []
        for label, pairing, lg in step_plan(args):
            t0 = time.time()
            inst = synthetic.make_groth16_instance(ctx, pairing, lg, seed=seed_base + pairing + 10 * lg)
            g = pcd_b200.Groth16(ctx, pairing)
            win = os.environ.get("PCD_WINDOW_" + label.upper())  # development aid: table window of one proof's key
            if win:
                ctx.set_msm_window(int(win))
            idx = g.index(pcd_b200.ProvingKey(pairing=pairing, **inst["pk"]),
                          pcd_b200.ConstraintMatrices(pairing, inst["num_inputs"], inst["num_witness"], inst["A"],
                                                      inst["B"], inst["C"]), precompute=True)
            ctx.set_msm_window(0)
            z_host = torch.from_numpy(inst["z"].view(np.int64)).pin_memory()
            self.parts.append(dict(label=label, pairing=pairing, log_n=lg, inst=inst, g=g, idx=idx, z_host=z_host,
                                   z_dev=z_host.to(dev), nvars=inst["num_inputs"] + inst["num_witness"]))
            if log:
                log("%s: 2^%d on pairing %d resident (%.1f s)" % (label, lg, pairing, time.time() - t0))
        ctx.sync()

    def gate(self, co):
        """every proof of the step == its known discrete logarithms, the scalar multiplications done by the oracle"""
        from pcd_b200 import synthetic
        for k, part in enumerate(self.parts):
            p = part["inst"]["p"]
            r_i, s_i = (0x1234567 * 3 ** (70 + k)) % p, (0x7654321 * 5 ** (60 + k)) % p
            proof = part["g"].create_proof_dev(part["idx"], part["z_dev"].data_ptr(), limbs(r_i), limbs(s_i))
            expect = synthetic.expected_proof(self.ctx, part["inst"], r_i, s_i, mul=co.fixed_base_mul)
            if not np.array_equal(proof.affine_limbs(), expect):
                raise SystemExit("bench: the %s proof does not match its known discrete logarithms -- refusing to time it"
                                 % part["label"])

    def draw(self, rng):
        return [draw_rs(rng, part["inst"]["p"]) for part in self.parts]

    def step_dev(self, rs):
        """the step's four proofs, in proving order"""
        return [part["g"].create_proof_dev(part["idx"], part["z_dev"].data_ptr(), r, s)
                for part, (r, s) in zip(self.parts, rs)]

    def step_host(self, rs):
        c = self.ctx
        for part, (r, s) in zip(self.parts, rs):
            out = np.zeros(50, dtype=np.uint64)
            c._check(c.lib.pcdgpu_groth16_prove(c.h, part["idx"].pk, part["idx"].r1cs, part["z_host"].data_ptr(),
                                                r.ctypes.data, s.ctypes.data, out.ctypes.data))
        return out

    def h2d_bytes(self):
        return sum(part["nvars"] * 40 + 80 for part in self.parts)

    def d2h_bytes(self):
        return sum(320 if part["pairing"] == 0 else 400 for part in self.parts)

    def close(self):
        for part in self.parts:
            part["idx"].close()


def run_gpu(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    import pcd_b200

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctx = pcd_b200.Context(local_rank)
    stream = torch.cuda.Stream(device=dev, priority=-1)  # a real (non-default) stream shared by torch's events and the library
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    log = (lambda m: print("[bench rank %d] %s" % (rank, m), file=sys.stderr, flush=True)) if rank == 0 else None
    co = oracle()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # the integer roof: IMAD.WIDE.U32 issue rate of the fmaheavy pipe (32 lanes/clk/SM on B200), independent
    # accumulate form and carry-chain form (the same pipe, the same rate)
    imad_indep, _ = ctx.bench_imad(0, 4000)
    imad_chain, _ = ctx.bench_imad(3, 4000)
    imad_peak = max(imad_indep, imad_chain)

    # ---- workload: the four resident proofs of a PCD step, gated by the oracle ----------------------------
    step = PcdStep(ctx, dev, args, seed_base=77 + 1000 * rank, log=log)
    step.gate(co)
    if log:
        log("all four proofs of the step verified against their discrete logarithms (oracle scalar multiplications)")
    rng = np.random.Generator(np.random.Philox(7 + rank))
    rs = [step.draw(rng) for _ in range(args.warmup + 2 * args.steps + 2)]
    for i in range(args.warmup):
        step.step_dev(rs[i])

    # ---- timed region 1: assignments resident in HBM --------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    NC = len(PROF_NAMES)
    ms = (ctypes.c_double * NC)()
    units = (ctypes.c_double * NC)()
    spans = (ctypes.c_uint64 * NC)()
    launches = ctypes.c_uint64()
    ctx.lib.pcdgpu_profile_enable(ctx.h, 0)  # no event spans in the timed region; resets the launch counter
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        proofs = step.step_dev(rs[args.warmup + i])
    e1.record(stream)
    barrier()
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    ctx._check(ctx.lib.pcdgpu_profile_read(ctx.h, ms, units, spans, ctypes.byref(launches)))
    n_launches = int(launches.value)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step.parts, proofs)

    # ---- timed region 2: end to end through the C ABI with host buffers ---------------------------------------
    step.step_host(rs[0])  # untimed: grows the host path's staging scratch
    barrier()
    w0 = time.perf_counter()
    e0.record(stream)
    for i in range(args.steps):
        step.step_host(rs[args.warmup + args.steps + i])
    e1.record(stream)
    torch.cuda.synchronize()
    wall_ms = 1e3 * (time.perf_counter() - w0)
    barrier()
    ms_e2e = max_over_ranks(max(e0.elapsed_time(e1), wall_ms))
    clocks = sampler.stop()

    # ---- per-kernel pass: the MSM lanes serialised, CUDA-event spans per kernel class ------------------------
    ctx.set_concurrency(False)
    step.step_dev(rs[0])  # grows lane 0's scratch outside the spans
    ctx.lib.pcdgpu_profile_enable(ctx.h, 1)
    e0.record(stream)
    for i in range(args.steps):
        step.step_dev(rs[args.warmup + i])
    e1.record(stream)
    torch.cuda.synchronize()
    ms_serial = e0.elapsed_time(e1)
    launches2 = ctypes.c_uint64()
    ctx._check(ctx.lib.pcdgpu_profile_read(ctx.h, ms, units, spans, ctypes.byref(launches2)))
    prof = {"ms": list(ms), "units": list(units), "spans": list(spans)}
    # the same pass proof by proof: the step mixes MSMs of 2^18, 2^16 and 2^10 points in one kernel class, the roofline
    # is stated for the dominant kernel of the dominant proof
    prof_parts = {}
    for part, (r, s) in zip(step.parts, rs[1]):
        for _ in range(args.steps):
            part["g"].create_proof_dev(part["idx"], part["z_dev"].data_ptr(), r, s)
        ctx._check(ctx.lib.pcdgpu_profile_read(ctx.h, ms, units, spans, ctypes.byref(launches2)))
        prof_parts[part["label"]] = {"ms": list(ms), "units": list(units), "spans": list(spans)}
    ctx.lib.pcdgpu_profile_enable(ctx.h, 0)
    ctx.set_concurrency(True)
    # per-proof latencies of the step (device time of each of the four calls)
    per_proof = {}
    for part, (r, s) in zip(step.parts, rs[1]):
        for _ in range(2):
            part["g"].create_proof_dev(part["idx"], part["z_dev"].data_ptr(), r, s)
        e0.record(stream)
        for _ in range(3):
            part["g"].create_proof_dev(part["idx"], part["z_dev"].data_ptr(), r, s)
        e1.record(stream)
        torch.cuda.synchronize()
        per_proof[part["label"]] = {"pairing": "MNT4-298" if part["pairing"] == 0 else "MNT6-298",
                                    "domain": "2^%d" % part["log_n"], "ms": e0.elapsed_time(e1) / 3}

    extra = {"pcd_step_proofs": per_proof}
    if not args.no_tree:
        extra["pcd_tree"] = tree_figure(args, ctx, step, stream, rank, world, barrier, max_over_ranks, log)
    if world > 1 and not args.no_sharded:
        extra.update(sharded_figures(args, ctx, dev, stream, rank, world, co, log))
    h2d, d2h = step.h2d_bytes(), step.d2h_bytes()
    step.close()
    if not args.no_kernel_figures:
        extra.update(kernel_figures(args, ctx, dev, stream, imad_peak, co, rank, world, log))
    if rank == 0 and world == 1 and not args.no_proof20:
        extra["groth16_2^%d" % args.log_n] = proof_figure(args, ctx, dev, stream, co, log)
    if rank == 0 and world == 1 and not args.no_gm17:
        extra["gm17"] = gm17_figure(args, ctx, dev, stream, co, log)
    if rank == 0 and world == 1 and not args.no_marlin:
        extra["marlin"] = marlin_figure(args, ctx, co, log)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        _, cinsts = cpu_step_setup(args, log)
        threads = co.hw_threads()
        crng = np.random.Generator(np.random.Philox(5))
        cdraw = lambda: [draw_rs(crng, inst["p"]) for _, inst in cinsts]
        cpu_step_once(co, cinsts, threads, cdraw())
        reps, t = 0, 0.0
        while t < 12.0 and reps < 6:
            t += cpu_step_once(co, cinsts, threads, cdraw())
            reps += 1
        cpu_baseline = {"value": reps / t, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": "%d full PCD steps (4 proofs each at the stated sizes), oracle/c on all host threads; key "
                                  "points tiled from 4096 distinct ones" % reps}
    if rank != 0:
        return
    # ---- roofline of the dominant kernel class ----------------------------------------------------------------
    total_ms = sum(prof["ms"]) or 1.0
    shares = {PROF_NAMES[i]: round(prof["ms"][i] / total_ms, 4) for i in range(NC)}
    # the dominant kernel: bucket accumulation of the large MSMs, per coordinate field (the default-circuit proofs'
    # MSMs of ~10^3 points are a latency-bound regime of their own and are reported as their own class)
    dom_part, dom = max(((lbl, i) for lbl in prof_parts for i in PROF_ACC), key=lambda t: prof_parts[t[0]]["ms"][t[1]])
    pp = prof_parts[dom_part]
    deg = PROF_ACC[dom]
    imads = pp["units"][dom] * MADD_MODMULS[deg] * MODMUL_IMADS
    work = "bucket entries x %d Montgomery products (XYZZ mixed addition 8M + 2S over %s) x %d IMAD" % (
        MADD_MODMULS[deg], {1: "Fq", 2: "Fq2", 3: "Fq3"}[deg], MODMUL_IMADS)
    achieved = imads / (pp["ms"][dom] * 1e-3) / 1e12 if pp["ms"][dom] > 0 else 0.0
    step_frac = (prof["units"][dom] * MADD_MODMULS[deg] * MODMUL_IMADS / (prof["ms"][dom] * 1e-3) / imad_peak
                 if prof["ms"][dom] > 0 else None)
    by_proof = {lbl: {PROF_NAMES[i]: {"ms_per_proof": q["ms"][i] / args.steps,
                                      "frac": (q["units"][i] * MADD_MODMULS[PROF_ACC[i]] * MODMUL_IMADS / (q["ms"][i] * 1e-3)
                                               / imad_peak)}
                      for i in PROF_ACC if q["ms"][i] > 0} for lbl, q in prof_parts.items()}
    hbm_peak, hbm_src = load_peaks()
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            traffic = json.load(f).get(PROF_NAMES[dom], {}).get("bytes_per_launch")
    except Exception:
        pass
    others = {PROF_NAMES[i]: {"frac": (prof["units"][i] * MADD_MODMULS[PROF_ACC[i]] * MODMUL_IMADS / (prof["ms"][i] * 1e-3)
                                        / imad_peak) if prof["ms"][i] > 0 else None,
                               "ms_per_step": prof["ms"][i] / args.steps} for i in PROF_ACC if i != dom}
    roofline = {
        "kernel": PROF_NAMES[dom], "proof": dom_part, "bound": "imad", "achieved": achieved, "peak": imad_peak / 1e12,
        "unit": "TIMAD/s",
        "frac": achieved / (imad_peak / 1e12), "traffic": traffic,
        "traffic_note": "DRAM bytes per launch (read + write, averaged over the class's launches) from the committed ncu "
                        "capture of the same proof (profiles/r02_traffic.json); algorithmic: 80 / 160 / 240 B per gathered "
                        "point + 4 B per entry",
        "algorithmic_bytes_per_launch": pp["units"][dom] / max(pp["spans"][dom], 1) * ({1: 80, 2: 160, 3: 240}[deg] + 4),
        "peak_source": "measured live: IMAD.WIDE.U32 issue rate of the fmaheavy pipe (32 lanes/clk/SM), max of the "
                       "independent accumulate form (%.2f T/s) and the carry-chain form (%.2f T/s)" % (imad_indep / 1e12, imad_chain / 1e12),
        "launch_ms_avg": pp["ms"][dom] / max(pp["spans"][dom], 1), "work": work,
        "scope": "msm_accumulate_kernel launches of the %s proof's MSMs of this class (CUDA events around each launch, "
                 "lanes serialised; work = the entries the kernel itself walks, read back from the device); the same "
                 "kernel over the whole step (2^18 and 2^16-point MSMs mixed): frac %s.  What follows each launch -- part "
                 "fold + heavy-bucket kernels, latency-bound trees over the buckets of repeated witness values -- is "
                 "the msm_accumulate_tail class: %.3f ms per %s proof for %.0f entries (%.1f %% of the proof's entries)"
                 % (dom_part, "%.3f" % step_frac if step_frac is not None else "n/a",
                    pp["ms"][PROF_TAIL] / args.steps, dom_part, pp["units"][PROF_TAIL] / args.steps,
                    100.0 * pp["units"][PROF_TAIL] / max(1.0, pp["units"][PROF_TAIL] + sum(pp["units"][i] for i in PROF_ACC))),
        "accumulation_by_proof": by_proof,
        "other_accumulation_classes": others,
    }
    value = world * args.steps / (ms_dev * 1e-3)
    e2e_value = world * args.steps / (ms_e2e * 1e-3)
    cfg = workload_config(args)
    cfg.update({"per_gpu": "independent chain per GPU (PCD nodes), no collective", "precomputed_window_tables": True,
                "proofs_in_flight": 1,
                "l2": "per-step inputs (proving-key tables: several GB per key) exceed the 126 MB L2"})
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 (10x32-bit limbs, Montgomery, integer only)", "data": "synthetic",
        "config": cfg,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": n_launches,
        "clocks": clocks,
        "roofline": roofline,
        "kernel_time_shares": shares,
        "kernel_ms_per_step": {PROF_NAMES[i]: round(prof["ms"][i] / args.steps, 3) for i in range(NC)},
        "serialized_ms_per_step": ms_serial / args.steps,
        "kernel_timing_note": "kernel_* and roofline come from a second pass over the same steps with the MSM lanes "
                              "serialised (pcdgpu_set_concurrency(0)); value / ms_per_step are the overlapped run",
        "imad_peak_measured": {"independent_TIMAD_s": imad_indep / 1e12, "carry_chain_TIMAD_s": imad_chain / 1e12},
        "hbm_peak_GBps": {"value": hbm_peak, "source": hbm_src},
        "gates": "every timed figure was first compared with the CPU oracle (proofs: discrete logarithms by oracle scalar "
                 "multiplication; MSMs: the oracle's Pippenger on the same bytes; NTT: the transform's definition at 64 indices)",
    }
    line.update(extra)
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    emit(line)


def dump_outputs(out_dir, parts, proofs):
    """The proofs of the last timed step as out_dir/<proof label>.npy: the affine limbs (A, then B, then C; Montgomery
    coordinates, as create_proof_dev returns them), one row per u64 limb holding its low and high 32-bit halves as
    float64, which represents them exactly.  The inputs are seeded, so two builds can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    for part, proof in zip(parts, proofs):
        limbs = proof.affine_limbs().astype(np.uint64)
        halves = np.stack([limbs & np.uint64(0xFFFFFFFF), limbs >> np.uint64(32)], axis=1).astype(np.float64)
        np.save(os.path.join(out_dir, part["label"] + ".npy"), halves)


def tree_figure(args, ctx, step, stream, rank, world, barrier, max_over_ranks, log):
    """BASELINE config 5: a binary tree of PCD nodes, every node one full step (its four proofs), children before
    parents, nodes of a round spread round-robin over the GPUs, each node drawing from its own generator
    (pcd_b200/tree.py).  Wall time of the whole tree, max over ranks."""
    import torch

    from pcd_b200 import tree
    n = args.tree_nodes

    def prove_node(node, child_proofs, rng):
        rs = [(tree.draw_scalar(rng, part["inst"]["p"]), tree.draw_scalar(rng, part["inst"]["p"])) for part in step.parts]
        return step.step_dev(rs)[-1].affine_limbs().tobytes()

    tree.prove_tree(min(n, 3), prove_node, rank, world)  # warm-up (and the collective's first call)
    barrier()
    t0 = time.perf_counter()
    proofs = tree.prove_tree(n, prove_node, rank, world)
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0)
    # determinism gate: node 1's helper proof re-proved alone with the node's generator
    again = prove_node(1, [], tree.node_rng(20261017, 1))
    return {"nodes": n, "gpus": world, "wall_ms": dt * 1e3, "nodes_per_s": n / dt, "rounds": len(tree.rounds(n)),
            "root_proof_reproducible": bool(again == proofs[1]),
            "note": "every node = one PCD step (4 proofs); host hands the children's proofs up (all_gather_object per "
                    "round); one node in flight per GPU"}


def sharded_figures(args, ctx, dev, stream, rank, world, co, log):
    """N > 1: one G1 MSM (2^20) and one main-size proof sharded over the GPUs by point range, the partial sums exchanged
    by the library's own NCCL all-gather (pcdgpu_msm_bases_sharded_dev, pcdgpu_groth16_prove_sharded_dev) -- no Python
    and no host on the data path.  Times are max over ranks; results are compared with the single-GPU ones."""
    import torch
    import torch.distributed as dist

    import pcd_b200
    from pcd_b200 import sharding, synthetic
    out = {}
    ctx.comm_init_torch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, reps):
        for _ in range(3):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = 1 << args.msm_log_n
    pts = synthetic.random_points_dev(ctx, 0, n, seed=3).cpu().numpy().view(np.uint64)  # the same points on every rank
    sc_host = synthetic.random_limbs(n, 0, 9)
    lo, hi = sharding.shard_range(n, world, rank)
    shard = pcd_b200.Bases(ctx, 0, pts[lo:hi], precompute=True)
    sc = torch.from_numpy(sc_host[lo:hi].copy().view(np.int64)).to(dev)
    res = torch.zeros(16, dtype=torch.int64, device=dev)
    ms_sh = timed(lambda: shard.msm_sharded_dev(sc.data_ptr(), hi - lo, res.data_ptr()), 10)
    got = res.cpu().numpy().view(np.uint64)[:10].copy()
    shard.close()
    ok = True
    ms_one = None
    if rank == 0:
        ok = bool(np.array_equal(got, co.msm(0, pts, sc_host, threads=co.hw_threads())))
        full = pcd_b200.Bases(ctx, 0, pts, precompute=True)
        scf = torch.from_numpy(sc_host.view(np.int64)).to(dev)
        for _ in range(3):
            full.msm_dev(scf.data_ptr(), n, res.data_ptr())
        e0.record(stream)
        for _ in range(10):
            full.msm_dev(scf.data_ptr(), n, res.data_ptr())
        e1.record(stream)
        torch.cuda.synchronize()
        ms_one = e0.elapsed_time(e1) / 10
        full.close()
    dist.barrier()
    out["g1_msm_sharded"] = {"points": n, "gpus": world, "ms": ms_sh, "mpts_per_s": n / ms_sh / 1e3,
                             "ms_one_gpu": ms_one, "speedup": (ms_one / ms_sh) if ms_one else None,
                             "matches_oracle": ok, "collective": "ncclAllGather of one 160-byte xyzz partial per rank, "
                             "inside libpcdgpu.so"}
    # one proof over all GPUs
    lg = args.pcd_main_log_n
    inst = synthetic.make_groth16_instance(ctx, 0, lg, seed=55)  # the same instance on every rank
    pk = pcd_b200.ProvingKey(pairing=0, **inst["pk"])
    cm = pcd_b200.ConstraintMatrices(0, inst["num_inputs"], inst["num_witness"], inst["A"], inst["B"], inst["C"])
    sh = sharding.ShardedGroth16(ctx, pk, cm, rank, world, dev)
    z = torch.from_numpy(inst["z"].view(np.int64)).to(dev)
    p = inst["p"]
    r, s = pow(3, 111, p), pow(7, 99, p)
    ms_p = timed(lambda: sh.prove(z, r, s), 5)
    proof = sh.prove(z, r, s)
    sh.close()
    ok_p = bool(np.array_equal(proof, synthetic.expected_proof(ctx, inst, r, s, mul=co.fixed_base_mul)))
    out["groth16_sharded"] = {"pairing": "MNT4-298", "domain": "2^%d" % lg, "gpus": world, "ms": ms_p,
                              "matches_trapdoor": ok_p,
                              "collective": "two ncclAllGather exchanges of xyzz partial sums per proof, inside libpcdgpu.so"}
    return out


def proof_figure(args, ctx, dev, stream, co, log):
    """BASELINE configs[1]: one Groth16 proof on MNT4-298 at the largest benchmarked radix-2 domain (2^20)."""
    import torch

    import pcd_b200
    from pcd_b200 import synthetic
    log_n = args.log_n
    inst = synthetic.make_groth16_instance(ctx, pcd_b200.MNT4_298, log_n, seed=20261017, verbose=log)
    g = pcd_b200.Groth16(ctx, pcd_b200.MNT4_298)
    idx = g.index(pcd_b200.ProvingKey(pairing=0, **inst["pk"]),
                  pcd_b200.ConstraintMatrices(0, inst["num_inputs"], inst["num_witness"], inst["A"], inst["B"], inst["C"]),
                  precompute=True)
    z = torch.from_numpy(inst["z"].view(np.int64)).to(dev)
    p = inst["p"]
    r_i, s_i = 0x1234567 * 3 ** 70 % p, 0x7654321 * 5 ** 60 % p
    proof = g.create_proof_dev(idx, z.data_ptr(), limbs(r_i), limbs(s_i))
    if not np.array_equal(proof.affine_limbs(), synthetic.expected_proof(ctx, inst, r_i, s_i, mul=co.fixed_base_mul)):
        raise SystemExit("bench: the 2^%d proof does not match its discrete logarithms" % log_n)
    for _ in range(3):
        g.create_proof_dev(idx, z.data_ptr(), limbs(r_i), limbs(s_i))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(5):
        g.create_proof_dev(idx, z.data_ptr(), limbs(r_i), limbs(s_i))
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    idx.close()
    return {"pairing": "MNT4-298", "domain": "2^%d" % log_n, "ms_per_proof": ms, "proofs_per_s": 1e3 / ms,
            "proofs_in_flight": 1, "note": "one proof at a time on resident window tables"}


def gm17_figure(args, ctx, dev, stream, co, log):
    """GM17 proofs/s on MNT4-298 (the second SNARK the reference plugs into ECCyclePCD, tests/mnt4_gm17.rs:27-28):
    2^(k-1) - 2 constraints, SAP domain 2^k; the proof is checked against GM17's verification equations in the
    exponent (known trapdoor, oracle scalar multiplications) before it is timed."""
    import torch

    import pcd_b200
    from pcd_b200 import synthetic
    k = args.gm17_log_n
    m = (1 << (k - 1)) - 2
    inst = synthetic.make_gm17_instance(ctx, pcd_b200.MNT4_298, m, seed=4242, verbose=log)
    assert inst["domain_size"] == 1 << k
    g = pcd_b200.GM17(ctx, pcd_b200.MNT4_298)
    idx = g.index(pcd_b200.GM17ProvingKey(pairing=0, **inst["pk"]),
                  pcd_b200.ConstraintMatrices(0, inst["num_inputs"], inst["num_witness"], inst["A"], inst["B"], inst["C"]),
                  precompute=True)
    z = torch.from_numpy(inst["z"].view(np.int64)).to(dev)
    p = inst["p"]
    d1, d2, r = 0x1234567 * 3 ** 70 % p, 0x7654321 * 5 ** 60 % p, 0xabcdef1 * 7 ** 50 % p
    proof = g.create_proof_dev(idx, z.data_ptr(), limbs(d1), limbs(d2), limbs(r))
    if not np.array_equal(proof.affine_limbs(), synthetic.expected_gm17_proof(ctx, inst, d1, d2, r, mul=co.fixed_base_mul)):
        raise SystemExit("bench: GM17 proof does not satisfy the verification equations in the exponent")
    for _ in range(3):
        g.create_proof_dev(idx, z.data_ptr(), limbs(d1), limbs(d2), limbs(r))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    reps = 5
    e0.record(stream)
    for _ in range(reps):
        g.create_proof_dev(idx, z.data_ptr(), limbs(d1), limbs(d2), limbs(r))
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    idx.close()
    return {"proofs_per_s": 1e3 / ms, "ms_per_proof": ms, "pairing": "MNT4-298", "constraints": m,
            "sap_domain": "2^%d" % k, "note": "SAP witness map (5 NTTs) + 4 G1 MSMs + 1 G2 MSM + assembly; one proof at a time"}


def marlin_figure(args, ctx, co, log):
    """Marlin proofs/s on MNT4-298 (BASELINE config 4; /root/reference/tests/mnt4_marlin.rs:72-75): synthetic R1CS with
    |H| = 2^k, KZG10 SRS with a known trapdoor built on the GPU.  The proof is checked before it is timed: every
    commitment against [p(beta) + gamma r(beta)] G by the oracle's scalar multiplication, the AHP verifier's sumcheck
    identities, and KZG10's equation in the exponent (tests/marlin_check.py).  Timed with the wall clock around the
    whole prover call: it hands commitments back to the host between rounds (the transcript lives there), so a proof is
    not one stream-ordered region."""
    import random
    import time

    import pcd_b200
    from pcd_b200 import kzg, marlin, synthetic
    import marlin_check
    pairing, field = pcd_b200.MNT4_298, 0
    p = synthetic.FIELD_P[field]
    m = (1 << args.marlin_log_h) - 4
    z, ra, rb, rc = synthetic._synthetic_rows(random.Random(99), p, m, 0.4)
    cm = pcd_b200.ConstraintMatrices(pairing, 2, len(z) - 2, synthetic._csr(ra, p), synthetic._csr(rb, p),
                                     synthetic._csr(rc, p))
    nnz = max(len(c[1]) for c in (cm.a, cm.b, cm.c))
    h, k = 1 << (len(z) - 1).bit_length(), 1 << (nnz - 1).bit_length()
    max_degree = max(3 * h, 4 * k)
    beta, gamma = pow(3, 4004, p), pow(5, 3003, p)
    pw = [1] * (max_degree + 2)
    for i in range(1, max_degree + 2):
        pw[i] = pw[i - 1] * beta % p
    G = synthetic.generator(0)
    pg = ctx.fixed_base_mul(0, G, synthetic._limbs_from_ints(pw[:max_degree + 1]))
    pgg = ctx.fixed_base_mul(0, G, synthetic._limbs_from_ints([gamma * x % p for x in pw]))
    powers = kzg.Powers(ctx, pairing, pg, pgg, precompute=True)
    snark = marlin.MarlinSNARK(ctx, pairing)
    t0 = time.perf_counter()
    ipk = snark.index(cm, powers, max_degree)
    ctx.sync()
    index_s = time.perf_counter() - t0
    R = (1 << 320) % p
    zl = synthetic._limbs_from_ints([v * R % p for v in z])
    blind = synthetic.random_limbs(4 * h + 64, field, 31337)

    class BulkRng:  # the caller's rng: consecutive draws from one precomputed stream, handed out in bulk
        def __init__(self):
            self.pos = 0

        def many(self, f, n):
            self.pos += n
            return blind[self.pos - n:self.pos]

        def __call__(self, f):
            return self.many(f, 1)[0]

    make_rng = BulkRng
    proof = snark.prove(ipk, zl, make_rng())
    marlin_check.check_in_exponent(snark, ipk, proof, beta, gamma, G)
    if log:
        log("Marlin proof (|H| = %d, |K| = %d, SRS %d) checked in the exponent" % (h, k, max_degree + 1))
    snark.prove(ipk, zl, make_rng())
    ctx.sync()
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        snark.prove(ipk, zl, make_rng())
    ctx.sync()
    ms = (time.perf_counter() - t0) / reps * 1e3
    ipk.close()
    powers.close()
    return {"proofs_per_s": 1e3 / ms, "ms_per_proof": ms, "pairing": "MNT4-298", "constraints": m, "H": h, "K": k,
            "srs_points": max_degree + 1, "index_s": index_s, "timing": "host wall clock around MarlinSNARK.prove",
            "note": "AHP rounds on device vectors (FFTs over H, K, 4K; CSR products; batch inversions), 9 KZG10 "
                    "commitments + 2 batched openings as MSMs over the resident SRS; host: Poseidon transcript only"}


def kernel_figures(args, ctx, dev, stream, imad_peak, co, rank=0, world=1, log=None):
    """G1 MSM Mpts/s at 2^20 (uniform scalars; resident bases with and without the window tables), the other sizes
    BASELINE.json names, and the largest radix-2 NTT (coset FFT over r4), each compared with the oracle once and then
    timed with CUDA events on the launching stream."""
    import torch

    import pcd_b200
    from pcd_b200 import synthetic
    out = {}
    if rank != 0:
        return out
    hbm_peak, _ = load_peaks()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    threads = co.hw_threads()

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    res = torch.zeros(64, dtype=torch.int64, device=dev)

    def msm_case(lg, seed, plain_too):
        n = 1 << lg
        pts = synthetic.random_points_dev(ctx, pcd_b200.MNT4_G1, n, seed=seed)
        pts_host = pts.cpu().numpy().view(np.uint64)
        sc_host = synthetic.random_limbs(n, 0, seed + 6)
        sc = torch.from_numpy(sc_host.view(np.int64)).to(dev)
        ref = co.msm(0, pts_host, sc_host, threads=threads)
        bases = pcd_b200.Bases(ctx, 0, pts_host, precompute=True)
        if not np.array_equal(bases.msm(sc_host), ref):
            raise SystemExit("bench: G1 MSM at 2^%d (window tables) differs from the oracle" % lg)
        r = {"ms": timed(lambda: bases.msm_dev(sc.data_ptr(), n, res.data_ptr()), 5)}
        r["mpts_per_s"] = n / r["ms"] / 1e3
        bases.close()
        if plain_too:
            if not np.array_equal(ctx.msm(0, pts_host, sc_host), ref):
                raise SystemExit("bench: variable-base G1 MSM at 2^%d differs from the oracle" % lg)
            r["variable_base_ms"] = timed(lambda: ctx.msm_dev(0, pts.data_ptr(), sc.data_ptr(), n, res.data_ptr()), 5)
            r["variable_base_mpts_per_s"] = n / r["variable_base_ms"] / 1e3
        return r

    r20 = msm_case(args.msm_log_n, 3, True)
    out["g1_msm"] = {"points": 1 << args.msm_log_n, "scalars": "uniform 298-bit", "mpts_per_s": r20["mpts_per_s"],
                     "ms": r20["ms"], "mode": "resident bases with precomputed window tables",
                     "variable_base_mpts_per_s": r20["variable_base_mpts_per_s"], "variable_base_ms": r20["variable_base_ms"],
                     "checked_against_oracle": True}
    if world == 1 and not args.no_sweep:
        sweep = {}
        for lg in (16, 18, 22):
            if lg != args.msm_log_n:
                sweep["2^%d" % lg] = msm_case(lg, 30 + lg, False)
        out["g1_msm_sweep"] = sweep
    log_n = args.ntt_log_n
    x_host = synthetic.random_limbs(1 << min(log_n, 20), 0, 5)
    if log_n > 20:
        x_host = np.tile(x_host, (1 << (log_n - 20), 1))
        x_host[::4097, 0] ^= np.uint64(0x5A5A)  # not periodic
    x = torch.from_numpy(x_host.view(np.int64)).to(dev)
    y = x.clone()
    ctx.ntt_dev(0, y.data_ptr(), log_n, False, True)
    ctx.sync()
    rng = np.random.Generator(np.random.Philox(5))
    idx = np.concatenate([[0, 1, (1 << log_n) - 1], rng.integers(0, 1 << log_n, 61)]).astype(np.uint64)
    got = y[torch.from_numpy(idx.astype(np.int64)).to(dev)].cpu().numpy().view(np.uint64)
    if not np.array_equal(got, co.dft_at(0, x_host, idx, coset=True)):
        raise SystemExit("bench: the 2^%d coset FFT differs from the transform's definition" % log_n)
    del y
    ms_ntt = timed(lambda: ctx.ntt_dev(0, x.data_ptr(), log_n, False, True), 5)
    gbs = 2 * 40 * (1 << log_n) / (ms_ntt * 1e-3) / 1e9
    butterflies = (1 << (log_n - 1)) * log_n
    timad = butterflies * MODMUL_IMADS / (ms_ntt * 1e-3) / 1e12
    out["ntt"] = {"log_n": log_n, "field": "r4 (MNT4-298 Fr)", "flavour": "coset_fft", "ms": ms_ntt, "GBps": gbs,
                  "checked_against_definition": True}
    if world == 1 and not args.no_sweep:
        nsw = {}
        for lg in (16, 20):
            if lg >= log_n:
                continue
            xs = torch.from_numpy(x_host[:1 << lg].copy().view(np.int64)).to(dev)  # x itself was transformed in place above
            ref = co.ntt(0, x_host[:1 << lg], False, True, threads=threads)
            ys = xs.clone()
            ctx.ntt_dev(0, ys.data_ptr(), lg, False, True)
            if not np.array_equal(ys.cpu().numpy().view(np.uint64), ref):
                raise SystemExit("bench: the 2^%d coset FFT differs from the oracle" % lg)
            t_ = timed(lambda: ctx.ntt_dev(0, xs.data_ptr(), lg, False, True), 10)
            nsw["2^%d" % lg] = {"ms": t_, "GBps": 2 * 40 * (1 << lg) / (t_ * 1e-3) / 1e9}
        yq = torch.from_numpy(synthetic.random_limbs(1 << 17, 1, 6).view(np.int64)).to(dev)
        t_ = timed(lambda: ctx.ntt_dev(1, yq.data_ptr(), 17, False, True), 10)  # the helper field's largest radix-2 domain
        nsw["q4_2^17"] = {"ms": t_, "GBps": 2 * 40 * (1 << 17) / (t_ * 1e-3) / 1e9, "note": "L2-resident, not an HBM figure"}
        out["ntt_sweep"] = nsw
    out["roofline_ntt"] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                           "traffic": None, "imad_frac": timad / (imad_peak / 1e12),
                           "note": "algorithmic bytes 2*N*40; a 298-bit NTT is bound by the integer pipe: imad_frac = "
                                   "(N/2 log2 N butterflies x 210 IMAD) / time / the IMAD.WIDE roof"}
    return out


_REAL_STDOUT = None


def emit(line: dict):
    """the ONE JSON line, on the process's real stdout (fd 1 is pointed at stderr while the job runs so that
    library chatter -- NCCL prints its version banner on stdout -- cannot end up next to it)"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pcd-main-log-n", type=int, default=18)
    ap.add_argument("--pcd-help-log-n", type=int, default=16)
    ap.add_argument("--pcd-tiny-log-n", type=int, default=10)
    ap.add_argument("--log-n", type=int, default=int(os.environ.get("PCD_BENCH_LOG_N", "20")),
                    help="domain of the extra single-proof figure (BASELINE configs[1])")
    ap.add_argument("--msm-log-n", type=int, default=20)
    ap.add_argument("--ntt-log-n", type=int, default=24)
    ap.add_argument("--tree-nodes", type=int, default=64)
    ap.add_argument("--gm17-log-n", type=int, default=18, help="SAP domain of the GM17 figure (2^k)")
    ap.add_argument("--no-gm17", action="store_true", help="skip the GM17 figure")
    ap.add_argument("--no-marlin", action="store_true", help="skip the Marlin figure")
    ap.add_argument("--marlin-log-h", type=int, default=15, help="|H| of the Marlin figure (2^k)")
    ap.add_argument("--no-proof20", action="store_true", help="skip the 2^20 single-proof figure")
    ap.add_argument("--no-tree", action="store_true")
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-figures", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the MSM / NTT size sweeps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the four proofs of the last timed step to DIR/<proof>.npy (rank 0; GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU arm's proofs")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_gpu(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
