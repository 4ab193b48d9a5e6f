#!/usr/bin/env python
"""bench.py — headline benchmark of spartan_b200 (driver contract: see the task statement).

metric   : R1CS constraints proved per second, SNARK::prove on Instance::produce_synthetic_r1cs (BASELINE.json `metric`)
workload : BASELINE.json configs[1] — 2^20 constraints, 2^20 variables, 10 inputs, 2^20 non-zeros per matrix, one B200
step     : one SNARK::prove (transcript creation + prove; gens, instance synthesis and SNARK::encode excluded, exactly what
           /root/reference/benches/snark.rs:55-68 times)
value    : inputs (the assignment) resident in HBM when the clock starts;   e2e: assignment in pinned HOST memory, copied to the device
           inside the timed region, proof bytes copied back to the host
N > 1    : one process per GPU (torchrun); every rank proves its own instance of the same size (independent proofs: no data-path
           collective), value = N * constraints / max-over-ranks time          -> "scaling": "weak"
           The same line carries `strong`: ONE proof sharded over the N GPUs (tables / commitment rows / product circuits partitioned,
           per-round partial sums exchanged over NVLink inside the kernels; spartan_b200/csrc/comm.cu), its latency and that its bytes equal
           the single-GPU proof's; and BASELINE.json configs[2]/[3] at N GPUs: `msm_var_2p24` (2^24-point MSM, point-add all-reduce) and
           `dense_sumcheck_2p22` (per-round fold GB/s of a 2^22-entry cubic sumcheck, scalar-add all-reduce).
--impl reference : the CPU restatement of the reference (oracle/, C loops under OpenMP on all host cores) on a bounded sample of the
           same workload (SNARK::prove at 2^SAMPLE_LOG constraints); rank 0 only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the CPU arm's OpenMP loops are short: spinning worker threads on every logical CPU slow it down 10x on the 2 x 32-core / 128-thread host
os.environ.setdefault("OMP_WAIT_POLICY", "passive")


def host_threads():
    """threads for the CPU arm: one per physical core (the oracle's loops do not profit from SMT siblings)"""
    n = os.cpu_count() or 1
    return max(1, n // 2) if n >= 4 else n

METRIC = "R1CS constraints/sec (SNARK::prove, synthetic R1CS)"
UNIT = "constraints/s"
LOG_N = int(os.environ.get("SP_BENCH_LOGN", "20"))
NUM_INPUTS = 10
CPU_SAMPLE_LOG = int(os.environ.get("SP_BENCH_CPU_LOGN", str(LOG_N)))   # the CPU arm proves the SAME configuration as the GPU arm
SHARDED_LEGS_DEFAULT = "1"   # the sharded prover passed its multi-GPU parity runs (tools/run_sharded.py; profiles/r02_sharded.md)
# world sizes at which the sharded prover has been byte-validated on hardware (profiles/r02_sharded.md).  At any other N the sharded legs stay off
# unless SP_BENCH_SHARDED=1 forces them: an unvalidated collective that stalls would take the whole bench line (the replica throughput) down with it.
SHARDED_VALIDATED_WORLDS = (2, 4, 8)
CPU_ARM_BUDGET_S = float(os.environ.get("SP_BENCH_CPU_BUDGET_S", "1200"))


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region"""

    def __init__(self, gpu_index):
        self.lines = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def _oracle_setup(n):
    from oracle.spartan_ref import core as oc, r1cs, spark
    cores = host_threads()
    oc.lib.oracle_set_threads(cores)
    inst, vars_arr, inputs = r1cs.Instance.produce_synthetic_r1cs(n, n, NUM_INPUTS, 0)
    gens = spark.SNARKGens(n, n, NUM_INPUTS, n)
    comm, decomm = spark.SNARK.encode(inst, gens)

    def step():
        return spark.SNARK.prove(inst, comm, decomm, vars_arr.copy(), inputs, gens, oc.Transcript(b"example"), r1cs.tape_seed(0))
    return step, cores


def run_reference(args):
    """CPU arm: the oracle's SNARK::prove (restatement of the reference; the Rust crate cannot be built here) on all host cores, on the SAME
    configuration as the GPU arm (2^LOG_N constraints / variables / non-zeros, same instance seed, tape seed and transcript label): one step =
    one whole proof.  A step takes tens of seconds, so at most one warm-up step is run and the timed loop stops early (reporting the steps it
    actually timed) if it would exceed CPU_ARM_BUDGET_S."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    n = 1 << CPU_SAMPLE_LOG
    step, cores = _oracle_setup(n)
    warm = min(args.warmup, 1)
    for _ in range(warm):
        step()
    t0 = time.perf_counter()
    done = 0
    while done < args.steps:
        step()
        done += 1
        el = time.perf_counter() - t0
        if done < args.steps and el / done * (done + 1) > CPU_ARM_BUDGET_S:
            break
    dt = (time.perf_counter() - t0) / done
    value = n / dt
    sample = ("SNARK::prove at 2^%d constraints/variables/non-zeros = the GPU arm's configuration, whole proof per step; oracle (C loops under OpenMP, Python "
              "protocol layer < 3%% of the time at this size); %d of %d requested steps timed (%.1f s each), %d warm-up" % (CPU_SAMPLE_LOG, done, args.steps, dt, warm))
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": done, "warmup": warm,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (4x64-bit Montgomery limbs)", "data": "synthetic",
        "config": {"workload": "SNARK::prove synthetic R1CS 2^%d cons/vars, 2^%d non-zero, %d inputs (BASELINE.json configs[1])" % (CPU_SAMPLE_LOG, CPU_SAMPLE_LOG, NUM_INPUTS),
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def cpu_baseline_leg():
    """one whole oracle proof of the same configuration on the box's host cores, reported beside the GPU number (rank 0, N = 1 only)"""
    n = 1 << CPU_SAMPLE_LOG
    step, cores = _oracle_setup(n)
    t0 = time.perf_counter()
    step()
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "one SNARK::prove at 2^%d = the GPU arm's configuration (oracle = CPU restatement of the reference, OpenMP over its C loops; %.1f s)" % (CPU_SAMPLE_LOG, dt)}


def msm_var_leg(sb, api, sd, ctx, rank, world, logn=24):
    """BASELINE.json configs[2]: standalone variable-base MSM, N = 2^24 ristretto255 points (MultiCommitGens::new(N, b"msm-bench").G, no
    precomputed tables), uniformly random scalars below q; bucket method of spartan_b200/csrc/kernels_pip.cu.  On W > 1 GPUs the vector is
    split by index range, every rank runs the bucket MSM on its slice and the partial sums meet in a point-add all-reduce (sp_msm_var_sharded)."""
    import numpy as np
    import torch
    n = 1 << logn
    P = api.Points.derive(n, b"msm-bench", ctx=ctx)
    rng = np.random.default_rng(0)
    t = rng.integers(0, 2 ** 63, size=(n, 4), dtype=np.uint64)
    t[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)          # < 2^252 < q: valid Montgomery residues, i.e. uniformly random field elements
    per = n // world
    S = sb.DensePolynomial(t[rank * per:(rank + 1) * per], ctx=ctx)
    del t
    run = (lambda: P.msm_sharded(S, offset=rank * per)) if world > 1 else (lambda: P.msm(S))
    out = run()
    ts = []
    for _ in range(3):
        sd.barrier(); torch.cuda.synchronize()
        api.timer_start(ctx)
        out2 = run()
        ts.append(api.timer_stop_ms(ctx))
        assert out == out2
    ms = sd.max_over_ranks([min(ts)])[0]
    golden = None
    try:   # the oracle's result for exactly these inputs (tests/golden/msm_2p24.json, made on the CPU by tests/golden/make_msm_golden.py)
        with open(os.path.join(ROOT, "tests", "golden", "msm_2p%d.json" % logn)) as f:
            golden = json.load(f)["encoding"] == out.hex()
    except Exception:
        pass
    return {"points": n, "n_gpus": world, "ms": ms, "result_equals_oracle_golden": golden, "Mpoint_adds_per_s_reference_equivalent": 33.0 * n / (ms / 1e3) / 1e6, "Mpoints_per_s": n / (ms / 1e3) / 1e6,
            "what": "2^%d caller-supplied points, 253-bit scalars, scalars and points resident in HBM, %s; 33 adds/point = dalek Pippenger w=8 (SURVEY.md 8d)"
                    % (logn, "split by index range over %d GPUs + point-add all-reduce over NVLink (sp_msm_var_sharded)" % world if world > 1 else "sp_msm_var_resident"),
            "result_prefix": out.hex()[:16]}


def dense_sumcheck_leg(sb, api, sd, ctx, rank, world, pk, logn=22, rounds=5):
    """BASELINE.json configs[3]: cubic-with-additive-term sumcheck (A*(B*C-D), sumcheck.rs:625-652 + dense_mlpoly.rs:215-223) on four 2^22-entry
    tables, rounds timed one by one: round 0 is the plain evaluation (32 B x len per table), rounds 1.. the fused bind + evaluate (48 B x len per
    table, len = the table length before the bind).  On W > 1 GPUs every rank holds the cyclic shard of each table and the kernels exchange
    their partial sums over NVLink (sp_sumcheck_*_sharded); GB/s is whole-job algorithmic bytes / max-over-ranks time."""
    import numpy as np
    import torch
    n = 1 << logn
    rng = np.random.default_rng(1)
    polys = []
    for _ in range(4):
        t = rng.integers(0, 2 ** 63, size=(n, 4), dtype=np.uint64)
        t[:, 3] &= np.uint64(0x0FFFFFFFFFFFFFFF)
        polys.append(sb.DensePolynomial(t[rank::world] if world > 1 else t, ctx=ctx))
        del t
    r = sb.prg_scalars("r", rounds + 1)
    ev = (lambda: api.sumcheck_eval_sharded(2, polys)) if world > 1 else (lambda: api.sumcheck_eval(2, polys))
    fe = (lambda rr: api.sumcheck_fold_eval_sharded(2, polys, rr)) if world > 1 else (lambda rr: api.sumcheck_fold_eval(2, polys, rr))
    ev()
    out = []
    length = n
    for j in range(rounds + 1):
        sd.barrier(); torch.cuda.synchronize()
        api.timer_start(ctx)
        e = ev() if j == 0 else fe(r[j])
        ms = sd.max_over_ranks([api.timer_stop_ms(ctx)])[0]
        by = 4 * (32.0 if j == 0 else 48.0) * length
        out.append({"round": j, "table_len": length, "us": ms * 1e3, "GBs": by / 1e9 / (ms / 1e3), "frac_of_hbm": by / 1e9 / (ms / 1e3) / (pk["hbm_gbs"] * world)})
        if j > 0:
            length //= 2
    return {"tables": 4, "log_len": logn, "n_gpus": world, "rounds": out, "evals_prefix": bytes(e.tobytes()[:8]).hex(),
            "note": "time = kernel + the device->host copy of the three evaluations (and, sharded, the NVLink exchange of 96 B per rank inside the kernel); frac_of_hbm against N x the measured copy bandwidth"}


def dump_outputs(out_dir, proofs):
    """The proofs the last timed step of each timed region returned, one float32 value per byte (0..255, exact), as <out_dir>/<name>.npy.
    The instance, assignment, generators, transcript label and random tape are all seeded, so two builds run with the same arguments
    can be compared output for output.  Rank 0's proofs only; at 2^20 each array holds 180,840 values (~720 KB)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, b in proofs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.frombuffer(b, dtype=np.uint8).astype(np.float32))


def run_b200(args):
    import numpy as np
    import torch
    from spartan_b200 import dist as sd
    rank, world, local = sd.init("nccl" if int(os.environ.get("WORLD_SIZE", "1")) > 1 else None)
    import spartan_b200 as sb
    from spartan_b200 import api
    ctx = sb.Context(local if world > 1 else 0)
    # the intra-proof (strong-scaling) legs need the sharded prover; SP_BENCH_SHARDED=0 leaves them out (replica throughput only)
    sharded_env = os.environ.get("SP_BENCH_SHARDED")
    sharded_legs = world > 1 and (sharded_env == "1" or (sharded_env is None and SHARDED_LEGS_DEFAULT != "0" and world in SHARDED_VALIDATED_WORLDS))
    if sharded_legs:
        sd.connect(ctx)            # IPC windows over NVLink; sharded proving is switched on only for the `strong` leg below
        ctx.set_sharding(False)
    n = 1 << LOG_N
    # every rank proves its own instance (seed = rank): independent proofs, no data-path collective
    inst, vars_, inputs = sb.Instance.produce_synthetic_r1cs(n, n, NUM_INPUTS, seed=sd.rank_seed(rank), ctx=ctx)
    gens = sb.SNARKGens(n, n, NUM_INPUTS, n, ctx=ctx)
    comm = sb.SNARK.encode(inst, gens)
    d_vars = sb.DensePolynomial(vars_.limbs, ctx=ctx)
    pinned = torch.empty((n, 4), dtype=torch.int64).pin_memory()
    pinned.numpy().view(np.uint64)[:] = vars_.limbs
    host_vars = sb.Assignment.__new__(sb.Assignment)
    host_vars.limbs = pinned.numpy().view(np.uint64)
    seed = sb.tape_seed(sd.rank_seed(rank))
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda:%d" % (local if world > 1 else 0))  # > L2 (126 MB)

    def barrier():
        sd.barrier()
        torch.cuda.synchronize()

    def step_resident():
        return sb.SNARK.prove(inst, comm, d_vars, inputs, gens, b"example", seed)

    def step_e2e():
        return sb.SNARK.prove(inst, comm, host_vars, inputs, gens, b"example", seed)

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local if world > 1 else 0)
    # ---- timed region 1: inputs resident ("value")
    launches0 = sb.kernel_launches()
    barrier()
    if rank == 0:
        sampler.start()
    per_step = []
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        api.timer_start(ctx)
        proof = step_resident()
        per_step.append(api.timer_stop_ms(ctx))
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = sb.kernel_launches() - launches0
    proof_resident = proof
    t_res = sum(per_step) / 1e3
    # ---- timed region 2: end to end through the public API with host buffers
    step_e2e()
    h0, d0 = api.io_bytes()
    barrier()
    per_step_e2e = []
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        w0 = time.perf_counter()                    # host wall-clock around the public call: the call is synchronous (it returns the proof bytes)
        proof = step_e2e()
        per_step_e2e.append((time.perf_counter() - w0) * 1e3)
    barrier()
    h1, d1 = api.io_bytes()
    t_e2e = sum(per_step_e2e) / 1e3
    t_res, t_e2e = sd.max_over_ranks([t_res, t_e2e])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"proof_bytes": proof_resident.bytes, "proof_bytes_e2e": proof.bytes})
    # ---- roofline leg: CUDA-event timing of every kernel family over one more step (separate from the timed regions above)
    roof = None
    if rank == 0:
        ctx.set_overlap(False)     # every kernel on the prover's stream: per-launch event times free of the background MSM (not a timed region)
        api.prof_enable(True)
        step_resident()
        rep = api.prof_report()
        api.prof_enable(False)
        ctx.set_overlap(True)
        pk, which = peaks()
        tot = sum(v["ms"] for v in rep.values())
        dom = max(rep.items(), key=lambda kv: kv[1]["ms"])
        fold = rep.get("sc_fold_eval")

        def rl(name, v, bound="hbm"):
            ach = v["bytes"] / 1e9 / (v["ms"] / 1e3) if v["ms"] else 0.0
            big = v["largest_bytes"] / 1e9 / (v["largest_ms"] / 1e3) if v["largest_ms"] else 0.0
            return {"kernel": name, "bound": bound, "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": None,
                    "launches": v["launches"], "ms_per_step": v["ms"], "share_of_kernel_time": v["ms"] / tot if tot else None, "peak_source": which,
                    "largest_launch": {"algorithmic_bytes": v["largest_bytes"], "us": v["largest_ms"] * 1e3, "achieved": big, "frac": big / pk["hbm_gbs"]}}
        # BASELINE.json asks for the fraction of the HBM roofline of the sumcheck fold: `roofline` is that kernel, k_sc_fold_eval (fused fold + round
        # evaluation on tables of >= 8192 entries, 48*len algorithmic bytes per distinct table per launch).  `achieved` averages over all its launches of
        # a step; `largest_launch` is the 18-instance first round of the ops proof.  The tiny late rounds run a different, latency-bound kernel
        # (k_sc_fold_eval_small, family sc_fold_eval_small in kernels_ms_per_step).
        roof = rl("sc_fold_eval", fold) if fold else None
        if roof:
            roof["note"] = ("algorithmic bytes = 48 B x len per table per launch (read len*32, write len/2*32); CUDA-event time per launch on the prover stream, measured in one extra "
                            "step with the background-stream overlap switched off (sp_ctx_set_overlap(0)) so that no other kernel shares the GPU; "
                            "ncu --set full of the same kernel: profiles/r02_ncu_full_sc_fold_eval.txt; the multiplications are FMA-pipe bound (IMAD.WIDE at quarter rate, "
                            "profiles/r02_tuning.md section 1): the pipe ceiling of the cubic-4 round is ~0.55 of the HBM copy bandwidth")
        if roof:
            # dram__bytes_read.sum + dram__bytes_write.sum of this kernel's first launch of a step, from the committed ncu capture (written by
            # tools/ncu_summary.py full ... --json); null when no capture of the current build is committed
            try:
                with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
                    tr = json.load(f)["sc_fold_eval"]
                roof["traffic"] = tr["dram_bytes"]
                roof["traffic_note"] = "%s; algorithmic bytes of that launch %.4g" % (tr["what"], tr["algorithmic_bytes"])
            except Exception:
                roof["traffic"] = None
        roof_msm = rl(dom[0], dom[1], "hbm")
        try:   # integer-issue roofline of the dominant kernel from the committed ncu capture: executed warp instructions / (duration x issue peak)
            with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
                cap = json.load(f)[dom[0]]
            peak_wi = 148 * 4 * pk.get("sm_max_mhz", 1965.0) * 1e6      # one warp instruction per cycle per SM sub-partition
            roof_msm["roofline_int"] = {"bound": "issue (INT32 pipe: IMAD.WIDE carry chains)", "warp_instructions": cap["warp_instructions"], "us": cap["us"],
                                        "achieved": cap["warp_instructions"] / (cap["us"] * 1e-6) / 1e9, "peak": peak_wi / 1e9, "unit": "G warp-instr/s",
                                        "frac": cap["warp_instructions"] / (cap["us"] * 1e-6) / peak_wi, "traffic": cap["dram_bytes"], "source": cap["what"]}
        except Exception:
            pass
        roof_msm["note"] = ("dominant kernel by time; fixed-base ristretto255 comb, INTEGER-ALU bound (20 table lookups x 7 field multiplications per term): its "
                            "algorithmic bytes are only scalars + bases, so the HBM fraction is honestly tiny")
        kernels = {k: {"launches": v["launches"], "ms": round(v["ms"], 4)} for k, v in sorted(rep.items(), key=lambda kv: -kv[1]["ms"])}
        # BASELINE.json's second metric: MSM point additions per second, on the largest MSM of the step (the 2048 x 4096 commitment to the
        # dereferenced values, 2^23 terms with 253-bit scalars): reference-equivalent adds (33 per term, dalek Pippenger w=8) and executed table additions
        m = rep.get("msm_rows")
        msm_rate = None
        if m and m["largest_ms"]:
            terms = m["largest_bytes"] / 32.0
            msm_rate = {"terms": terms, "ms": m["largest_ms"], "Mpoint_adds_per_s_reference_equivalent": 33.0 * terms / (m["largest_ms"] / 1e3) / 1e6,
                        "Mpoint_adds_per_s_executed": 20.0 * terms / (m["largest_ms"] / 1e3) / 1e6, "Mterms_per_s": terms / (m["largest_ms"] / 1e3) / 1e6,
                        "what": "largest msm_rows launch of the step: commit_nondet_witness, 2048 rows x 4096 generators (sparse_mlpoly.rs:64-67)"}
    # ---- strong scaling: ONE proof (rank 0's instance: seed 0) sharded over all N GPUs
    strong = None
    if world > 1 and not sharded_legs:
        strong = {"skipped": "sharded legs are on by default only at the world sizes validated on hardware %s; SP_BENCH_SHARDED=1 forces them" % (SHARDED_VALIDATED_WORLDS,)}
    if sharded_legs and not args.no_strong:
        import hashlib
        if rank == 0:
            inst0, inputs0, comm0, dv0 = inst, inputs, comm, d_vars
        else:
            inst0, vars0, inputs0 = sb.Instance.produce_synthetic_r1cs(n, n, NUM_INPUTS, seed=0, ctx=ctx)
            comm0 = sb.SNARK.encode(inst0, gens)
            dv0 = sb.DensePolynomial(vars0.limbs, ctx=ctx)
        seed0 = sb.tape_seed(0)
        single = sb.SNARK.prove(inst0, comm0, dv0, inputs0, gens, b"example", seed0)          # every rank alone: the reference bytes
        ctx.set_sharding(True)
        for _ in range(max(args.warmup, 3)):
            sharded = sb.SNARK.prove(inst0, comm0, dv0, inputs0, gens, b"example", seed0)
        barrier()
        ts = []
        for _ in range(args.steps):
            flush.zero_()
            barrier()
            api.timer_start(ctx)
            sharded = sb.SNARK.prove(inst0, comm0, dv0, inputs0, gens, b"example", seed0)
            ts.append(api.timer_stop_ms(ctx))
        barrier()
        phases = {k: round(v, 3) for k, v in ctx.timings().items() if not k.startswith("fine:")}
        ctx.set_sharding(False)
        t_strong = sd.max_over_ranks([sum(ts) / 1e3])[0]
        same = sd.max_over_ranks([0.0 if sharded.bytes == single.bytes else 1.0])[0] == 0.0
        strong = {"what": "ONE SNARK::prove of the same configuration sharded over %d GPUs (intra-proof: cyclic table shards, row-sharded commitments, "
                          "partial sums exchanged over NVLink inside the reduction kernels); latency, not throughput" % world,
                  "scaling": "strong", "ms_per_proof": t_strong / args.steps * 1e3, "constraints_per_s": n * args.steps / t_strong,
                  "speedup_vs_one_gpu_same_run": (t_res / args.steps) / (t_strong / args.steps),
                  "proof_bytes_identical_to_single_gpu_on_every_rank": same, "proof_sha256": hashlib.sha256(sharded.bytes).hexdigest(), "phases_ms": phases,
                  "limiter": "the ~490 transcript-serialised rounds (latency-bound, replicated on every rank) and the replicated inner-product arguments; only the "
                             "streaming rounds, the commitments and the product-circuit layers shard"}
    # ---- BASELINE.json configs[2] and configs[3] at N GPUs (all ranks take part)
    msm_var, dense_sc = None, None
    if not args.no_msm_var and (world == 1 or sharded_legs):
        if world > 1:
            ctx.set_sharding(True)
        try:
            dense_sc = dense_sumcheck_leg(sb, api, sd, ctx, rank, world, peaks()[0])
            msm_var = msm_var_leg(sb, api, sd, ctx, rank, world)
        except Exception as ex:   # extras, never the headline: report instead of failing the bench line
            msm_var = {"error": str(ex)}
    if rank != 0:
        sd.finalize()
        return
    cpu = cpu_baseline_leg() if world == 1 and not args.no_cpu_baseline else None
    out = {
        "metric": METRIC, "value": sd.aggregate_throughput(n * args.steps, world, t_res), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": t_res / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 (8x32-bit limbs, 256-bit modular integer arithmetic)", "data": "synthetic",
        "config": {"workload": "SNARK::prove synthetic R1CS 2^%d cons/vars, 2^%d non-zero, %d inputs (BASELINE.json configs[1])" % (LOG_N, LOG_N, NUM_INPUTS),
                   "per_gpu": "one independent proof per GPU per step", "l2": "512 MiB buffer zeroed between timed iterations (L2 flush); working set ~2.5 GB >> 126 MB L2",
                   "timed_region": "Transcript::new + SNARK::prove (benches/snark.rs:55-68); gens / instance / encode excluded", "timer": "CUDA events on the prover stream, max over ranks"},
        "clocks": clocks,
        "e2e": {"value": sd.aggregate_throughput(n * args.steps, world, t_e2e), "unit": UNIT, "ms_per_step": t_e2e / args.steps * 1e3, "h2d_bytes_per_step": (h1 - h0) // args.steps,
                "d2h_bytes_per_step": (d1 - d0) // args.steps, "api": "spartan_b200.SNARK.prove -> sp_snark_prove (C ABI), assignment in pinned host memory", "timer": "host wall-clock (perf_counter) around the synchronous call, max over ranks"},
        "gpu_launches": launches,
        "proof_bytes": len(proof.bytes),
        "roofline": roof, "roofline_dominant_kernel": roof_msm, "msm": msm_rate, "msm_var_2p24": msm_var, "dense_sumcheck_2p22": dense_sc, "strong": strong, "kernels_ms_per_step": kernels,
        "phases_ms": {k: round(v, 3) for k, v in ctx.timings().items()},
        "cpu_baseline": cpu,
        "reference_published": {"value": 2 ** 20 / 39.1297568, "unit": UNIT, "what": "README.md:375 SNARK::prove 2^20 on one core of an i7-1065G7 (other hardware)"},
    }
    print(json.dumps(out), flush=True)
    sd.finalize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-msm-var", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proof bytes of the last timed step of each timed region to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
