#!/usr/bin/env python3
"""bench.py -- candidates scored / s of PLinOpt's candidate-search hot path on 1..8 B200, one process per GPU.

  python bench.py --gpus N --steps K --warmup W            (engine arm; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  (CPU arm: the oracle restatement on the box's host cores)

Headline (BASELINE.json configs[1], "C2"): DeGroote-orbit sweep of 2x2x2_7_Winograd_{L,R,P} minimising the growth factor G2.
A step = one sweep of 2^batch_log2 Philox candidates per GPU (weak scaling: every rank owns a disjoint contiguous index range)
+ the single min-allreduce that picks the global winner (done on the device buffer, no host hop).
The same JSON line carries a `configs` object with the other BASELINE configs measured at the run's N:
  C4  orbit + sparsity / growth search on 3x4x7_63_rational          (src/orbiter.cpp:272-324)
  C3  sparsifier CoB search on 4x4x4_48_rational mod 2^31-1: one c = 128 search sharded over the ranks, and the whole
      `sparsifier -q 2147483647 -c 11` pipeline through plo_sparsifier (include/plinopt_sparsify.inl:299-314, 666-748)
  C5  batched MMchecker mod 2^31-1 of 32x32x32_15096, batch 4096 and 32  (include/plinopt_library.inl:472-558)
each with value, roofline (lanes-aware roof stated), e2e through the host-buffer C call and, at N = 1, the CPU oracle beside it.
Prints ONE JSON line on rank 0.  --dump-outputs DIR also writes what the last timed step of each path returned (rank 0's view) as
DIR/<name>.npy in float64; the inputs depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 0x504C494E4F505431
P31 = 2147483647
STEM = "2x2x2_7_Winograd"
WORKLOAD = "orbit sweep of 2x2x2_7_Winograd_{L,R,P}, measure G2 (growthfactor.cpp:117-125), Philox4x32-10 candidates"
METRIC = "candidates scored/sec"
NCU_INPUTS = os.path.join(ROOT, "profiles", "ncu_inputs.json")


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def orbit_ops(m, k, n, r):
    """Algorithmic work per orbit candidate (SURVEY.md section 8d): int32 MAC of the three transforms + one test/square per entry;
    FP64: 3r sqrt + 2r mul + r add for G2."""
    return r * (m * m * k + m * k * k + k * k * n + k * n * n + m * m * n + m * n * n) + r * (m * k + k * n + m * n), 6 * r


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU while the timed region runs (NVML, 20 ms)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")  # NVML numbers the physical devices: map the CUDA ordinal through the mask
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if ids and all(v.isdigit() for v in ids) and index < len(ids):
                index = int(ids[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, rs))
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        nv = self.nv
        sms = sorted(s for s, _ in self.samples)
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
                 "hw_power_brake_slowdown": 0x80, "sync_boost": 0x10, "applications_clocks_setting": 0x2}
        seen = set()
        for _, r in self.samples:
            for k, bit in names.items():
                if r & bit:
                    seen.add(k)
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        return {"sm_mhz": sms[len(sms) // 2], "sm_max_mhz": mx, "reasons": sorted(seen), "samples": len(sms)}


def load_triple(stem):
    import numpy as np
    from plinopt_b200 import hm
    L, R, P = hm.load_fixture(stem)
    mkn = hm.LRP2MM(L, R, P)
    (Li, dl), (Ri, dr), (Pi, dp) = (hm.scaled(M, np.int32) for M in (L, R, P))
    return (L, R, P), mkn, (Li, Ri, Pi), (dl, dr, dp)


def host_threads():
    """Every host core this process may use (torchrun exports OMP_NUM_THREADS=1: the CPU arms override it explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    return O


def ncu_inputs():
    """Per-kernel constants taken from committed ncu captures (profiles/ncu_inputs.json, written by tools/ncu_inputs.py): a value is
    only quoted for the kernel the plan really launches, so a changed kernel selection cannot silently reuse a stale profile."""
    try:
        with open(NCU_INPUTS) as fh:
            return json.load(fh)
    except Exception:
        return {}


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"])
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------------------------------
# CPU arms (the oracle = checker; here only as the timed baseline)
# ------------------------------------------------------------------------------------------------------------------------
def cpu_orbit_rate(fr, measure, target_s, threads):
    """Oracle restatement of the orbiter loop body (src/orbiter.cpp:272-324), OpenMP over candidates; returns (candidates/s, n)."""
    O = oracle()
    L, R, P = fr
    probe = 2000 if len(L) > 20 else 20000
    t0 = time.perf_counter()
    O.orbit_sweep(L, R, P, measure, 1, SEED, 0, probe, nthreads=threads, table=False)
    dt = time.perf_counter() - t0
    n = max(probe, int(probe / max(dt, 1e-6) * target_s))
    t0 = time.perf_counter()
    O.orbit_sweep(L, R, P, measure, 1, SEED, 0, n, nthreads=threads, table=False)
    return n / (time.perf_counter() - t0), n


def c3_problem(c, blocks=(0, 1, 2, 3)):
    """Column blocks of 4x4x4_48_rational_L mod 2^31-1 as (TM 4x48 residues, Coeffs) pairs (plinopt_sparsify.inl:256-270 order)."""
    import numpy as np
    from plinopt_b200 import hm
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from bench_kernels import coeff_list
    L, _, _ = hm.load_fixture("4x4x4_48_rational")
    tms, cfs = [], []
    for blk in blocks:
        TM = [[L[i][4 * blk + t] for i in range(len(L))] for t in range(4)]
        tm = np.array([[(v.numerator % P31) * pow(v.denominator % P31, -1, P31) % P31 for v in row] for row in TM], dtype=np.int64)
        tms.append(tm); cfs.append(coeff_list(tm.tolist(), P31, c))
    return L, tms, cfs


def cpu_c3(target_s, threads):
    """The oracle's literal testLinComb loop (plinopt_sparsify.inl:166-197, 299-314) on block 0, c = 20: one core (the reference loop
    is sequential) and every core (an added outer `omp for`); and the oracle's whole pipeline for -q 2147483647 -c 11."""
    import numpy as np
    O = oracle()
    L, tms, cfs = c3_problem(20, blocks=(0,))
    z = np.zeros((4, 4), dtype=np.int64)
    out = {}
    for nt, key in ((1, "search_1core"), (threads, "search_allcores")):
        i_hi = max(1, min(20, int(round(target_s * (2 if nt == 1 else 2 * nt)))))
        t0 = time.perf_counter()
        tot = O.lincomb_bench(P31, tms[0], np.ones_like(tms[0]), 0, 0, cfs[0], np.ones_like(cfs[0]), z, np.ones_like(z), 0, i_hi, nthreads=nt)[0]
        out[key] = {"value": tot / (time.perf_counter() - t0), "unit": "candidates/s", "cores": nt, "kind": "port",
                    "sample": f"{tot} candidates (i < {i_hi} of 20) of the c = 20 search on block 0, oracle testLinComb loop"}
    t0 = time.perf_counter()
    _, _, ok, tr = O.sparsifier(L, P31, 4, 11, True, trace=True)
    dt = time.perf_counter() - t0
    cand = sum(t["c"] ** 4 for t in tr)
    out["pipeline_c11"] = {"value": cand / dt, "unit": "candidates/s", "cores": 1, "kind": "port", "seconds": dt,
                           "sample": f"one run of the oracle's blockSparsifier pipeline, {len(tr)} (block,num) steps, {cand} candidates"}
    return out


def cpu_c5(big, nsamples, threads):
    """Oracle MMchecker mod p (plinopt_library.inl:472-558), one random (ua, ub) per call, calls spread over the host threads."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    O = oracle()
    mkn, r, (Lc, Rc, Pc) = big
    f = O.lib().orc_mmcheck_modp
    f.argtypes = [C.c_int64] + [C.c_int] * 4 + [O._i64p, O._i32p, O._i64p] * 3 + [O._i64p, O._i64p]
    arrs = []
    for rows, cols, ptr, col, val in (Lc, Rc, Pc):
        arrs += [np.ascontiguousarray(ptr, dtype=np.int64), np.ascontiguousarray(col, dtype=np.int32), np.ascontiguousarray(val, dtype=np.int64)]
    rng = np.random.default_rng(1)
    ins = [(rng.integers(0, P31, Lc[1]).astype(np.int64), rng.integers(0, P31, Rc[1]).astype(np.int64)) for _ in range(nsamples)]

    def one(ab):
        return f(P31, r, Lc[1], Rc[1], Pc[0], *arrs, ab[0], ab[1])
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        verdicts = list(ex.map(one, ins))
    dt = time.perf_counter() - t0
    return {"value": nsamples / dt, "unit": "samples/s", "cores": threads, "kind": "port", "sample": f"{nsamples} random evaluations of the oracle MMchecker on the same triple",
            "all_correct": all(v == 0 for v in verdicts)}


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    fr, mkn, _, _ = load_triple(STEM)
    O = oracle()
    cores = host_threads()
    rate0, _ = cpu_orbit_rate(fr, 3, 1.0, cores)
    n = max(1000, int(rate0 * 4.0))  # each "step" = a bounded sample of the same workload (about 4 s with every host thread)
    for _ in range(args.warmup):
        O.orbit_sweep(*fr, 3, 1, SEED, 0, max(1000, n // 8), nthreads=cores, table=False)
    t0 = time.perf_counter()
    for s in range(args.steps):
        O.orbit_sweep(*fr, 3, 1, SEED, s * n, (s + 1) * n, nthreads=cores, table=False)
    dt = time.perf_counter() - t0
    val = args.steps * n / dt
    configs = {}
    if not args.no_configs:
        fr4, _, _, _ = load_triple("3x4x7_63_rational")
        for meas, name in ((0, "nnz"), (3, "G2")):
            rate, cnt = cpu_orbit_rate(fr4, meas, 3.0, cores)
            configs[f"C4_orbit_3x4x7_{name}"] = {"value": rate, "unit": "candidates/s", "cores": cores, "kind": "port", "sample": f"{cnt} Philox candidates"}
        configs["C3_sparsifier_4x4x4"] = cpu_c3(2.0, cores)
        from plinopt_b200 import hm
        big = hm.load_large_csr(P31)
        if big is not None:
            configs["C5_mmcheck_32x32x32"] = cpu_c5(big, 4 * cores, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "candidates/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64 rationals + f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "candidates_per_gpu_per_step": n,
                   "note": "CPU oracle (port of src/orbiter.cpp:272-324; the reference itself needs LinBox/Givaro and cannot be built here); a step is a bounded sample of the workload"},
        "cpu_baseline": {"value": val, "unit": "candidates/s", "cores": cores, "kind": "port", "sample": f"{args.steps} x {n} Philox candidates, OpenMP over candidates"},
        "e2e": {"value": val, "unit": "candidates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "configs": configs,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------------------
# engine arm
# ------------------------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def keep_output(ctx, name, values):
    """What the last timed step of a path returned to its caller, for --dump-outputs (rank 0's view)."""
    if ctx.rank == 0:
        import numpy as np
        ctx.outputs[name] = np.asarray(values, dtype=np.float64)


def orbit_record(g):
    """(score, nnz, nno, index) of a sweep's winner, the fields of plo_orbit_best; NaN when no candidate was swept."""
    return [float("nan")] * 4 if g is None else [g["score"], g["nnz"], g["nno"], g["index"]]


def barrier(ctx):
    import torch
    if ctx.world > 1:
        ctx.dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ctx, x):
    import torch
    if ctx.world == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=ctx.dev)
    ctx.dist.all_reduce(t, op=ctx.dist.ReduceOp.MAX)
    return float(t.item())


def timed_steps(ctx, step, steps, warmup):
    """W untimed steps, then K steps each bracketed by CUDA events on the launch stream (the L2 flush between steps sits outside the
    event pairs); barrier + synchronize on both sides; returns the max-over-ranks sum of the K device times in ms."""
    import torch
    for s in range(warmup):
        ctx.flush.zero_()
        step(s)
    barrier(ctx)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s in range(steps):
        ctx.flush.zero_()
        evs[s][0].record(ctx.stream)
        step(warmup + s)
        evs[s][1].record(ctx.stream)
    barrier(ctx)
    return max_over_ranks(ctx, sum(a.elapsed_time(b) for a, b in evs))


def wall_steps(ctx, step, steps, warmup=1):
    """End-to-end timing: wall clock around calls that take host buffers and return host results (copies inside)."""
    for s in range(warmup):
        step(s)
    barrier(ctx)
    t0 = time.perf_counter()
    for s in range(steps):
        step(warmup + s)
    barrier(ctx)
    return max_over_ranks(ctx, time.perf_counter() - t0)


def orbit_roofline(ctx, plan, ops_int, ops_fp, cand_per_s, kern_ms, units_per_launch):
    """Lanes-aware integer roof: one 32-bit multiply-add of the selected kernel carries `lanes` candidate-matrix entries, so the roof
    of the algorithmic int32 operation rate is lanes x the measured IMAD peak.  The issue-slot view is quoted only when the
    committed ncu capture is of the kernel this plan launches."""
    peaks = ctx.peaks
    imad = peaks["imad_per_s"] / 1e12
    achieved = ops_int * cand_per_s / 1e12
    peak = plan.lanes * imad
    prof = ctx.ncu.get(f"{plan.kernel}|{'x'.join(str(v) for v in plan.mkn)}|{'G2' if plan.measure == 3 else 'nnz'}")
    issue = None
    traffic = None
    if prof:
        inst = prof["inst_per_candidate"]
        issue_peak = peaks["issue_inst_per_s"] / 1e12
        if ctx.clock_peak:
            issue_peak = max(issue_peak, ctx.clock_peak)
        issue = {"thread_instructions_per_candidate": inst, "achieved": inst * cand_per_s / 1e12, "peak": issue_peak, "frac": inst * cand_per_s / 1e12 / issue_peak,
                 "unit": "T thread-instructions/s", "source": prof["source"]}
        traffic = prof.get("dram_bytes_per_launch")
        if prof.get("smem_wavefronts_per_candidate") and ctx.clock_peak:
            wpeak = ctx.clock_peak / 128.0  # T wavefronts/s: one 128 B shared-memory wavefront per SM per clock (clock_peak = SMs x 4 x 32 x clock)
            w = prof["smem_wavefronts_per_candidate"]
            issue["shared_memory"] = {"wavefronts_per_candidate": w, "achieved": w * cand_per_s / 1e12, "peak": wpeak, "frac": w * cand_per_s / 1e12 / wpeak,
                                      "unit": "T wavefronts/s", "note": "the table-driven kernels are bound by issue slots and by shared-memory bandwidth together"}
    hbm_peak = measured_hbm_peak()
    return {"bound": "int32", "achieved": achieved, "peak": peak, "unit": "T int32 ops/s (algorithmic)", "frac": achieved / peak, "traffic": traffic,
            "kernel": plan.kernel, "lanes_per_imad": plan.lanes, "kernel_ms": kern_ms,
            "ops_per_candidate": {"int32": ops_int, "fp64": ops_fp},
            "peak_source": f"{plan.lanes} lanes x plo_measure_peaks IMAD peak ({imad:.2f} T/s, measured in this run; MEASURED_PEAKS.json has no int32 entry)",
            "vs_scalar_imad_peak": achieved / imad,
            "issue_slots": issue if issue else "no committed ncu capture of this kernel: not quoted",
            "fp64": {"achieved_tflop": ops_fp * cand_per_s / 1e12, "peak_dfma_tflop": 2 * peaks["dfma_per_s"] / 1e12},
            "hbm": {"bytes_per_launch": traffic, "achieved_GBs": (traffic / (kern_ms * 1e-3) / 1e9) if traffic else None, "peak_GBs": hbm_peak,
                    "note": "the sweep reads its matrices from constant memory and writes one 16 B key per block"},
            "bound_note": "contract bound classes are hbm|tensor; this kernel is neither: integer multiply-add throughput (fma-heavy pipe) and instruction issue bind it"}


def bench_orbit(ctx, name, stem, measure, batch_log2, steps, warmup, cpu_seconds, headline=False):
    """Weak-scaling orbit sweep: every rank sweeps its own 2^batch_log2 candidates per step; winner through one device-side
    min-allreduce over a world x 4 table."""
    import torch
    from plinopt_b200 import capi, sharding
    fr, mkn, (Li, Ri, Pi), dens = load_triple(stem)
    m, k, n = mkn
    r = len(fr[0])
    B = 1 << batch_log2
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, measure, capi.MODE_PHILOX, SEED)
    plan.mkn, plan.measure = mkn, measure
    slots = torch.empty((steps + warmup + 8, ctx.world * 4), dtype=torch.int64, device=ctx.dev)

    def step(s):
        lo = (s * ctx.world + ctx.rank) * B
        plan.run(lo, lo + B, ctx.sp)
        row = slots[s % slots.shape[0]]
        plan.pack(row.data_ptr(), ctx.rank, ctx.world, ctx.sp)
        if ctx.world > 1:  # the engine's own NCCL all-reduce on the device table, same stream: no host hop, no torch on the data path
            ctx.comm.allreduce_i64(row.data_ptr(), ctx.world * 4, capi.REDUCE_MIN, ctx.sp)

    sampler = ClockSampler(ctx.local) if headline else None
    if sampler:
        for s in range(warmup):
            ctx.flush.zero_()
            step(s)
        barrier(ctx)
        sampler.start()
        t_wall0 = time.perf_counter()
        ms = timed_steps(ctx, lambda s: step(s + warmup), steps, 0)
        t_wall = time.perf_counter() - t_wall0
        sampler.stop_flag = True
        sampler.join()
    else:
        t_wall0 = time.perf_counter()
        ms = timed_steps(ctx, step, steps, warmup)
        t_wall = time.perf_counter() - t_wall0
    table = slots[warmup:warmup + steps].cpu().tolist()  # every step's gathered winners, read once after the timed region
    keep_output(ctx, name, orbit_record(sharding.pick_global(table[-1], ctx.world, measure_nnz=(measure == capi.MEASURE_NNZ))))
    overall = None
    for words in table:
        g = sharding.pick_global(words, ctx.world, measure_nnz=(measure == capi.MEASURE_NNZ))
        if g is not None and (overall is None or (g["score"], g["index"]) < (overall["score"], overall["index"])):
            overall = g
    value = steps * ctx.world * B / (ms * 1e-3)

    # the sweep kernel alone (sweep + final launches back to back, no collective): roofline numerator
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(3, min(steps, 10))
    torch.cuda.synchronize()
    k0.record(ctx.stream)
    for s in range(reps):
        plan.run((1000 + s) * B, (1001 + s) * B, ctx.sp)
    k1.record(ctx.stream)
    torch.cuda.synchronize()
    kern_ms = k0.elapsed_time(k1) / reps

    # end to end through the host-buffer C call: upload of L/R/P, plan, sweep, 24 B result download, every step
    e_steps = max(3, min(steps, 10))
    h2d = int(Li.nbytes + Ri.nbytes + Pi.nbytes)

    def e2e_step(s):
        lo = ((5000 + s) * ctx.world + ctx.rank) * B
        best = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, measure, capi.MODE_PHILOX, SEED, lo, lo + B)
        if ctx.world > 1:
            sharding.allreduce_best(best, measure_nnz=(measure == capi.MEASURE_NNZ), device=ctx.dev)
    e_dt = wall_steps(ctx, e2e_step, e_steps)
    e2e_val = e_steps * ctx.world * B / e_dt

    out = None
    if ctx.rank == 0:
        ops_int, ops_fp = orbit_ops(m, k, n, r)
        if measure != capi.MEASURE_G2:
            ops_fp = 0
        if sampler:
            ctx.clocks = sampler.summary()
            try:
                if ctx.clocks.get("sm_mhz"):
                    ctx.clock_peak = torch.cuda.get_device_properties(ctx.dev).multi_processor_count * 4 * 32 * float(ctx.clocks["sm_mhz"]) * 1e6 / 1e12
            except Exception:
                pass
        cpu = None
        if ctx.world == 1 and cpu_seconds > 0:
            rate, cnt = cpu_orbit_rate(fr, measure, cpu_seconds, host_threads())
            cpu = {"value": rate, "unit": "candidates/s", "cores": host_threads(), "kind": "port",
                   "sample": f"{cnt} Philox candidates of the same workload (oracle, OpenMP over candidates)"}
        out = {"workload": f"orbit sweep of {stem}_{{L,R,P}}, measure {'G2' if measure == capi.MEASURE_G2 else 'nnz/nno'}, Philox candidates",
               "metric": METRIC, "value": value, "unit": "candidates/s", "scaling": "weak", "n_gpus": ctx.world, "steps": steps,
               "ms_per_step": ms / steps, "candidates_per_gpu_per_step": B,
               "e2e": {"value": e2e_val, "unit": "candidates/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 24, "steps": e_steps, "api": "plo_orbit_sweep (host buffers)"},
               "gpu_launches": steps * (plan.launches + 1),
               "roofline": orbit_roofline(ctx, plan, ops_int, ops_fp, B / (kern_ms * 1e-3), kern_ms, B),
               "cpu_baseline": cpu, "best": overall, "wall_s": t_wall}
    plan.close()
    return out


def bench_orbit_strong(ctx, stem, measure, total_log2, steps):
    """Strong scaling: ONE fixed sweep of 2^total_log2 candidates per step, split into contiguous shards over the ranks."""
    from plinopt_b200 import capi, sharding
    import torch
    fr, mkn, (Li, Ri, Pi), dens = load_triple(stem)
    total = 1 << total_log2
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, measure, capi.MODE_PHILOX, SEED)
    lo, hi = sharding.shard_range(0, total, ctx.rank, ctx.world)
    slots = torch.empty((ctx.world * 4,), dtype=torch.int64, device=ctx.dev)

    def step(s):
        plan.run(lo, hi, ctx.sp)
        plan.pack(slots.data_ptr(), ctx.rank, ctx.world, ctx.sp)
        if ctx.world > 1:
            ctx.comm.allreduce_i64(slots.data_ptr(), ctx.world * 4, capi.REDUCE_MIN, ctx.sp)
    ms = timed_steps(ctx, step, steps, 1)
    g = sharding.pick_global(slots.cpu().tolist(), ctx.world, measure_nnz=(measure == capi.MEASURE_NNZ))
    keep_output(ctx, "C2_strong", orbit_record(g))
    plan.close()
    if ctx.rank != 0:
        return None
    return {"workload": f"one fixed sweep of 2^{total_log2} candidates of {stem} split over the ranks", "scaling": "strong", "n_gpus": ctx.world,
            "value": steps * total / (ms * 1e-3), "unit": "candidates/s", "ms_per_step": ms / steps, "steps": steps, "best": g}


def bench_c3(ctx, steps, warmup, cpu_seconds):
    """C3: (a) one c = 128 search over the 4 column blocks of 4x4x4_48_rational_L mod 2^31-1, its prefix range sharded over the
    ranks (strong scaling), winners merged by one max-allreduce; (b) the whole `-q 2147483647 -c 11` pipeline through plo_sparsifier
    (host buffers in, CoB/Res out) on rank 0."""
    import numpy as np
    import torch
    from plinopt_b200 import capi, sharding
    c = 128
    L, tms, cfs = c3_problem(c)
    m = 48
    plan = capi.LincombPlan(P31, np.stack(tms), 0, np.stack(cfs))
    lo, hi = sharding.shard_range(0, c ** 3, ctx.rank, ctx.world)
    merged = {}

    def step(s):
        plan.run_range(lo, hi, ctx.sp)
        if ctx.world > 1:
            mine = [(int(a), int(b), None if int(i) == capi.NO_INDEX else int(i)) for a, b, i in zip(*plan.result(ctx.sp))]
            merged["best"] = sharding.allreduce_lincomb(mine, device=ctx.dev)
    ms = timed_steps(ctx, step, steps, warmup)
    if ctx.world == 1:
        merged["best"] = [(int(a), int(b), None if int(i) == capi.NO_INDEX else int(i)) for a, b, i in zip(*plan.result(ctx.sp))]
    keep_output(ctx, "C3_sparsifier_4x4x4_search_c128", [(rl, cl, -1 if i is None else i) for rl, cl, i in merged["best"]])  # (rl, cl, index) per block
    cand = plan.candidates
    value = steps * cand / (ms * 1e-3)
    launches = plan.launches
    plan.close()

    # e2e of the search: all FOUR rows of the four blocks through the host-buffer quad call (score once, filter four times)
    quad = None
    pipe = None
    if ctx.rank == 0:
        probs = [dict(TM=tm, off=0, coeffs=cf) for tm, cf in zip(tms, cfs)]
        capi.lincomb_quad(P31, probs)
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            res = capi.lincomb_quad(P31, probs)
        dt = (time.perf_counter() - t0) / reps
        covered = 4 * len(probs) * c ** 4
        h2d = sum(tm.nbytes + cf.nbytes for tm, cf in zip(tms, cfs))
        quad = {"value": covered / dt, "unit": "candidates/s (reference-loop evaluations covered: 4 rows x 4 blocks x c^4; each candidate is scored once)",
                "seconds_per_call": dt, "scored_per_s": len(probs) * c ** 4 / dt, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 36 * len(probs),
                "api": "plo_lincomb_quad (host buffers)", "rows": [r for _, r in res][0]}
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import time_sparsifier_c as T
        pipe = T.time_case(L, P31, 11, reps=30)
    out = None
    if ctx.rank == 0:
        pair_peak = ctx.peaks["ialu_pairs_per_s"]
        out = {"search_c128": {
                   "workload": "sparsifier CoB search, 4x4x4_48_rational_L mod 2^31-1, 4 column blocks, c = 128 (one row per block), prefix range sharded over the ranks",
                   "metric": METRIC, "value": value, "unit": "candidates/s", "scaling": "strong", "n_gpus": ctx.world, "steps": steps, "ms_per_step": ms / steps,
                   "candidates_per_step": cand, "gpu_launches": steps * launches, "best_per_block": merged.get("best"),
                   "roofline": {"bound": "int32 alu", "achieved": value / ctx.world * m / 1e12, "peak": pair_peak / 1e12, "unit": "T compare+add pairs/s per GPU",
                                "frac": value / ctx.world * m / pair_peak, "traffic": None, "kernel": "lincomb_inv_kernel<48> (c >= 32 mod p; lincomb_kernel<u32,48,modp> below)",
                                "work_per_candidate": f"{m} compare+add pairs (the 4m MAC of the reference formulation are folded into the host-built product tables)",
                                "note": "frac > 1 is not a measurement error: for c >= 32 mod p the kernel does not compare every (candidate, coordinate) pair -- per prefix and "
                                        "coordinate ONE multiplication by -A3^-1 and one hash probe find the l that make the coordinate vanish (lincomb_inv_kernel), c-fold fewer "
                                        "operations than the compare formulation the unit of work is taken from; results are identical (tests/test_gpu_lincomb.py)",
                                "peak_source": "plo_measure_peaks ISETP+IADD pair peak, measured in this run"},
                   "e2e": quad},
               "pipeline_c11": None if pipe is None else {
                   "workload": "bin/sparsifier -q 2147483647 -c 11 on 4x4x4_48_rational_L: whole blockSparsifier pipeline through plo_sparsifier (host buffers in, CoB/Res out)",
                   "metric": METRIC, "value": pipe["candidates_per_s"], "unit": "candidates/s (reference-loop evaluations covered)", "n_gpus": 1,
                   "seconds_per_run": pipe["seconds"], "candidates": pipe["candidates"], "device_round_trips": pipe["round_trips"], "consistent": pipe["consistent"],
                   "nnz_res": pipe["nnz_res"],
                   "e2e": {"value": pipe["candidates_per_s"], "unit": "candidates/s", "h2d_bytes_per_step": 48 * 16 * 16, "d2h_bytes_per_step": (16 * 16 + 48 * 16) * 16,
                           "api": "plo_sparsifier (host buffers)"},
                   "roofline": {"bound": "latency", "note": "three device round trips of ~14 641 candidates per block: launch + instruction-fetch latency and the host's exact "
                                "algebra bind this path, not a pipe; the search kernels' roofline is the search_c128 entry", "frac": None, "traffic": None},
                   "round1_value": 3.9e7}}
        if ctx.world == 1 and cpu_seconds > 0:
            cpu = cpu_c3(min(cpu_seconds, 2.0), host_threads())
            out["search_c128"]["cpu_baseline"] = {"one_core": cpu["search_1core"], "all_cores": cpu["search_allcores"]}
            out["pipeline_c11"]["cpu_baseline"] = cpu["pipeline_c11"]
    return out


def bench_c5(ctx, steps, warmup, cpu_seconds):
    """C5: batched MMchecker mod 2^31-1 of 32x32x32_15096 (regenerated from the reference's .slp): every rank checks its own batch of
    Philox (ua, ub) samples per step (weak scaling); verdicts AND-ed."""
    import torch
    from plinopt_b200 import capi, hm
    big = hm.load_large_csr(P31)
    if big is None:
        return {"unavailable": "tests/golden/large/32x32x32_15096.npz is missing"} if ctx.rank == 0 else None
    mkn, r, (Lc, Rc, Pc) = big
    nnz = sum(len(x[3]) for x in (Lc, Rc, Pc))
    mac = nnz + r + mkn[0] * mkn[1] * mkn[2]
    out = {}
    for batch in (4096, 32):
        t0 = time.perf_counter()
        plan = capi.MMcheckPlan(P31, mkn, r, Lc, Rc, Pc, batch)
        create_s = time.perf_counter() - t0
        ms = timed_steps(ctx, lambda s: plan.run(SEED, (s * ctx.world + ctx.rank) * batch, ctx.sp), steps, warmup)
        v, ok = plan.result(ctx.sp)
        keep_output(ctx, f"C5_mmcheck_32x32x32_batch_{batch}_verdict", [v])
        keep_output(ctx, f"C5_mmcheck_32x32x32_batch_{batch}_ok", ok)
        allok = torch.tensor([int(v == 0 and ok.all())], dtype=torch.int64, device=ctx.dev)
        if ctx.world > 1:
            ctx.dist.all_reduce(allok, op=ctx.dist.ReduceOp.MIN)
        value = steps * ctx.world * batch / (ms * 1e-3)

        def e2e_step(s):
            plan.run(SEED, ((9000 + s) * ctx.world + ctx.rank) * batch, ctx.sp)
            plan.result(ctx.sp)  # batch verdict bytes + the verdict word, device -> host
        e_steps = max(3, min(steps, 10))
        e_dt = wall_steps(ctx, e2e_step, e_steps)
        launches = plan.launches
        enc = plan.encoding
        plan.close()
        if ctx.rank == 0:
            wave_peak = torch.cuda.get_device_properties(ctx.dev).multi_processor_count * 32 * (ctx.clocks.get("sm_mhz") or 1965.0) * 1e6
            per_gpu = value / ctx.world
            entry = {"workload": f"batched MMchecker mod 2^31-1, 32x32x32_15096_{{L,R,P}} ({nnz} non-zeroes), {batch} Philox samples per GPU per step",
                     "metric": "samples checked/sec", "value": value, "unit": "samples/s", "scaling": "weak", "n_gpus": ctx.world, "steps": steps,
                     "ms_per_step": ms / steps, "modmac_per_s": value * mac, "all_samples_agree": bool(allok.item()), "gpu_launches": steps * launches,
                     "e2e": {"value": e_steps * ctx.world * batch / e_dt, "unit": "samples/s", "h2d_bytes_per_step": 16, "d2h_bytes_per_step": batch + 4, "steps": e_steps,
                             "api": "plo_mmcheck_plan_run + plo_mmcheck_plan_result (the CSR triple is uploaded once at plan creation, like the reference's loaded matrices; "
                                    f"plan creation {create_s:.2f} s)"},
                     "roofline": {"bound": "shared-memory wavefronts", "achieved": per_gpu * mac / 1e12, "peak": wave_peak / 1e12, "unit": "T modular MAC/s per GPU",
                                  "frac": per_gpu * mac / wave_peak, "traffic": (ctx.ncu.get(f"mmcheck_pass|32x32x32_15096|batch_{batch}") or {}).get("dram_bytes_per_pass"),
                                  "traffic_note": "DRAM bytes of the five launches of one pass (profiles/ncu_inputs.json): the vectors va, vc and the partial products of P "
                                                  "(batch x 60 / 60 / 48 KB) exceed the L2 at batch 4096 and make one round trip each",
                                  "kernel": "mm_slab_spmm_kernel x3 (+ gen, verify)",
                                  "peak_source": "one 128 B shared-memory wavefront per multiply-add of the CSR per warp: SMs x 32 lanes x SM clock",
                                  "encoded": {"x_loads_per_sample": sum(enc["loads"]), "csr_entries": nnz, "col_stride": enc["col_stride"], "row_stride": enc["row_stride"],
                                              "wavefront_frac": per_gpu * 2 * sum(enc["loads"]) / wave_peak,
                                              "note": "the plan's encoder rewrites the rows with column / row block sums (csrc/mmcheck.cu): the kernels read x_loads_per_sample "
                                                      "words of X per sample instead of one per CSR entry, so `frac` (CSR multiply-adds against the one-wavefront-per-entry roof) can "
                                                      "exceed 1; wavefront_frac = (X loads + as many wavefronts of 8-byte stream words) x samples / 32 against the same peak"},
                                  "hbm": {"encoded_bytes": sum(enc["blob_bytes"]), "peak_GBs": measured_hbm_peak(),
                                          "note": "the encoded matrices (3 MB) stay L2-resident; va, vc and the partial products of P (batch x 60 / 60 / 48 KB) are the HBM "
                                                  "traffic (1.35 GB per pass at batch 4096 = 1 TB/s); small batches are latency-bound (slab fill + block sums per launch)"}}}
            out[f"batch_{batch}"] = entry
    if ctx.rank == 0 and ctx.world == 1 and cpu_seconds > 0:
        out["cpu_baseline"] = cpu_c5(big, 4 * host_threads(), host_threads())
    return out if ctx.rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--batch-log2", type=int, default=31, help="C2 candidates per GPU per step = 2^this")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline sample budget of the headline (the configs use a quarter each)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline only (skip C3/C4/C5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of each path's last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the engine arm (the reference arm sizes its steps from a timed probe)")
    if args.warmup < 3 and args.impl == "engine":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from plinopt_b200 import capi

    ctx = Ctx()
    ctx.rank, ctx.world, ctx.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if capi.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(ctx.local)
    capi.set_device(ctx.local)
    ctx.dev = torch.device("cuda", ctx.local)
    ctx.dist = dist
    ctx.comm = None
    if ctx.world > 1:
        dist.init_process_group("nccl", device_id=ctx.dev)  # launch plumbing: barriers, max-over-ranks of the timings, the id exchange below

        def exchange(ident):
            box = [ident]
            dist.broadcast_object_list(box, src=0)
            return box[0]
        ctx.comm = capi.Comm(ctx.rank, ctx.world, exchange)  # the data-path collective is the engine's own (plo_comm_*, NCCL via dlopen)
    ctx.stream = torch.cuda.current_stream()
    ctx.sp = ctx.stream.cuda_stream
    ctx.flush = torch.empty(256 << 20, dtype=torch.uint8, device=ctx.dev)  # > 126 MB L2
    ctx.peaks = capi.measure_peaks(5)
    ctx.ncu = ncu_inputs()
    ctx.clocks, ctx.clock_peak = {}, None
    ctx.outputs = {}
    cpu_s = 0.0 if args.no_cpu_baseline else args.cpu_seconds

    head = bench_orbit(ctx, "C2", STEM, capi.MEASURE_G2, args.batch_log2, args.steps, args.warmup, cpu_s, headline=True)
    configs = {}
    if not args.no_configs:
        configs["C2_strong"] = bench_orbit_strong(ctx, STEM, capi.MEASURE_G2, 33, args.steps)
        configs["C4_orbit_3x4x7_nnz"] = bench_orbit(ctx, "C4_orbit_3x4x7_nnz", "3x4x7_63_rational", capi.MEASURE_NNZ, 22, args.steps, 3, cpu_s / 4)
        configs["C4_orbit_3x4x7_G2"] = bench_orbit(ctx, "C4_orbit_3x4x7_G2", "3x4x7_63_rational", capi.MEASURE_G2, 22, args.steps, 3, cpu_s / 4)
        configs["C3_sparsifier_4x4x4"] = bench_c3(ctx, args.steps, 3, cpu_s / 4)
        configs["C5_mmcheck_32x32x32"] = bench_c5(ctx, args.steps, 3, cpu_s / 4)

    if ctx.rank == 0:
        line = {
            "metric": METRIC, "value": head["value"], "unit": "candidates/s", "n_gpus": ctx.world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32 + f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "candidates_per_gpu_per_step": 1 << args.batch_log2, "seed": hex(SEED),
                       "parallelism": f"index-range sharding x{ctx.world} + one min-allreduce (plo_comm_allreduce_i64: NCCL issued by the engine on the device table)",
                       "l2": "256 MiB buffer rewritten between timed iterations (outside the event pairs); the path reads 84 ints from constant memory"},
            "clocks": ctx.clocks,
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "roofline": head["roofline"], "cpu_baseline": head["cpu_baseline"],
            "best": head["best"], "wall_s": head["wall_s"], "peaks_measured": ctx.peaks,
            "configs": configs,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, values in ctx.outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), values)
    if ctx.world > 1:
        ctx.comm.close()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
