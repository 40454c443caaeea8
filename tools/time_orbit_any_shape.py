#!/usr/bin/env python3
"""Candidates/s of the runtime-shape orbit kernel (plo_set_orbit_any_shape) on shapes without a compiled kernel, of 3x4x7 forced
through it (PLO_ORBIT_RUNTIME_SHAPE) next to the compiled 3x4x7 kernel, and of the CPU oracle on all host cores for the same
inputs.  One JSON line per case, then the card name and power limit of the run:
    python tools/time_orbit_any_shape.py [out.jsonl]"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from plinopt_b200 import capi  # noqa: E402
import oracle_lib as O  # noqa: E402
import orbit_any_shape_fixtures as F  # noqa: E402

SEED = 0x504C494E4F505431


def gpu_rate(T, measure, forced=False, lg=20):
    """Device events around 5 plan runs of 2^lg Philox candidates after 3 warm-up runs."""
    if forced:
        os.environ["PLO_ORBIT_RUNTIME_SHAPE"] = "1"
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, measure, capi.MODE_PHILOX, SEED)
    os.environ.pop("PLO_ORBIT_RUNTIME_SHAPE", None)
    st = torch.cuda.current_stream()
    B = 1 << lg
    for _ in range(3):
        plan.run(0, B, st.cuda_stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for s in range(5):
        plan.run(s * B, (s + 1) * B, st.cuda_stream)
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    kernel = plan.kernel
    plan.close()
    return kernel, B / ms * 1e3


def cpu_rate(T, measure, count):
    t0 = time.perf_counter()
    O.orbit_sweep(*T, measure, 1, SEED, 0, count, table=False)
    return count / (time.perf_counter() - t0)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    capi.set_device(0)
    capi.set_orbit_any_shape(1)
    fx = F.fixtures()
    cases = [("4x7x3", fx["4x7x3_63_rotated"], False, 20000), ("7x3x4", fx["7x3x4_63_rotated"], False, 20000),
             ("2x2x4 Strassen(x)<1,1,2>", fx["2x2x2_7_Strassen_kron_112"], False, 200000), ("5x5x5 naive r=125", fx["naive_5x5x5"], False, 5000),
             ("3x4x7 forced", O.triple("3x4x7_63_rational"), True, 20000), ("3x4x7 compiled", O.triple("3x4x7_63_rational"), False, 0)]
    lines = []
    for name, T, forced, cpu_count in cases:
        for measure, mname in ((capi.MEASURE_NNZ, "nnz"), (capi.MEASURE_G2, "G2")):
            kernel, rate = gpu_rate(T, measure, forced)
            rec = dict(case=name, measure=mname, kernel=kernel, gpu_candidates_per_s=float("%.4g" % rate))
            if cpu_count:
                crate = cpu_rate(T, measure, cpu_count)
                rec.update(cpu_oracle_candidates_per_s=float("%.4g" % crate), cpu_threads=os.cpu_count(), speedup=float("%.4g" % (rate / crate)))
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    card = dict(card=smi.splitlines()[0] if smi else "unknown", torch_device=torch.cuda.get_device_name(0))
    lines.append(card)
    print(json.dumps(card))
    if out:
        with open(out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
