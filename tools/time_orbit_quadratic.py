#!/usr/bin/env python3
"""Candidates/s of the orbit sweep over Q(sqrt d) (plo_orbit_plan_create_quad) on DPS-accurate over Q(sqrt 3) (2x2x2, r = 7) and on
DPS-accurate (x) Strassen (<4,4,4>, r = 49), next to the rational runtime-shape kernel on the same rational parts (forced through it
with PLO_ORBIT_RUNTIME_SHAPE: both shapes have compiled kernels).  One JSON line per case, then the card name and power limit:
    python tools/time_orbit_quadratic.py [out.jsonl]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from plinopt_b200 import capi  # noqa: E402
from test_quadratic_host import FX, scaled_quad  # noqa: E402

SEED = 0x504C494E4F505431


def timed(plan, lg):
    """Device events around 5 plan runs of 2^lg Philox candidates after 3 warm-up runs."""
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
    rate = B / (e0.elapsed_time(e1) / 5) * 1e3
    kernel = plan.kernel
    plan.close()
    return kernel, rate


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    capi.set_device(0)
    lines = []
    for name, lg in (("DPS-accurate", 24), ("DPS-accurate_kron_Strassen", 20)):
        d, T = FX[name]
        mkn, parts, dens = scaled_quad(T)
        for measure, mname in ((capi.MEASURE_NNZ, "nnz"), (capi.MEASURE_G2, "G2")):
            kq, rq = timed(capi.OrbitPlan.quad(d, mkn, *parts, dens, measure, capi.MODE_PHILOX, SEED), lg)
            os.environ["PLO_ORBIT_RUNTIME_SHAPE"] = "1"
            rat = [p.astype(np.int32) for p in parts[0::2]]
            plan = capi.OrbitPlan(mkn, *rat, dens, measure, capi.MODE_PHILOX, SEED)
            os.environ.pop("PLO_ORBIT_RUNTIME_SHAPE", None)
            kr, rr = timed(plan, lg)
            rec = dict(case=f"{name} over Q(sqrt {d})", shape="%dx%dx%d" % mkn, r=int(parts[0].shape[0]), measure=mname, quad_kernel=kq,
                       quad_candidates_per_s=float("%.4g" % rq), rational_kernel=kr, rational_part_candidates_per_s=float("%.4g" % rr),
                       ratio=float("%.3g" % (rq / rr)))
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
