#!/usr/bin/env python3
"""Candidates/s of the runtime-shape orbit kernel on triples beyond the constant bank (L | R | P^T from device memory,
orbit_rt_kernel+global), both measures, and the per-row A/B of the two triple sources: 4x7x3_63_rotated from the constant bank
against the same triple padded with zero rows to 4 x 63 from device memory (candidates x rows per second; the kernel's work per
row does not depend on the entries).  One JSON line per case, then the card name, power limit and maximum SM clock of the run:
    python tools/time_orbit_large.py [out.jsonl]      (profiles/orbit_large_r01.jsonl is one such run)"""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from plinopt_b200 import capi  # noqa: E402
import oracle_lib as O  # noqa: E402
import orbit_any_shape_fixtures as F  # noqa: E402
from test_gpu_orbit_large import pad  # noqa: E402
from test_orbit_large_host import dps_accurate_x_23_58, fixtures  # noqa: E402
from test_quadratic_host import scaled_quad  # noqa: E402

SEED = 0x504C494E4F505431


def timed(plan, lg):
    """Device events around 5 plan runs of 2^lg Philox candidates after 3 warm-up runs: candidates/s."""
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
    return B / (e0.elapsed_time(e1) / 5) * 1e3


def rational_plan(T, measure):
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    return capi.OrbitPlan(mkn, Li, Ri, Pi, dens, measure, capi.MODE_PHILOX, SEED)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    capi.set_device(0)
    capi.set_orbit_any_shape(1)
    fx = fixtures()
    d, Q = dps_accurate_x_23_58()
    qmkn, qparts, qdens = scaled_quad(Q)
    cases = [("<6,6,6> Strassen (x) 3x3x3_23_58, r=161", lambda ms: rational_plan(fx["Strassen_x_3x3x3_23_58"], ms), 161),
             ("<7,7,7> naive, r=343", lambda ms: rational_plan(fx["naive_7x7x7"], ms), 343),
             ("<8,8,8> Winograd (x) 4x4x4_48_rational, r=336", lambda ms: rational_plan(fx["Winograd_x_4x4x4_48_rational"], ms), 336),
             ("<6,6,6> DPS-accurate (x) 3x3x3_23_58 over Q(sqrt 3), r=161",
              lambda ms: capi.OrbitPlan.quad(d, qmkn, *qparts, qdens, ms, capi.MODE_PHILOX, SEED), 161)]
    rotated = F.fixtures()["4x7x3_63_rotated"]
    ab = [("per-row A/B: 4x7x3_63_rotated, constant bank, r=63", lambda ms: rational_plan(rotated, ms), 63),
          ("per-row A/B: 4x7x3_63_rotated padded, device memory, r=252", lambda ms: rational_plan(pad(rotated, 4 * 63), ms), 252)]
    lines = []
    for name, make, rows in cases + ab:
        for measure, mname in ((capi.MEASURE_NNZ, "nnz"), (capi.MEASURE_G2, "G2")):
            plan = make(measure)
            rate = timed(plan, 20)
            rec = dict(case=name, measure=mname, kernel=plan.kernel, rows=rows, gpu_candidates_per_s=float("%.4g" % rate),
                       candidate_rows_per_s=float("%.4g" % (rate * rows)))
            plan.close()
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
