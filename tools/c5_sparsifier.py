#!/usr/bin/env python3
"""blockSparsifier on column blocks of the C5 matrix (32x32x32_15096_L, 15096 x 1024, regenerated from the reference's .slp):
    python tools/c5_sparsifier.py [ncols=16] [q=2147483647] [c=5]
runs plo_sparsifier on the first `ncols` columns (ncols/4 independent column blocks, TM = 4 x 15096 each: the wide tiled search kernels)
and reports time, non-zeroes before/after and the reference's own check M == Res.CoB (bin/FDT.sh)."""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from plinopt_b200 import capi, hm  # noqa: E402

ncols = int(sys.argv[1]) if len(sys.argv) > 1 else 16
q = int(sys.argv[2]) if len(sys.argv) > 2 else 2147483647
c = int(sys.argv[3]) if len(sys.argv) > 3 else 5
z = hm.load_large()
rows, cols = (int(v) for v in z["L_shape"])
ptr, col, num, den = z["L_ptr"], z["L_col"], z["L_num"].astype(np.int64), z["L_den"].astype(np.int64)
N = np.zeros((rows, ncols), dtype=np.int64); D = np.ones((rows, ncols), dtype=np.int64)
ri = np.repeat(np.arange(rows), np.diff(ptr))
sel = col < ncols
N[ri[sel], col[sel]] = num[sel]; D[ri[sel], col[sel]] = den[sel]
import ctypes as C
cn = np.zeros((ncols, ncols), dtype=np.int64); cd = np.ones((ncols, ncols), dtype=np.int64)
rn = np.zeros((rows, ncols), dtype=np.int64); rd = np.ones((rows, ncols), dtype=np.int64)
ok = C.c_int(0)
stats = np.zeros(3, dtype=np.uint64)
capi.set_device(0)
f = capi.lib().plo_sparsifier
f.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.POINTER(C.c_int), C.c_void_p, C.c_int]
t0 = time.perf_counter()
rc = f(q, rows, ncols, capi._ptr(N), capi._ptr(D), 4, c, 1, capi._ptr(cn), capi._ptr(cd), capi._ptr(rn), capi._ptr(rd), C.byref(ok), capi._ptr(stats), -1)
dt = time.perf_counter() - t0
print(json.dumps({"case": f"32x32x32_15096_L[:, :{ncols}] -q {q} -c {c}", "rc": rc, "error": capi.lib().plo_last_error().decode() if rc else None, "seconds": dt,
                  "nnz_before": int(np.count_nonzero(N)), "nnz_res": int(np.count_nonzero(rn)), "consistent": bool(ok.value),
                  "candidates": int(stats[0]), "device_round_trips": int(stats[1]), "fallbacks": int(stats[2])}))
