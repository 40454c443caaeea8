#!/usr/bin/env python3
"""Regenerates the 32x32x32_15096 HM triple from the reference's straight-line programs
(data/32x32x32_15096_{L,R,P}.slp; the .sms are missing upstream, .MISSING_LARGE_BLOBS:1-3) with the
engine's SLP builder (plo_slp_build = matrixBuilder, rule data/Makefile:31-32) and stores the CSR with
rational values in tests/golden/large/32x32x32_15096.npz (committed, 0.2 MB in the encoding of hm.save_large, so that the
tests and bench.py need no copy of the reference).  PLINOPT_REFERENCE names the reference's source tree."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from plinopt_b200 import capi, hm  # noqa: E402

REF = os.environ.get("PLINOPT_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden", "large", "32x32x32_15096.npz")
EXPECT = {"L": (15096, 1024, 1257376), "R": (15096, 1024, 1260960), "P": (1024, 15096, 1259424)}  # SURVEY.md section 0.6


def main():
    arrays = {}
    for x in "LRP":
        text = open(os.path.join(REF, "data", f"32x32x32_15096_{x}.slp")).read()
        rows, cols, ptr, col, num, den = capi.slp_to_csr(text)
        assert (rows, cols, len(col)) == EXPECT[x], (x, rows, cols, len(col))
        arrays.update({f"{x}_shape": np.array([rows, cols]), f"{x}_ptr": ptr, f"{x}_col": col, f"{x}_num": num.astype(np.int32), f"{x}_den": den.astype(np.int32)})
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    hm.save_large(OUT, arrays)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
