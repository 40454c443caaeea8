"""The 2x2x2 r = 7 table kernels score every candidate from per-class-pair records (orbit_sweep8x_kernel: growth factor,
orbit_sweep2x_kernel: sparsity).  Survivors at EVERY distinct key value of the oracle's per-candidate table must be exactly the
candidates the table keeps at that threshold: this pins the key of every candidate, not only the winner's, in both numberings."""
import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu
SEED = 0x504C494E4F505431
G2, NNZ = 3, 0
KERNEL = {G2: "orbit_sweep8x_kernel", NNZ: "orbit_sweep2x_kernel"}
RANGES = {0: (0, 48 ** 3), 1: (2 ** 33 + 5, 2 ** 33 + 5 + (1 << 20))}  # mode 0: the whole orbit; mode 1: 2^20 Philox candidates


def ints(stem):
    L, R, P = O.triple(stem)
    (Li, dl), (Ri, dr), (Pi, dp) = O.scaled_int(L), O.scaled_int(R), O.scaled_int(P)
    return (L, R, P), O.LRP2MM(L, R, P), (Li.astype(np.int32), Ri.astype(np.int32), Pi.astype(np.int32)), (dl, dr, dp)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("measure", [G2, NNZ])
@pytest.mark.parametrize("stem", ["2x2x2_7_Winograd", "2x2x2_7_Strassen"])
def test_survivors_at_every_key_value(capi, stem, measure, mode):
    (L, R, P), mkn, (Li, Ri, Pi), dens = ints(stem)
    lo, hi = RANGES[mode]
    ref = O.orbit_sweep(L, R, P, 3, mode, SEED if mode else 0, lo, hi)
    idx = np.arange(lo, hi, dtype=np.uint64)
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, measure, mode, SEED)
    try:
        assert plan.kernel == KERNEL[measure]
        if measure == G2:
            values = np.unique(ref["g2"])
            assert stem != "2x2x2_7_Winograd" or values.size == 34
            cases = [(dict(score=float(v)), ref["g2"] <= v) for v in values]
        else:
            key = (ref["nnz"].astype(np.uint64) << np.uint64(32)) | ref["nno"].astype(np.uint64)
            cases = [(dict(nnz=int(k >> np.uint64(32)), nno=int(k & np.uint64(0xFFFFFFFF))), key <= k) for k in np.unique(key)]
        for thr, keep in cases:
            cnt, got = plan.survivors_array(lo, hi, capacity=hi - lo, **thr)
            assert cnt == int(keep.sum()) and np.array_equal(got["index"], idx[keep]), thr
    finally:
        plan.close()
