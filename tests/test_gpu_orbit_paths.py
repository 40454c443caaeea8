"""Which sweep kernel a plan launches.  Every expected (kernel, lanes) pair was observed on a B200, not derived from the selection
code: each input below reaches one path of plo_orbit_plan_create (the table-driven 2x2x2 kernels, the four-lane kernels with and
without their three-phase / triangular variants, the plain kernel, the 64-bit kernel, the runtime-shape kernel), so a change to
that code that moves any input to another kernel fails here.  bench.py and profiles/ncu_inputs.json key on these names."""
import numpy as np
import pytest

from plinopt_b200 import hm

pytestmark = pytest.mark.gpu
SEED = 0x504C494E4F505431
G2, NNZ = 3, 0


def triple(stem, scale=1):
    L, R, P = hm.load_fixture(stem)
    (Li, dl), (Ri, dr), (Pi, dp) = (hm.scaled(M, np.int64) for M in (L, R, P))
    return hm.LRP2MM(L, R, P), (Li * scale, Ri, Pi), (dl * scale, dr, dp)


def naive_222():
    """The 8-product definition of 2x2 matrix multiplication: a 2x2x2 triple with r != 7 (the generic (2,2,2) kernels)."""
    L, R, P = np.zeros((8, 4), np.int64), np.zeros((8, 4), np.int64), np.zeros((4, 8), np.int64)
    for l, (i, k, j) in enumerate((i, k, j) for i in range(2) for k in range(2) for j in range(2)):
        L[l, 2 * i + k] = R[l, 2 * k + j] = P[2 * i + j, l] = 1
    return (2, 2, 2), (L, R, P), (1, 1, 1)


CASES = {
    "2x2x2_7_Winograd": lambda: triple("2x2x2_7_Winograd"),
    "3x3x3_23_58": lambda: triple("3x3x3_23_58"),
    "3x4x7_63_rational": lambda: triple("3x4x7_63_rational"),
    # one bound of 128: just outside the 8-bit lanes
    "4x4x4_48_rational": lambda: triple("4x4x4_48_rational"),
    "naive_2x2x2": naive_222,
    # row norms^2 up to 4 . 24^2: the sqrt table holds them all, but it is too large for the shared memory of orbit_sweep8x_kernel
    "2x2x2_7_Winograd_x6": lambda: triple("2x2x2_7_Winograd", 6),
    # row norms^2 up to 4 . 80^2: beyond the 4096 entries of a sqrt table
    "2x2x2_7_Winograd_x20": lambda: triple("2x2x2_7_Winograd", 20),
    # beyond the 8-bit lanes of the four-lane kernels, inside the int32 product bound
    "2x2x2_7_Winograd_x1000": lambda: triple("2x2x2_7_Winograd", 1000),
    "3x3x3_23_58_x1000": lambda: triple("3x3x3_23_58", 1000),
    # common denominators ~10^9: beyond the int32 product bound, the 64-bit kernel
    "2x2x2_7_DPS-integral-12.0662": lambda: triple("2x2x2_7_DPS-integral-12.0662"),
}

EXPECTED = {
    ("2x2x2_7_Winograd", G2): ("orbit_sweep8x_kernel", 4),
    ("2x2x2_7_Winograd", NNZ): ("orbit_sweep2x_kernel", 2),
    ("3x3x3_23_58", G2): ("orbit_sweep8_kernel", 4),
    ("3x3x3_23_58", NNZ): ("orbit_sweepn8_kernel", 4),
    ("3x4x7_63_rational", G2): ("orbit_sweep8_kernel+tri", 4),
    ("3x4x7_63_rational", NNZ): ("orbit_sweepn8_kernel+3phase+tri", 4),
    ("4x4x4_48_rational", G2): ("orbit_sweep_kernel", 2),
    ("4x4x4_48_rational", NNZ): ("orbit_sweep_kernel", 2),
    ("naive_2x2x2", G2): ("orbit_sweep8_kernel", 4),
    ("naive_2x2x2", NNZ): ("orbit_sweepn8_kernel", 4),
    ("2x2x2_7_Winograd_x6", G2): ("orbit_sweep8_kernel", 4),
    ("2x2x2_7_Winograd_x20", G2): ("orbit_sweep8_kernel", 4),
    ("2x2x2_7_Winograd_x1000", G2): ("orbit_sweep_kernel", 2),
    ("2x2x2_7_Winograd_x1000", NNZ): ("orbit_sweep2x_kernel", 2),
    ("3x3x3_23_58_x1000", G2): ("orbit_sweep_kernel", 2),
    ("3x3x3_23_58_x1000", NNZ): ("orbit_sweep_kernel", 2),
    ("2x2x2_7_DPS-integral-12.0662", G2): ("orbit_wide_kernel", 1),
    ("2x2x2_7_DPS-integral-12.0662", NNZ): ("orbit_wide_kernel", 1),
}


def plan(capi, name, measure):
    mkn, (L, R, P), dens = CASES[name]()
    return capi.OrbitPlan(mkn, L.astype(np.int32), R.astype(np.int32), P.astype(np.int32), dens, measure, 1, SEED)


@pytest.mark.parametrize("name,measure", sorted(EXPECTED))
def test_plan_kernel(capi, name, measure):
    pl = plan(capi, name, measure)
    try:
        assert (pl.kernel, pl.lanes) == EXPECTED[(name, measure)]
        pl.run(0, 5000)
        assert pl.result()["index"] is not None
    finally:
        pl.close()


@pytest.mark.parametrize("measure", [G2, NNZ])
def test_runtime_shape_environment_switch(capi, monkeypatch, measure):
    """PLO_ORBIT_RUNTIME_SHAPE sends a compiled shape to the runtime-shape kernel."""
    monkeypatch.setenv("PLO_ORBIT_RUNTIME_SHAPE", "1")
    pl = plan(capi, "3x4x7_63_rational", measure)
    try:
        assert (pl.kernel, pl.lanes) == ("orbit_rt_kernel", 1)
    finally:
        pl.close()


def test_wide_plan_refuses_pack(capi):
    """The 64-bit path picks its winner on the host, so it has no device record to pack."""
    import torch
    pl = plan(capi, "2x2x2_7_DPS-integral-12.0662", G2)
    try:
        pl.run(0, 1000)
        slots = torch.empty(4, dtype=torch.int64, device="cuda")
        with pytest.raises(capi.PloError) as e:
            pl.pack(slots.data_ptr(), 0, 1)
        assert e.value.code == capi.E_SHAPE
    finally:
        pl.close()
