"""The checks the host entry points make before any device work, through ctypes: a zero denominator (which a Fraction cannot
carry) is PLO_E_RANGE with the entry point's own name in plo_last_error(); an inner dimension mismatch of the three MMcheckers is
2 with the counts of the input; an outer dimension mismatch is 3 with "<entry point>: outer dimension mismatch"."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
from plinopt_b200 import capi

STRASSEN = O.triple("2x2x2_7_Strassen")
MMCHECKERS = ("plo_mmchecker", "plo_mmchecker_bits", "plo_mmchecker_quad")


def arrays(T, quad):
    """The int64 arrays of a rational triple at the C ABI: (num, den) per matrix, or (an, ad, bn, bd) with zero sqrt(d) parts."""
    out = []
    for M in T:
        num, den = capi._numden(M)
        out += [num, den] + ([np.zeros_like(num), np.ones_like(den)] if quad else [])
    return out


def last_error():
    return capi.lib().plo_last_error().decode()


def mmchecker(name, T, zero_den=False):
    """plo_mmchecker[_bits|_quad] (d = 3) on T: (rc, [nnz, nno], nprimes), nprimes -1 where the entry point has none."""
    quad = name == "plo_mmchecker_quad"
    arrs = arrays(T, quad)
    if zero_den:
        arrs[1][0, 0] = 0
    lead = {"plo_mmchecker": [(C.c_uint64, 0), (C.c_uint64, 1), (C.c_int, 32)],
            "plo_mmchecker_bits": [(C.c_uint64, 0), (C.c_int, 32), (C.c_uint64, 1), (C.c_int, 32)],
            "plo_mmchecker_quad": [(C.c_int64, 3), (C.c_int, 32), (C.c_uint64, 1), (C.c_int, 32)]}[name]
    npr = C.c_int(-1)
    tail = [] if name == "plo_mmchecker" else [C.byref(npr)]
    cnt = np.full(2, 7, dtype=np.uint32)
    f = getattr(capi.lib(), name)
    f.argtypes = [t for t, _ in lead] + [C.c_int] * 6 + [C.c_void_p] * (len(arrs) + 1) + [C.POINTER(C.c_int)] * len(tail)
    dims = [x for M in T for x in (len(M), len(M[0]))]
    rc = f(*(v for _, v in lead), *dims, *(capi._ptr(a) for a in arrs), capi._ptr(cnt), *tail)
    return rc, cnt.tolist(), npr.value


def triple_pass(name, T, zero_den=False, flag=0):
    """plo_negater or plo_rotater on T (outputs shaped as the inputs: square shapes only)."""
    arrs = arrays(T, False)
    if zero_den:
        arrs[3][0, 0] = 0
    outs = [np.zeros_like(a) for a in arrs]
    stats = [capi._ptr(np.zeros(12, dtype=np.uint64))] if name == "plo_negater" else []
    f = getattr(capi.lib(), name)
    f.argtypes = [C.c_int] * 5 + [C.c_void_p] * (12 + len(stats))
    L, R, P = T
    return f(flag, len(L), len(L[0]), len(R[0]), len(P), *(capi._ptr(a) for a in arrs + outs), *stats)


@pytest.mark.parametrize("name", MMCHECKERS)
def test_mmcheckers_refuse_a_zero_denominator(name):
    rc, _, _ = mmchecker(name, STRASSEN, zero_den=True)
    assert rc == capi.E_RANGE
    assert last_error().startswith(name + ": ") and "zero denominator" in last_error()


@pytest.mark.parametrize("name", MMCHECKERS)
def test_mmcheckers_inner_mismatch_reports_the_counts(name):
    L, R, P = STRASSEN
    T = (L, R[:-1], P)
    entries = [v for M in T for row in M for v in row if v != 0]
    rc, cnt, npr = mmchecker(name, T)
    assert rc == 2
    assert cnt == [len(entries), sum(1 for v in entries if abs(v) != 1)]
    assert npr == (-1 if name == "plo_mmchecker" else 0)


@pytest.mark.parametrize("name", ["plo_negater", "plo_rotater"])
def test_triple_passes_refuse_a_zero_denominator(name):
    assert triple_pass(name, STRASSEN, zero_den=True) == capi.E_RANGE
    assert last_error().startswith(name + ": ") and "zero denominator" in last_error()


def test_rotater_outer_mismatch():
    L, R, P = STRASSEN
    assert triple_pass("plo_rotater", (L, [row[:3] for row in R], P)) == 3
    assert last_error() == "plo_rotater: outer dimension mismatch"


@pytest.mark.gpu
def test_orbiters_outer_mismatch():
    """After the device check: 3 and the entry point's name, for every orbiter."""
    L, R, P = STRASSEN
    R3 = [row[:3] for row in R]
    Q = tuple((M, [[0] * len(M[0]) for _ in M]) for M in (L, R3, P))
    calls = {"plo_orbiter": lambda: capi.orbiter(L, R3, P),
             "plo_orbiter_progress": lambda: capi.orbiter_progress(L, R3, P),
             "plo_orbiter_modp": lambda: capi.orbiter_modp(L, R3, P, 513083),
             "plo_orbiter_quad": lambda: capi.orbiter_quad(3, *Q),
             "plo_orbiter_progress_quad": lambda: capi.orbiter_progress_quad(3, *Q)}
    for name, call in calls.items():
        with pytest.raises(capi.PloError) as e:
            call()
        assert e.value.code == 3 and str(e.value).endswith(f"{name}: outer dimension mismatch"), (name, str(e.value))
