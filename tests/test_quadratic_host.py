"""CPU tests of the orbit sweep over Q(sqrt d): the fixtures over Q(sqrt d) are matrix-multiplication algorithms (exact pair
arithmetic at every pair of unit vectors), the new entry points are exported, refuse fields they do not support, and fail loudly
without a device.  The fixture builders here are shared with tests/test_gpu_quadratic.py.

An entry over Q(sqrt d) is a pair (a, b) of Fractions standing for a + b.sqrt(d); a matrix is a pair (A, B) of lists of rows."""
from fractions import Fraction

import numpy as np
import pytest

import oracle_lib as O
import orbit_any_shape_fixtures as F
from plinopt_b200 import capi

DPS = "2x2x2_7_DPS-accurate"
PLACEHOLDER = 1013  # the rational copy of DPS-accurate writes sqrt(3) as 1013 (valid modulo (1013^2 - 3) / 2 = 513083 only)
G2_DPS_ACCURATE = 12.0660314317802


def zeros_like(M):
    return [[Fraction(0)] * len(M[0]) for _ in M]


def split_placeholder(M):
    """(A, B) with M = A + 1013.B entrywise, every entry of M being q or q.1013 (q rational, written without a factor 1013)."""
    A, B = zeros_like(M), zeros_like(M)
    for i, row in enumerate(M):
        for j, v in enumerate(row):
            if v.numerator % PLACEHOLDER == 0 and v != 0:
                B[i][j] = v / PLACEHOLDER
            else:
                A[i][j] = v
    return A, B


def dps_accurate():
    """DPS-accurate over Q(sqrt 3): the 1013 placeholder lifted to sqrt(3)."""
    return tuple(split_placeholder(M) for M in O.triple(DPS))


def rational(T):
    """A rational triple as a triple over Q(sqrt d) with zero sqrt(d) parts."""
    return tuple((M, zeros_like(M)) for M in T)


def scale_rows(T, d, rows):
    """Row l of L times sqrt(d) and column l of P times sqrt(d)/d for l in `rows`: the products of the algorithm do not change."""
    L, R, P = (([list(r) for r in M], zeros_like(M)) for M in T)
    for l in rows:
        L[1][l], L[0][l] = L[0][l], [Fraction(0)] * len(L[0][l])
        for e in range(len(P[0])):
            P[1][e][l], P[0][e][l] = P[0][e][l] / d, Fraction(0)
    return L, R, P


def kron_rational(Q, T):
    """Q (x) T with Q over Q(sqrt d) and T rational: the Kronecker product of each part with T."""
    (La, Lb), (Ra, Rb), (Pa, Pb) = Q
    A = F.kron((La, Ra, Pa), T)
    B = F.kron((Lb, Rb, Pb), T)
    return tuple(zip(A, B))


def fixtures():
    """name -> (d, triple over Q(sqrt d))."""
    out = {"DPS-accurate": (3, dps_accurate())}
    for stem, rows in (("2x2x2_7_Winograd", (0, 3)), ("3x3x3_23_58", (1, 7, 22)), ("3x4x7_63_rational", (0, 30, 62))):
        for d in (2, 3, 5, -1, -3):
            out[f"{stem}_sqrt{d}"] = (d, scale_rows(O.triple(stem), d, rows))
    out["DPS-accurate_kron_Strassen"] = (3, kron_rational(dps_accurate(), O.triple("2x2x2_7_Strassen")))
    return out


def pmul(x, y, d):
    return (x[0] * y[0] + d * x[1] * y[1], x[0] * y[1] + x[1] * y[0])


def is_algorithm_quad(T, d):
    """Exact check over Q(sqrt d) at every pair of unit vectors (ua, ub): P.((L.ua) o (R.ub)) = vec(ua . ub) with ua an m x k and ub
    a k x n matrix, row-major.  The triple computes a bilinear map, so this proves it is a <m,k,n> algorithm."""
    (La, Lb), (Ra, Rb), (Pa, Pb) = T
    m, k, n = O.LRP2MM(La, Ra, Pa)
    r = len(La)
    for i in range(m * k):
        for j in range(k * n):
            t = [pmul((La[l][i], Lb[l][i]), (Ra[l][j], Rb[l][j]), d) for l in range(r)]
            for e in range(m * n):
                c = (sum(Pa[e][l] * t[l][0] + d * Pb[e][l] * t[l][1] for l in range(r)),
                     sum(Pa[e][l] * t[l][1] + Pb[e][l] * t[l][0] for l in range(r)))
                want = 1 if (i // k == e // n and i % k == j // n and j % n == e % n) else 0
                if c != (want, 0):
                    return False
    return True


def scaled_quad(T):
    """(shape, six int64 arrays La, Lb, Ra, Rb, Pa, Pb, (denL, denR, denP)): one common denominator per matrix over both parts."""
    parts, dens = [], []
    for A, B in T:
        den = O.lcm_den(A + B)
        dens.append(den)
        parts += [np.array([[int(v * den) for v in row] for row in M], dtype=np.int64) for M in (A, B)]
    return O.LRP2MM(T[0][0], T[1][0], T[2][0]), parts, tuple(dens)


def g2_float(T, d):
    """G2 of a triple over Q(sqrt d), d > 0: every entry to a double a + b.sqrt(d) first (growthfactor.cpp:25-28)."""
    s = float(np.sqrt(d))
    L, R, P = (np.array([[float(a) + float(b) * s for a, b in zip(ra, rb)] for ra, rb in zip(*M)]) for M in T)
    return float(sum(np.linalg.norm(L[l]) * np.linalg.norm(R[l]) * np.linalg.norm(P[:, l]) for l in range(L.shape[0])))


FX = fixtures()


def test_dps_accurate_entries_are_rational_or_rational_times_the_placeholder():
    for M in O.triple(DPS):
        A, B = split_placeholder(M)
        for row, ra, rb in zip(M, A, B):
            for v, a, b in zip(row, ra, rb):
                assert a == 0 or b == 0
                assert v == a + PLACEHOLDER * b
                assert v == 0 or (a if a else b).numerator % PLACEHOLDER != 0
    assert any(any(v != 0 for v in row) for _, B in dps_accurate() for row in B)


@pytest.mark.parametrize("name", sorted(FX))
def test_fixture_is_an_algorithm_over_the_field(name):
    d, T = FX[name]
    assert is_algorithm_quad(T, d)


def test_a_wrong_sign_of_sqrt_d_is_not_an_algorithm():
    """Conjugating one entry breaks DPS-accurate over Q(sqrt 3): the exact check above can fail."""
    (La, Lb), R, P = dps_accurate()
    Lb = [list(row) for row in Lb]
    i, j = next((i, j) for i, row in enumerate(Lb) for j, v in enumerate(row) if v != 0)
    Lb[i][j] = -Lb[i][j]
    assert not is_algorithm_quad(((La, Lb), R, P), 3)


def test_dps_accurate_growth_factor_in_float64():
    assert abs(g2_float(dps_accurate(), 3) - G2_DPS_ACCURATE) <= 1e-12 * G2_DPS_ACCURATE


def test_new_symbols_are_exported():
    L = capi.lib()
    for s in ("plo_orbit_plan_create_quad", "plo_orbit_table_quad", "plo_growth_factors_quad"):
        assert s in capi.SYMBOLS and hasattr(L, s)


@pytest.mark.parametrize("d", [0, 1, 4, 9, 1 << 40])
def test_perfect_squares_are_refused(d):
    """X^2 - d with d a perfect square is not irreducible: no field, PLO_E_ARG before any device work."""
    mkn, parts, dens = scaled_quad(FX["DPS-accurate"][1])
    with pytest.raises(capi.PloError) as e:
        capi.OrbitPlan.quad(d, mkn, *parts, dens, capi.MEASURE_NNZ, capi.MODE_PHILOX, 0)
    assert e.value.code == capi.E_ARG
    with pytest.raises(capi.PloError) as e:
        capi.orbit_table_quad(d, mkn, *parts, dens, capi.MODE_PHILOX, 0, 0, 4)
    assert e.value.code == capi.E_ARG


def test_growth_factor_needs_a_real_embedding():
    mkn, parts, dens = scaled_quad(FX["2x2x2_7_Winograd_sqrt-3"][1])
    with pytest.raises(capi.PloError) as e:
        capi.OrbitPlan.quad(-3, mkn, *parts, dens, capi.MEASURE_G2, capi.MODE_PHILOX, 0)
    assert e.value.code == capi.E_ARG
    with pytest.raises(capi.PloError) as e:
        capi.growth_factors_quad(-3, *FX["2x2x2_7_Winograd_sqrt-3"][1])
    assert e.value.code == capi.E_ARG


@pytest.mark.skipif(capi.device_count() > 0, reason="checks the no-device behaviour")
def test_quadratic_entry_points_fail_loudly_without_a_device():
    mkn, parts, dens = scaled_quad(FX["DPS-accurate"][1])
    calls = (lambda: capi.OrbitPlan.quad(3, mkn, *parts, dens, capi.MEASURE_G2, capi.MODE_PHILOX, 0),
             lambda: capi.orbit_table_quad(3, mkn, *parts, dens, capi.MODE_PHILOX, 0, 0, 4),
             lambda: capi.orbit_table_quad(-1, mkn, *parts, dens, capi.MODE_EXHAUSTIVE, 0, 0, 4),
             lambda: capi.growth_factors_quad(3, *FX["DPS-accurate"][1]))
    for call in calls:
        with pytest.raises(capi.PloError) as e:
            call()
        assert e.value.code == capi.E_NODEVICE
