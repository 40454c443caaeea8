"""Host side of the orbit sweep on triples beyond the constant bank (L | R | P^T over 12000 ints, read from device memory with
plo_set_orbit_any_shape(1)): the large fixtures of tests/test_gpu_orbit_large.py are matrix-multiplication algorithms.  The fixture
builders here are shared with that file."""
import functools

import pytest

import oracle_lib as O
import orbit_any_shape_fixtures as F
from test_quadratic_host import dps_accurate, is_algorithm_quad, kron_rational

BANK_INTS = 12000  # the constant bank's share for L | R | P^T


@functools.lru_cache(maxsize=None)
def fixtures():
    """name -> rational triple; none of them fits the constant bank."""
    return {
        "Strassen_x_3x3x3_23_58": F.kron(O.triple("2x2x2_7_Strassen"), O.triple("3x3x3_23_58")),
        "3x3x6_40_x_naive_221": F.kron(O.triple("3x3x6_40"), F.naive(2, 2, 1)),
        "naive_7x7x7": F.naive(7, 7, 7),
        "Winograd_x_4x4x4_48_rational": F.kron(O.triple("2x2x2_7_Winograd"), O.triple("4x4x4_48_rational")),
        "4x4x4_49_156_x_Strassen": F.kron(O.triple("4x4x4_49_156"), O.triple("2x2x2_7_Strassen")),
    }


SHAPES = {"Strassen_x_3x3x3_23_58": ((6, 6, 6), 161), "3x3x6_40_x_naive_221": ((6, 6, 6), 160), "naive_7x7x7": ((7, 7, 7), 343),
          "Winograd_x_4x4x4_48_rational": ((8, 8, 8), 336), "4x4x4_49_156_x_Strassen": ((8, 8, 8), 343)}


@functools.lru_cache(maxsize=None)
def dps_accurate_x_23_58():
    """(d, triple over Q(sqrt 3)): DPS-accurate (x) 3x3x3_23_58, <6,6,6> of rank 161, both parts 2 x 17388 ints."""
    return 3, kron_rational(dps_accurate(), O.triple("3x3x3_23_58"))


def ints(mkn, r):
    m, k, n = mkn
    return r * (m * k + k * n + m * n)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_fixture_is_an_algorithm_beyond_the_bank(name):
    T = fixtures()[name]
    mkn, r = SHAPES[name]
    assert O.LRP2MM(*T) == mkn and len(T[0]) == r
    assert ints(mkn, r) > BANK_INTS
    assert F.is_algorithm(T)


def test_quadratic_fixture_is_an_algorithm_beyond_the_bank():
    d, T = dps_accurate_x_23_58()
    (La, _), (Ra, _), (Pa, _) = T
    assert O.LRP2MM(La, Ra, Pa) == (6, 6, 6) and len(La) == 161
    assert 2 * ints((6, 6, 6), 161) > BANK_INTS
    assert is_algorithm_quad(T, d)
