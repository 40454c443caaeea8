"""Host-side pieces of the runtime-shape orbit sweep: the fixtures of test_gpu_orbit_any_shape are valid algorithms, the host
decode matches the oracle for shapes with dimensions 1 and 8, and the switch validates its argument without a device."""
import numpy as np
import pytest

import oracle_lib as O
import orbit_any_shape_fixtures as F

FX = F.fixtures()


@pytest.mark.parametrize("name", sorted(FX))
def test_fixture_is_an_algorithm(name):
    T = FX[name]
    assert (len(T[0]), len(T[1]), len(T[2][0])) == (len(T[1]), len(T[2][0]), len(T[0]))  # one rank r for L, R, P
    assert F.is_algorithm(T)


def test_broken_fixture_is_rejected():
    L, R, P = F.naive(2, 3, 4)
    P[0][0] += 1
    assert not F.is_algorithm((L, R, P))


@pytest.mark.parametrize("mkn", [(1, 2, 2), (1, 1, 8), (8, 1, 3), (2, 8, 1), (8, 8, 8), (5, 5, 5)])
@pytest.mark.parametrize("mode", [0, 1])
def test_host_decode_matches_oracle(mkn, mode):
    from plinopt_b200 import capi
    space = capi.orbit_space(*mkn)
    indices = [0, 1, 12345, 2 ** 33 + 17, 2 ** 64 - 1]
    if mode == 0 and space:  # exhaustive codes inside the space
        indices = [0, 1, 4607 % space, space - 1]
    for index in indices:
        got = capi.orbit_decode(*mkn, mode, 0x504C494E4F505431, index)
        ref = O.orbit_decode(*mkn, mode, 0x504C494E4F505431, index)
        assert all(np.array_equal(a, b) for a, b in zip(got, ref))


def test_switch_rejects_other_values():
    from plinopt_b200 import capi
    for bad in (-1, 2, 7):
        with pytest.raises(capi.PloError) as e:
            capi.set_orbit_any_shape(bad)
        assert e.value.code == capi.E_ARG
    capi.set_orbit_any_shape(1)
    capi.set_orbit_any_shape(0)
