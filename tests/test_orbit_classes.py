"""The fact the 2x2x2 table kernels (orbit_sweep8x_kernel, orbit_sweep2x_kernel) rest on, checked on the CPU oracle over all 48^3
mode-0 candidates: every measure of a candidate (U, V, W) depends only on the class triple (cl(U), cr(V), cr(W)).  For a zoi
matrix M = Pi_P T Pi_Q^T, T = [d0 t; 0 d1], cl(M) = (Q[0], t.d0) and cr(M) = (P[0], t.d1) (zoi2_cl / zoi2_cr in orbit_sweep.cu).
Mode-0 digits of matrix number e: P[0] = e % 2, Q[0] = e / 2 % 2, d0 = e / 4 % 2, d1 = e / 8 % 2 (1: +1, 0: -1), t = e / 16 - 1."""
import numpy as np
import pytest

import oracle_lib as O

SPACE = 48 ** 3


def classes():
    e = np.arange(48)
    P, Q = e % 2, e // 2 % 2
    d0, d1, t = 2 * (e // 4 % 2) - 1, 2 * (e // 8 % 2) - 1, e // 16 - 1
    return 3 * Q + 1 + t * d0, 3 * P + 1 + t * d1


def class_triples():
    cl, cr = classes()
    idx = np.arange(SPACE)
    eu, ev, ew = idx % 48, idx // 48 % 48, idx // (48 * 48)
    return (cl[eu] * 6 + cr[ev]) * 6 + cr[ew]


def spread_within_classes(key, values):
    """max - min of `values` inside every class, and the number of classes."""
    lo = np.full(216, np.inf)
    hi = np.full(216, -np.inf)
    np.minimum.at(lo, key, values)
    np.maximum.at(hi, key, values)
    seen = np.isfinite(lo)
    return (hi - lo)[seen], int(seen.sum())


def test_every_class_has_eight_matrices_per_side():
    cl, cr = classes()
    assert np.bincount(cl, minlength=6).tolist() == [8] * 6 and np.bincount(cr, minlength=6).tolist() == [8] * 6


@pytest.mark.parametrize("stem", ["2x2x2_7_Winograd", "2x2x2_7_Strassen", "2x2x2_7_DPS-evenpow-12.2034", "2x2x2_7_DPS-smallrat-12.2034"])
def test_measures_are_class_invariant(stem):
    L, R, P = O.triple(stem)
    ref = O.orbit_sweep(L, R, P, 3, 0, 0, 0, SPACE)
    key = class_triples()
    for m in ("nnz", "nno"):
        spread, n = spread_within_classes(key, ref[m].astype(np.float64))
        assert n == 216 and spread.max() == 0, m
    g2 = ref["g2"]
    if stem == "2x2x2_7_DPS-smallrat-12.2034":
        # the oracle converts every rational entry to a double first: class-invariant up to rounding
        spread, _ = spread_within_classes(key, g2)
        assert spread.max() <= 1e-15 * g2.max()
    else:
        bits = g2.view(np.int64)
        for c in range(216):
            assert np.unique(bits[key == c]).size == 1
