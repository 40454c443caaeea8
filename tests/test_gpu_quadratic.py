"""GPU tests of the orbit sweep over Q(sqrt d) (plo_orbit_plan_create_quad, plo_orbit_table_quad, plo_growth_factors_quad) against a
reference built on the oracle: the oracle's decode gives (U, V, W), the exact transform is applied to the rational and the sqrt(d)
part separately (checked against the oracle's orbit_apply on sampled candidates), entries are counted as pairs in Python and G2 is
taken in float64.  nnz / nno exact, G2 within 1e-12 relative."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
from test_quadratic_host import FX, G2_DPS_ACCURATE, rational, scaled_quad

pytestmark = pytest.mark.gpu
SEED = 0x504C494E4F505431
RTOL = 1e-12
P513083 = 513083  # 1013^2 = 3 mod 513083: the rational DPS-accurate file is DPS-accurate over Z/513083Z


def decode_all(mkn, mode, seed, lo, hi):
    U, V, W = zip(*(O.orbit_decode(*mkn, mode, seed, i) for i in range(lo, hi)))
    return (np.array(X, dtype=np.int64) for X in (U, V, W))


def inv(X):
    return np.rint(np.linalg.inv(X.astype(np.float64))).astype(np.int64)


def transform(mkn, part, U, V, W):
    """L.(U^-1 (x) V), R.(V^-T (x) W), (U (x) W^-1).P of one integer part for every candidate: (N, r, m.k), (N, r, k.n), (N, r, m.n)."""
    m, k, n = mkn
    L, R, P = part
    r = L.shape[0]
    A, B, Cm = L.reshape(r, m, k), R.reshape(r, k, n), P.T.reshape(r, m, n)
    A2 = np.einsum("nix,lij,njy->nlxy", inv(U), A, V, optimize=True)
    B2 = np.einsum("nxi,lij,njy->nlxy", inv(V), B, W, optimize=True)
    C2 = np.einsum("nxi,lij,nyj->nlxy", U, Cm, inv(W), optimize=True)
    N = U.shape[0]
    return A2.reshape(N, r, -1), B2.reshape(N, r, -1), C2.reshape(N, r, -1)


def reference(d, T, mode, seed, lo, hi, samples=3):
    """Per-candidate (nnz, nno, g2) over Q(sqrt d); g2 is None for d < 0."""
    mkn, parts, dens = scaled_quad(T)
    U, V, W = decode_all(mkn, mode, seed, lo, hi)
    ta = transform(mkn, parts[0::2], U, V, W)
    tb = transform(mkn, parts[1::2], U, V, W)
    # the transform of each part is the oracle's exact one
    for s in np.linspace(0, hi - lo - 1, samples).astype(int):
        for t, q in ((ta, 0), (tb, 1)):
            got = O.orbit_apply(T[0][q], T[1][q], T[2][q], U[s], V[s], W[s])
            for x, (M, den) in enumerate(zip(got, dens)):
                rows = M if x < 2 else [list(c) for c in zip(*M)]
                assert [[v * den for v in row] for row in rows] == t[x][s].tolist()
    nnz = np.zeros(hi - lo, dtype=np.int64); nno = np.zeros_like(nnz)
    g2 = np.zeros(hi - lo) if d > 0 else None
    norms = []
    for a, b, den in zip(ta, tb, dens):
        nz = (a != 0) | (b != 0)
        nnz += nz.sum(axis=(1, 2))
        nno += (nz & ~((b == 0) & (np.abs(a) == den))).sum(axis=(1, 2))
        if d > 0:
            v = (a + b * np.sqrt(d)) / den
            norms.append(np.sqrt((v * v).sum(axis=2)))
    if d > 0:
        g2 = (norms[0] * norms[1] * norms[2]).sum(axis=1)
    return nnz, nno, g2


def check(ref, got):
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    if ref[2] is None:
        assert got[2] is None
    else:
        np.testing.assert_allclose(got[2], ref[2], rtol=RTOL, atol=0)


def table(d, T, mode, lo, hi, capi, seed=SEED):
    mkn, parts, dens = scaled_quad(T)
    return capi.orbit_table_quad(d, mkn, *parts, dens, mode, seed, lo, hi)


def test_exhaustive_dps_accurate_table(capi):
    d, T = FX["DPS-accurate"]
    check(reference(d, T, 0, SEED, 0, 48 ** 3), table(d, T, 0, 0, 48 ** 3, capi))


@pytest.mark.parametrize("name", sorted(n for n in FX if n != "DPS-accurate"))
def test_philox_tables(capi, name):
    d, T = FX[name]
    lo = 2 ** 33 + 17
    check(reference(d, T, 1, SEED, lo, lo + 2000), table(d, T, 1, lo, lo + 2000, capi))


def residues(M, p):
    return np.array([[(v.numerator % p) * pow(v.denominator % p, -1, p) % p for v in row] for row in M], dtype=np.int32)


@pytest.mark.parametrize("mode,lo,hi", [(0, 0, 48 ** 3), (1, 2 ** 40, 2 ** 40 + 20000)])
def test_a_zero_over_the_field_is_a_zero_modulo_513083(capi, mode, lo, hi):
    """DPS-accurate over Q(sqrt 3) sees at least the nonzeros and non-units that its 1013 image sees modulo 513083."""
    d, T = FX["DPS-accurate"]
    nnz, nno, _ = table(d, T, mode, lo, hi, capi)
    Lp, Rp, Pp = (residues(M, P513083) for M in O.triple("2x2x2_7_DPS-accurate"))
    pnnz, pnno = capi.orbit_table_modp(P513083, (2, 2, 2), Lp, Rp, Pp, mode, SEED, lo, hi)
    assert (nnz >= pnnz).all() and (nno >= pnno).all()


@pytest.mark.parametrize("stem", ["2x2x2_7_Winograd", "3x3x3_23_58", "3x4x7_63_rational"])
def test_zero_sqrt_part_matches_the_rational_path(capi, stem):
    T = O.triple(stem)
    lo, hi = 777, 777 + 3000
    (Li, dl), (Ri, dr), (Pi, dp) = (O.scaled_int(M) for M in T)
    rn, ro, rg = capi.orbit_table(O.LRP2MM(*T), Li.astype(np.int32), Ri.astype(np.int32), Pi.astype(np.int32), (dl, dr, dp), 1, SEED, lo, hi)
    nnz, nno, g2 = table(2, rational(T), 1, lo, hi, capi)
    assert np.array_equal(nnz, rn) and np.array_equal(nno, ro)
    np.testing.assert_allclose(g2, rg, rtol=RTOL, atol=0)


def test_int64_storage_gives_the_same_table(capi):
    """Entries and denominators scaled by 2^32 do not fit int32: the plan keeps int64 words, with the same results."""
    d, T = FX["DPS-accurate"]
    mkn, parts, dens = scaled_quad(T)
    lo, hi = 2 ** 20, 2 ** 20 + 5000
    small = capi.orbit_table_quad(d, mkn, *parts, dens, 1, SEED, lo, hi)
    big = capi.orbit_table_quad(d, mkn, *(p << 32 for p in parts), tuple(x << 32 for x in dens), 1, SEED, lo, hi)
    assert np.array_equal(small[0], big[0]) and np.array_equal(small[1], big[1])
    np.testing.assert_allclose(big[2], small[2], rtol=RTOL, atol=0)


@pytest.mark.parametrize("name,mode", [("DPS-accurate", 0), ("DPS-accurate", 1), ("DPS-accurate_kron_Strassen", 1),
                                       ("3x3x3_23_58_sqrt-1", 1), ("3x4x7_63_rational_sqrt5", 1)])
def test_plan_winner_pack_and_survivors(capi, name, mode):
    d, T = FX[name]
    mkn, parts, dens = scaled_quad(T)
    lo, hi = (0, 48 ** 3) if mode == 0 else (12345, 12345 + 20000)
    nnz, nno, g2 = capi.orbit_table_quad(d, mkn, *parts, dens, mode, SEED, lo, hi)
    idx = np.arange(lo, hi, dtype=np.uint64)
    measures = [capi.MEASURE_NNZ] + ([capi.MEASURE_G2] if d > 0 else [])
    for measure in measures:
        plan = capi.OrbitPlan.quad(d, mkn, *parts, dens, measure, mode, SEED)
        assert (plan.kernel, plan.lanes) == ("orbit_rt_kernel+quad", 1)
        plan.run(lo, hi)
        best = plan.result()
        if measure == capi.MEASURE_NNZ:
            w = int(np.lexsort((nno, nnz))[0])  # lexsort is stable: the lowest index among ties
            assert (best["index"], best["nnz"], best["nno"], best["score"]) == (lo + w, nnz[w], nno[w], float(nnz[w]))
            order = np.lexsort((nno, nnz))
            tn, to = int(nnz[order[len(order) // 50]]), int(nno[order[len(order) // 50]])
            keep = (nnz < tn) | ((nnz == tn) & (nno <= to))
            got = plan.survivors(lo, hi, nnz=tn, nno=to, capacity=16)
        else:
            w = int(np.argmin(g2))
            assert (best["index"], best["nnz"], best["nno"]) == (lo + w, nnz[w], nno[w])
            assert best["score"] == g2[w]
            thr = float(np.quantile(g2, 0.02))
            keep = g2 <= thr
            got = plan.survivors(lo, hi, score=thr, capacity=16)
        assert [g["index"] for g in got] == idx[keep].tolist()
        assert [g["nnz"] for g in got] == nnz[keep].tolist() and [g["nno"] for g in got] == nno[keep].tolist()
        if d > 0:
            assert [g["score"] for g in got] == g2[keep].tolist()
        import torch
        plan.run(lo, hi)
        slots = torch.empty(2 * 4, dtype=torch.int64, device="cuda")
        plan.pack(slots.data_ptr(), 1, 2)
        torch.cuda.synchronize()
        s = slots.cpu().numpy()
        assert (s[:4] == np.iinfo(np.int64).max).all()
        assert s[4].view(np.float64) == best["score"] and (s[5], s[6], s[7]) == (best["index"], best["nnz"], best["nno"])
        plan.close()


def test_growth_factor_of_the_identity_input(capi):
    d, T = FX["DPS-accurate"]
    eye = next(i for i in range(48 ** 3) if all((X == np.eye(2)).all() for X in O.orbit_decode(2, 2, 2, 0, SEED, i)))
    g2 = table(d, T, 0, eye, eye + 1, capi)[2][0]
    assert abs(g2 - G2_DPS_ACCURATE) <= RTOL * G2_DPS_ACCURATE
    assert abs(capi.growth_factors_quad(d, *T)["G2"] - G2_DPS_ACCURATE) <= RTOL * G2_DPS_ACCURATE


def test_limits(capi):
    d, T = FX["3x4x7_63_rational_sqrt2"]
    mkn, parts, dens = scaled_quad(T)
    create = lambda ps, ds=dens, dd=d, measure=capi.MEASURE_NNZ: capi.OrbitPlan.quad(dd, mkn, *ps, ds, measure, 1, SEED)
    create(parts).close()  # 2 x 3843 int32 words fit the constant bank
    wide = [p.copy() for p in parts]
    wide[1][0, 0] = 2 ** 33  # int64 storage: 4 x 3843 words do not
    with pytest.raises(capi.PloError) as e:
        create(wide)
    assert e.value.code == capi.E_SHAPE
    # <8,8,1>, r = 1: a row of 64 entries 2^52 in the sqrt(d) part of L reaches the 2^62 transform bound (128 x 8 x 2^52) while the
    # entries stay below the 2^53 that keeps the bound itself inside int64; one entry more than that is refused on its own
    m8 = (8, 8, 1)
    La, Ra, Pa = np.ones((1, 64), np.int64), np.ones((1, 8), np.int64), np.ones((8, 1), np.int64)
    Z = [np.zeros_like(x) for x in (La, Ra, Pa)]
    plan = lambda lb: capi.OrbitPlan.quad(3, m8, La, lb, Ra, Z[1], Pa, Z[2], (1, 1, 1), capi.MEASURE_NNZ, 1, SEED)
    plan(np.full((1, 64), 2 ** 52 - 2 ** 45, np.int64)).close()
    for lb in (np.full((1, 64), 2 ** 52, np.int64), np.full((1, 64), 2 ** 53, np.int64)):
        with pytest.raises(capi.PloError) as e:
            plan(lb)
        assert e.value.code == capi.E_RANGE
    for dd, measure in ((-2, capi.MEASURE_G2), (16, capi.MEASURE_NNZ)):
        with pytest.raises(capi.PloError) as e:
            create(parts, dd=dd, measure=measure)
        assert e.value.code == capi.E_ARG
    with pytest.raises(capi.PloError) as e:  # no G2 table without a real embedding
        lib = capi.lib()
        f = lib.plo_orbit_table_quad
        g = np.zeros(4)
        ps = [np.ascontiguousarray(p) for p in parts]
        f.argtypes = [C.c_int64] + [C.c_int] * 4 + [C.c_void_p] * 6 + [C.c_int64] * 3 + [C.c_int, C.c_uint64, C.c_uint64, C.c_uint64] + [C.c_void_p] * 3
        capi._check(f(-2, *mkn, ps[0].shape[0], *(p.ctypes.data for p in ps), *dens, 1, SEED, 0, 4, None, None, g.ctypes.data))
    assert e.value.code == capi.E_ARG
