"""GPU parity of the orbit sweep on triples beyond the constant bank: with plo_set_orbit_any_shape(1), L | R | P^T of more than 12000
ints is read from device memory (orbit_rt_kernel+global).  Against the CPU oracle with the rules of test_gpu_orbit_any_shape: nnz /
nno / index exact, G2 bit-exact for integer triples, within 1e-12 relative otherwise; and against the constant-bank kernel on the
same triple padded with zero rows."""
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import oracle_lib as O
import orbit_any_shape_fixtures as F
from plinopt_b200 import hm
from test_gpu_orbit_any_shape import check_table, check_winners, residues
from test_gpu_quadratic import check, reference
from test_orbit_large_host import dps_accurate_x_23_58, fixtures
from test_quadratic_host import FX as QFX, scaled_quad

pytestmark = pytest.mark.gpu
SEED = 0x504C494E4F505431
RTOL = 1e-12
BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bin")
NAMES = ["Strassen_x_3x3x3_23_58", "3x3x6_40_x_naive_221", "naive_7x7x7", "Winograd_x_4x4x4_48_rational", "4x4x4_49_156_x_Strassen"]
COUNT = {"naive_7x7x7": 400, "Winograd_x_4x4x4_48_rational": 300, "4x4x4_49_156_x_Strassen": 300}
S666 = "Strassen_x_3x3x3_23_58"


@pytest.fixture(scope="module", autouse=True)
def any_shape(capi):
    capi.set_orbit_any_shape(1)
    yield
    capi.set_orbit_any_shape(0)


def pad(T, r):
    """T with zero rows of L and R and zero columns of P up to rank r: the same algorithm, a longer triple."""
    L, R, P = T
    extra = r - len(L)
    return ([list(x) for x in L] + [[Fraction(0)] * len(L[0]) for _ in range(extra)],
            [list(x) for x in R] + [[Fraction(0)] * len(R[0]) for _ in range(extra)],
            [list(x) + [Fraction(0)] * extra for x in P])


@pytest.mark.parametrize("name", NAMES)
def test_philox_tables_and_winners(capi, name):
    T = fixtures()[name]
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    lo = 2 ** 33 + 17
    hi = lo + COUNT.get(name, 1000)
    ref = O.orbit_sweep(*T, 3, 1, SEED, lo, hi)
    check_table(ref, *capi.orbit_table(mkn, Li, Ri, Pi, dens, 1, SEED, lo, hi), dens == (1, 1, 1))
    got0 = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, 0, 1, SEED, lo, hi)
    got3 = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, 3, 1, SEED, lo, hi)
    check_winners(T, got0, got3, 1, SEED, lo, hi, ref)
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, 0, 1, SEED)
    assert (plan.kernel, plan.lanes) == ("orbit_rt_kernel+global", 1)
    plan.close()


def test_int64_entry_points(capi):
    T = fixtures()[S666]
    mkn, (Li, Ri, Pi), dens = F.scaled(T, np.int64)
    lo = 2 ** 33 + 5
    hi = lo + 1000
    ref = O.orbit_sweep(*T, 3, 1, SEED, lo, hi)
    check_table(ref, *capi.orbit_table64(mkn, Li, Ri, Pi, dens, 1, SEED, lo, hi), False)
    got0 = capi.orbit_sweep64(mkn, Li, Ri, Pi, dens, 0, 1, SEED, lo, hi)
    got3 = capi.orbit_sweep64(mkn, Li, Ri, Pi, dens, 3, 1, SEED, lo, hi)
    check_winners(T, got0, got3, 1, SEED, lo, hi, ref)


@pytest.mark.parametrize("p", [3, 513083, 2 ** 31 - 1])
def test_modp(capi, p):
    T = fixtures()[S666]
    mkn = O.LRP2MM(*T)
    Lr, Rr, Pr = (residues(M, p) for M in T)
    lo = 2 ** 33 + 99
    hi = lo + 1000
    ref = O.orbit_sweep(*T, 0, 1, SEED, lo, hi, p=p)
    nnz, nno = capi.orbit_table_modp(p, mkn, Lr, Rr, Pr, 1, SEED, lo, hi)
    assert np.array_equal(nnz, ref["nnz"]) and np.array_equal(nno, ref["nno"])
    got = capi.orbit_sweep(mkn, Lr, Rr, Pr, (1, 1, 1), 0, 1, SEED, lo, hi, p=p)
    assert (got["index"], got["nnz"], got["nno"]) == ref["best"][:3]


def test_quadratic_table_winners_and_survivors(capi):
    d, T = dps_accurate_x_23_58()
    mkn, parts, dens = scaled_quad(T)
    lo, hi = 12345, 12345 + 1000
    nnz, nno, g2 = capi.orbit_table_quad(d, mkn, *parts, dens, 1, SEED, lo, hi)
    check(reference(d, T, 1, SEED, lo, hi), (nnz, nno, g2))
    idx = np.arange(lo, hi, dtype=np.uint64)
    for measure in (capi.MEASURE_NNZ, capi.MEASURE_G2):
        plan = capi.OrbitPlan.quad(d, mkn, *parts, dens, measure, 1, SEED)
        assert (plan.kernel, plan.lanes) == ("orbit_rt_kernel+quad+global", 1)
        plan.run(lo, hi)
        best = plan.result()
        if measure == capi.MEASURE_NNZ:
            w = int(np.lexsort((nno, nnz))[0])
            assert (best["index"], best["nnz"], best["nno"], best["score"]) == (lo + w, nnz[w], nno[w], float(nnz[w]))
            order = np.lexsort((nno, nnz))
            tn, to = int(nnz[order[len(order) // 50]]), int(nno[order[len(order) // 50]])
            keep = (nnz < tn) | ((nnz == tn) & (nno <= to))
            got = plan.survivors(lo, hi, nnz=tn, nno=to, capacity=4)
        else:
            w = int(np.argmin(g2))
            assert (best["index"], best["nnz"], best["nno"], best["score"]) == (lo + w, nnz[w], nno[w], g2[w])
            thr = float(np.quantile(g2, 0.05))
            keep = g2 <= thr
            got = plan.survivors(lo, hi, score=thr, capacity=4)
        assert [g["index"] for g in got] == idx[keep].tolist()
        assert [g["nnz"] for g in got] == nnz[keep].tolist() and [g["nno"] for g in got] == nno[keep].tolist()
        assert [g["score"] for g in got] == g2[keep].tolist()
        plan.close()


def test_quadratic_int64_storage_runs_beyond_the_bank(capi):
    """3x4x7_63_rational over Q(sqrt 2) scaled by 2^32: int64 storage, 4 x 3843 words, refused with the switch off
    (test_gpu_quadratic::test_limits); with it on, the same table as the int32 storage in the constant bank."""
    d, T = QFX["3x4x7_63_rational_sqrt2"]
    mkn, parts, dens = scaled_quad(T)
    lo, hi = 2 ** 20, 2 ** 20 + 2000
    small = capi.orbit_table_quad(d, mkn, *parts, dens, 1, SEED, lo, hi)
    wide, wide_dens = [p << 32 for p in parts], tuple(x << 32 for x in dens)
    big = capi.orbit_table_quad(d, mkn, *wide, wide_dens, 1, SEED, lo, hi)
    assert np.array_equal(small[0], big[0]) and np.array_equal(small[1], big[1])
    np.testing.assert_allclose(big[2], small[2], rtol=RTOL, atol=0)
    kernels = []
    for ps, ds in ((parts, dens), (wide, wide_dens)):
        plan = capi.OrbitPlan.quad(d, mkn, *ps, ds, capi.MEASURE_NNZ, 1, SEED)
        kernels.append(plan.kernel)
        plan.close()
    assert kernels == ["orbit_rt_kernel+quad", "orbit_rt_kernel+quad+global"]


def test_entry_points_agree(capi):
    T = fixtures()[S666]
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    lo, hi = 1000, 1000 + 4000
    for measure in (0, 3):
        whole = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, measure, 1, SEED, lo, hi)
        cuts = [lo, lo + 1, lo + 1234, lo + 2000, hi]
        parts = [capi.orbit_sweep(mkn, Li, Ri, Pi, dens, measure, 1, SEED, a, b) for a, b in zip(cuts, cuts[1:])]
        key = (lambda g: (g["nnz"], g["nno"], g["index"])) if measure == 0 else (lambda g: (g["score"], g["index"]))
        assert min(parts, key=key) == whole
        assert capi.orbit_sweep_devices(capi.device_count(), mkn, Li, Ri, Pi, dens, measure, 1, SEED, lo, hi) == whole
    # survivors, both measures, with the capacity protocol
    lo, count = 12345, 1001
    ref = O.orbit_sweep(*T, 3, 1, SEED, lo, lo + count)
    idx = np.arange(lo, lo + count, dtype=np.uint64)
    order = np.lexsort((ref["nno"], ref["nnz"]))
    tn, to = int(ref["nnz"][order[count // 50]]), int(ref["nno"][order[count // 50]])
    keep = (ref["nnz"] < tn) | ((ref["nnz"] == tn) & (ref["nno"] <= to))
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, capi.MEASURE_NNZ, 1, SEED)
    got = plan.survivors(lo, lo + count, nnz=tn, nno=to, capacity=4)
    assert [g["index"] for g in got] == idx[keep].tolist()
    assert [g["nnz"] for g in got] == ref["nnz"][keep].tolist() and [g["nno"] for g in got] == ref["nno"][keep].tolist()
    assert [g["score"] for g in got] == ref["g2"][keep].tolist()
    plan.close()
    thr = float(np.quantile(ref["g2"], 0.05))
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, capi.MEASURE_G2, 1, SEED)
    got = plan.survivors(lo, lo + count, score=thr, capacity=4)
    assert [g["index"] for g in got] == idx[ref["g2"] <= thr].tolist()
    # plan.pack: the winner lands in the plan's device record and from there in its slot
    import torch
    plan.run(lo, lo + count)
    best = plan.result()
    assert best["index"] == lo + int(np.argmin(ref["g2"])) and best["score"] == ref["g2"].min()
    slots = torch.empty(3 * 4, dtype=torch.int64, device="cuda")
    plan.pack(slots.data_ptr(), 1, 3)
    torch.cuda.synchronize()
    s = slots.cpu().numpy()
    big = np.iinfo(np.int64).max
    assert (s[[0, 1, 2, 3, 8, 9, 10, 11]] == big).all()
    assert s[4].view(np.float64) == best["score"] and (s[5], s[6], s[7]) == (best["index"], best["nnz"], best["nno"])
    plan.close()


def test_global_and_bank_plans_on_two_streams(capi):
    """A device-memory plan and a constant-bank plan alternated on two non-blocking streams give their single-stream answers:
    the pointer slot and the bank are re-written under the same event guard."""
    import torch
    torch.cuda.set_device(0)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    big_mkn, big_ints, big_dens = F.scaled(fixtures()[S666])
    small_mkn, small_ints, small_dens = F.scaled(O.triple("3x3x3_23_58"))
    plans = [capi.OrbitPlan(big_mkn, *big_ints, big_dens, capi.MEASURE_G2, capi.MODE_PHILOX, SEED),
             capi.OrbitPlan(small_mkn, *small_ints, small_dens, capi.MEASURE_NNZ, capi.MODE_PHILOX, SEED)]
    assert plans[0].kernel == "orbit_rt_kernel+global" and "global" not in plans[1].kernel
    ranges = [(0, 1 << 14), (5, (1 << 18) + 5)]
    expect = []
    for pl, (lo, hi) in zip(plans, ranges):
        pl.run(lo, hi, 0)
        expect.append(pl.result(0))
    for _ in range(10):
        plans[0].run(*ranges[0], s1.cuda_stream)
        plans[1].run(*ranges[1], s2.cuda_stream)
    got = [plans[0].result(s1.cuda_stream), plans[1].result(s2.cuda_stream)]
    assert got == expect
    for pl in plans:
        pl.close()


def _padded_equal(capi, T, r, mode, seed, lo, hi):
    """Tables of T (constant bank) and of T padded to rank r (device memory) are bit-identical, and so are both winners."""
    out = []
    for X in (T, pad(T, r)):
        mkn, ints, dens = F.scaled(X)
        out.append((capi.orbit_table(mkn, *ints, dens, mode, seed, lo, hi),
                    [capi.orbit_sweep(mkn, *ints, dens, ms, mode, seed, lo, hi) for ms in (0, 3)],
                    capi.OrbitPlan(mkn, *ints, dens, 0, mode, seed).kernel))
    (t0, w0, k0), (t1, w1, k1) = out
    assert all(np.array_equal(a, b) for a, b in zip(t0, t1))
    assert w0 == w1
    assert k0 != k1 and k1 == "orbit_rt_kernel+global"
    return t0


@pytest.mark.parametrize("name,r", [("4x7x3_63_rotated", 4 * 63), ("2x2x2_7_Strassen_kron_112", 640)])
def test_zero_rows_give_the_same_table_from_either_source(capi, name, r):
    T = F.fixtures()[name]
    lo = 2 ** 33 + 17
    _padded_equal(capi, T, r, 1, SEED, lo, lo + 20000)


def test_zero_rows_winograd_exhaustive(capi):
    """Winograd padded to r = 1001 (12012 ints) over all 48^3 candidates: the oracle's exhaustive table of plain Winograd."""
    T = O.triple("2x2x2_7_Winograd")
    nnz, nno, g2 = _padded_equal(capi, T, 1001, 0, 0, 0, 48 ** 3)
    check_table(O.orbit_sweep(*T, 3, 0, 0, 0, 48 ** 3), nnz, nno, g2, True)


def test_limits(capi):
    """Beyond 2^24 ints of L | R | P^T: PLO_E_SHAPE with its own message.  With the switch off nothing changes: a compiled shape
    beyond the bank gets the bank's message, a shape without a compiled kernel the shape's."""
    r = (1 << 24) // (3 * 64) + 1
    Z = (np.zeros((r, 64), np.int32), np.zeros((r, 64), np.int32), np.zeros((64, r), np.int32))
    with pytest.raises(capi.PloError) as e:
        capi.OrbitPlan((8, 8, 8), *Z, (1, 1, 1), 0, 1, SEED)
    assert e.value.code == capi.E_SHAPE and "a triple in device memory holds at most 16777216" in str(e.value)
    T = pad(O.triple("2x2x2_7_Winograd"), 1001)
    mkn, ints, dens = F.scaled(T)
    modp = [residues(M, 513083) for M in T]
    capi.set_orbit_any_shape(0)
    try:
        for call in (lambda: capi.OrbitPlan(mkn, *ints, dens, 0, 1, SEED), lambda: capi.orbit_sweep(mkn, *ints, dens, 0, 1, SEED, 0, 10),
                     lambda: capi.orbit_table64(mkn, *(x.astype(np.int64) for x in ints), dens, 1, SEED, 0, 10),
                     lambda: capi.orbit_table_modp(513083, mkn, *modp, 1, SEED, 0, 10)):
            with pytest.raises(capi.PloError) as e:
                call()
            assert e.value.code == capi.E_SHAPE and "the bank holds 12000" in str(e.value)
        mkn, ints, dens = F.scaled(fixtures()[S666])
        with pytest.raises(capi.PloError) as e:
            capi.OrbitPlan(mkn, *ints, dens, 0, 1, SEED)
        assert e.value.code == capi.E_SHAPE and "not compiled in" in str(e.value)
    finally:
        capi.set_orbit_any_shape(1)


def test_orbiter_cli(capi, tmp_path):
    files = []
    for x, M in zip("LRP", fixtures()[S666]):
        p = tmp_path / f"s666_{x}.sms"
        hm.write_sms(M, str(p))
        files.append(str(p))
    outs = [f.replace(".sms", ".nnz.sms") for f in files]
    run = lambda extra: subprocess.run([os.path.join(BIN, "orbiter")] + extra + ["-O", "2000", "--seed", "5"] + files, capture_output=True, text=True, timeout=600)
    p = run(["--any-shape"])
    assert p.returncode == 0, p.stderr
    if any(os.path.exists(o) for o in outs):
        q = subprocess.run([os.path.join(BIN, "MMchecker")] + outs, capture_output=True, text=True, timeout=600)
        assert q.returncode == 0 and "SUCCESS: correct 6x6x6" in q.stderr
        for o in outs:
            os.remove(o)
    p = run([])
    assert p.returncode != 0 and "not compiled in" in p.stderr
    assert not any(os.path.exists(o) for o in outs)
