"""GPU parity of the runtime-shape orbit kernels (plo_set_orbit_any_shape) against the CPU oracle on shapes without a compiled
kernel, and against the compiled kernels on the shipped shapes (PLO_ORBIT_RUNTIME_SHAPE).  nnz / nno / index exact; G2 bit-exact
for integer triples, within 1e-12 relative for rational ones."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
import orbit_any_shape_fixtures as F
from plinopt_b200 import hm

pytestmark = pytest.mark.gpu
SEED = 0x504C494E4F505431
RTOL = 1e-12
BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bin")
FX = F.fixtures()
BIG = "2x2x2_7_DPS-intermediate-12.0695_kron_112"  # common denominator 1e11: the int64 entry points
INT32 = [name for name in FX if name != BIG]
COUNT = {"naive_5x5x5": 300, "4x7x3_63_rotated": 600, "7x3x4_63_rotated": 600}


@pytest.fixture(autouse=True)
def any_shape(capi):
    capi.set_orbit_any_shape(1)
    yield
    capi.set_orbit_any_shape(0)
    os.environ.pop("PLO_ORBIT_RUNTIME_SHAPE", None)


def check_table(ref, nnz, nno, g2, integer):
    assert np.array_equal(nnz, ref["nnz"]) and np.array_equal(nno, ref["nno"])
    np.testing.assert_allclose(g2, ref["g2"], rtol=RTOL, atol=0)
    if integer:
        assert np.array_equal(g2, ref["g2"])


def check_winners(T, got0, got3, mode, seed, lo, hi, ref):
    ref0 = O.orbit_sweep(*T, 0, mode, seed, lo, hi, table=False)["best"]
    assert (got0["index"], got0["nnz"], got0["nno"]) == ref0[:3]
    gmin = ref["g2"].min()
    assert abs(got3["score"] - gmin) <= RTOL * gmin
    assert abs(ref["g2"][got3["index"] - lo] - got3["score"]) <= RTOL * gmin


def residues(M, p):
    return np.array([[(v.numerator % p) * pow(v.denominator % p, -1, p) % p for v in row] for row in M], dtype=np.int32)


@pytest.mark.parametrize("name", INT32)
def test_philox_tables_and_winners(capi, name):
    T = FX[name]
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    lo = 2 ** 33 + 17
    hi = lo + COUNT.get(name, 1500)
    ref = O.orbit_sweep(*T, 3, 1, SEED, lo, hi)
    check_table(ref, *capi.orbit_table(mkn, Li, Ri, Pi, dens, 1, SEED, lo, hi), dens == (1, 1, 1))
    got0 = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, 0, 1, SEED, lo, hi)
    got3 = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, 3, 1, SEED, lo, hi)
    check_winners(T, got0, got3, 1, SEED, lo, hi, ref)
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, 0, 1, SEED)
    assert (plan.kernel, plan.lanes) == ("orbit_rt_kernel", 1)
    plan.close()


def test_int64_entry_points(capi):
    T = FX[BIG]
    mkn, (Li, Ri, Pi), dens = F.scaled(T, np.int64)
    assert max(dens) > 2 ** 31
    lo = 2 ** 33 + 5
    hi = lo + 1500
    ref = O.orbit_sweep(*T, 3, 1, SEED, lo, hi)
    check_table(ref, *capi.orbit_table64(mkn, Li, Ri, Pi, dens, 1, SEED, lo, hi), False)
    got0 = capi.orbit_sweep64(mkn, Li, Ri, Pi, dens, 0, 1, SEED, lo, hi)
    got3 = capi.orbit_sweep64(mkn, Li, Ri, Pi, dens, 3, 1, SEED, lo, hi)
    check_winners(T, got0, got3, 1, SEED, lo, hi, ref)


def test_exhaustive_space_122(capi):
    T = FX["naive_1x2x2"]
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    space = capi.orbit_space(*mkn)
    assert space == 4608
    ref = O.orbit_sweep(*T, 3, 0, 0, 0, space)
    check_table(ref, *capi.orbit_table(mkn, Li, Ri, Pi, dens, 0, 0, 0, space), True)
    for measure in (0, 3):
        refb = O.orbit_sweep(*T, measure, 0, 0, 0, space, table=False)["best"]
        got = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, measure, 0, 0, 0, space)
        assert (got["index"], got["nnz"], got["nno"]) == refb[:3]
        if measure == 3:
            assert got["score"] == refb[3]


@pytest.mark.parametrize("name", ["2x2x2_7_Strassen_kron_112", "4x7x3_63_rotated", "naive_2x3x4"])
@pytest.mark.parametrize("p", [3, 513083, 2 ** 31 - 1])
def test_modp(capi, name, p):
    T = FX[name]
    mkn = O.LRP2MM(*T)
    Lr, Rr, Pr = (residues(M, p) for M in T)
    lo = 2 ** 33 + 99
    hi = lo + 1000
    ref = O.orbit_sweep(*T, 0, 1, SEED, lo, hi, p=p)
    nnz, nno = capi.orbit_table_modp(p, mkn, Lr, Rr, Pr, 1, SEED, lo, hi)
    assert np.array_equal(nnz, ref["nnz"]) and np.array_equal(nno, ref["nno"])
    got = capi.orbit_sweep(mkn, Lr, Rr, Pr, (1, 1, 1), 0, 1, SEED, lo, hi, p=p)
    assert (got["index"], got["nnz"], got["nno"]) == ref["best"][:3]
    if p == 2 ** 31 - 1 and name != "4x7x3_63_rotated":  # small integer entries: the residues' counts are the exact ones
        exact = O.orbit_sweep(*T, 3, 1, SEED, lo, hi)
        assert np.array_equal(nnz, exact["nnz"]) and np.array_equal(nno, exact["nno"])


@pytest.mark.parametrize("name", ["2x2x2_7_Winograd_kron_121", "7x3x4_63_rotated", "naive_2x2x8"])
def test_entry_points_agree(capi, name):
    T = FX[name]
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    lo, hi = 1000, 1000 + 40000
    for measure in (0, 3):
        whole = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, measure, 1, SEED, lo, hi)
        cuts = [lo, lo + 1, lo + 12345, lo + 20000, hi]
        parts = [capi.orbit_sweep(mkn, Li, Ri, Pi, dens, measure, 1, SEED, a, b) for a, b in zip(cuts, cuts[1:])]
        key = (lambda g: (g["nnz"], g["nno"], g["index"])) if measure == 0 else (lambda g: (g["score"], g["index"]))
        assert min(parts, key=key) == whole
        assert capi.orbit_sweep_devices(capi.device_count(), mkn, Li, Ri, Pi, dens, measure, 1, SEED, lo, hi) == whole
    # survivors, both measures, with the capacity protocol
    lo, count = 12345, 3001
    ref = O.orbit_sweep(*T, 3, 1, SEED, lo, lo + count)
    idx = np.arange(lo, lo + count, dtype=np.uint64)
    order = np.lexsort((ref["nno"], ref["nnz"]))
    tn, to = int(ref["nnz"][order[count // 50]]), int(ref["nno"][order[count // 50]])
    keep = (ref["nnz"] < tn) | ((ref["nnz"] == tn) & (ref["nno"] <= to))
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, capi.MEASURE_NNZ, 1, SEED)
    got = plan.survivors(lo, lo + count, nnz=tn, nno=to, capacity=8)
    assert [g["index"] for g in got] == idx[keep].tolist()
    assert [g["nnz"] for g in got] == ref["nnz"][keep].tolist() and [g["nno"] for g in got] == ref["nno"][keep].tolist()
    np.testing.assert_allclose([g["score"] for g in got], ref["g2"][keep], rtol=RTOL, atol=0)
    with pytest.raises(capi.PloError):
        import ctypes as C
        cnt = C.c_uint64(0)
        thr = capi.OrbitBest(score=0.0, nnz=tn, nno=to, index=0)
        buf = (capi.OrbitBest * 1)()
        rc = capi.lib().plo_orbit_plan_survivors(plan._h, lo, lo + count, C.byref(thr), 1, buf, C.byref(cnt))
        assert rc == capi.E_RANGE and cnt.value == int(keep.sum())
        capi._check(rc)
    plan.close()
    thr = float(np.quantile(ref["g2"], 0.05))
    plan = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, capi.MEASURE_G2, 1, SEED)
    got = plan.survivors(lo, lo + count, score=thr)
    assert [g["index"] for g in got] == idx[ref["g2"] <= thr].tolist()
    # plan.pack: the winner lands in the plan's device record and from there in its slot
    import torch
    plan.run(lo, lo + count)
    best = plan.result()
    slots = torch.empty(3 * 4, dtype=torch.int64, device="cuda")
    plan.pack(slots.data_ptr(), 1, 3)
    torch.cuda.synchronize()
    s = slots.cpu().numpy()
    big = np.iinfo(np.int64).max
    assert (s[[0, 1, 2, 3, 8, 9, 10, 11]] == big).all()
    assert s[4].view(np.float64) == best["score"] and (s[5], s[6], s[7]) == (best["index"], best["nnz"], best["nno"])
    plan.close()


@pytest.mark.parametrize("name", ["4x7x3_63_rotated", "2x2x2_7_Strassen_kron_211", "naive_2x3x4"])
def test_winner_is_a_valid_algorithm(capi, name):
    T = FX[name]
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    got = capi.orbit_sweep(mkn, Li, Ri, Pi, dens, 0, 1, SEED, 0, 100000)
    U, V, W = capi.orbit_decode(*mkn, 1, SEED, got["index"])
    Lj, Rg, hP = O.orbit_apply(*T, U, V, W)
    assert F.is_algorithm((Lj, Rg, hP))
    assert sum(1 for M in (Lj, Rg, hP) for row in M for v in row if v != 0) == got["nnz"]
    *_, rep = capi.orbiter(*T, seed=5, loops=20000)
    assert rep["mm_verdict"] == 0 and rep["mkn"] == mkn
    recs = capi.orbiter_progress(*T, seed=5, loops=20000)
    keys = [(r["nnz"], r["nno"]) for r in recs]
    assert all(a < b for a, b in zip(keys[1:], keys)) and [r["index"] for r in recs] == sorted(r["index"] for r in recs)


def test_switch_off(capi):
    capi.set_orbit_any_shape(0)
    for name in INT32:
        mkn, (Li, Ri, Pi), dens = F.scaled(FX[name])
        with pytest.raises(capi.PloError) as e:
            capi.orbit_sweep(mkn, Li, Ri, Pi, dens, 0, 1, SEED, 0, 100)
        assert e.value.code == capi.E_SHAPE
    mkn, (Li, Ri, Pi), dens = F.scaled(O.triple("3x3x3_23_58"))
    off = [capi.orbit_sweep(mkn, Li, Ri, Pi, dens, ms, 1, SEED, 0, 50000) for ms in (0, 3)]
    capi.set_orbit_any_shape(1)
    assert [capi.orbit_sweep(mkn, Li, Ri, Pi, dens, ms, 1, SEED, 0, 50000) for ms in (0, 3)] == off
    assert capi.OrbitPlan(mkn, Li, Ri, Pi, dens, 0, 1, SEED).kernel != "orbit_rt_kernel"


def _forced_equal(capi, T, mode, seed, lo, hi):
    mkn, (Li, Ri, Pi), dens = F.scaled(T)
    out = []
    for forced in (False, True):
        if forced:
            os.environ["PLO_ORBIT_RUNTIME_SHAPE"] = "1"
        else:
            os.environ.pop("PLO_ORBIT_RUNTIME_SHAPE", None)
        tab = capi.orbit_table(mkn, Li, Ri, Pi, dens, mode, seed, lo, hi)
        wins = [capi.orbit_sweep(mkn, Li, Ri, Pi, dens, ms, mode, seed, lo, hi) for ms in (0, 3)]
        p = 513083
        Lr, Rr, Pr = (residues(M, p) for M in T)
        modp = (capi.orbit_table_modp(p, mkn, Lr, Rr, Pr, mode, seed, lo, hi), capi.orbit_sweep(mkn, Lr, Rr, Pr, (1, 1, 1), 0, mode, seed, lo, hi, p=p))
        kernel = capi.OrbitPlan(mkn, Li, Ri, Pi, dens, 0, mode, seed).kernel
        out.append((tab, wins, modp, kernel))
    (t0, w0, m0, k0), (t1, w1, m1, k1) = out
    assert all(np.array_equal(a, b) for a, b in zip(t0, t1))
    assert w0 == w1
    assert all(np.array_equal(a, b) for a, b in zip(m0[0], m1[0])) and m0[1] == m1[1]
    assert k0 != "orbit_rt_kernel" and k1 == "orbit_rt_kernel"


def test_forced_parity_winograd_exhaustive(capi):
    _forced_equal(capi, O.triple("2x2x2_7_Winograd"), 0, 0, 0, 110592)


@pytest.mark.parametrize("stem,count", [("3x3x3_23_58", 4000), ("4x4x4_48_rational", 2000), ("3x4x7_63_rational", 1000), ("3x3x6_40", 1000)])
def test_forced_parity_philox(capi, stem, count):
    lo = 2 ** 33 + 17
    _forced_equal(capi, O.triple(stem), 1, SEED, lo, lo + count)


def test_orbiter_cli_any_shape(capi, tmp_path):
    # a dense point of the orbit of Strassen (x) <1,1,2>: the seeded search improves on it
    T = FX["2x2x2_7_Strassen_kron_112"]
    ref = O.orbit_sweep(*T, 0, 1, 7, 0, 2000)
    worst = int(np.lexsort((ref["nno"], ref["nnz"]))[-1])
    dense = O.orbit_apply(*T, *O.orbit_decode(2, 2, 4, 1, 7, worst))
    Lj, Rg, hP, rep = capi.orbiter(*dense, seed=77, loops=20000)
    assert rep["improved"] and rep["mm_verdict"] == 0
    files = []
    for x, M in zip("LRP", dense):
        p = tmp_path / f"dense_{x}.sms"
        hm.write_sms(M, str(p))
        files.append(str(p))
    outs = [f.replace(".sms", ".nnz.sms") for f in files]
    run = lambda extra: subprocess.run([os.path.join(BIN, "orbiter")] + extra + ["-O", "20000", "--seed", "77"] + files, capture_output=True, text=True, timeout=300)
    p = run(["--any-shape"])
    assert p.returncode == 0, p.stderr
    assert [hm.read_sms(o) for o in outs] == [Lj, Rg, hP]
    q = subprocess.run([os.path.join(BIN, "MMchecker")] + outs, capture_output=True, text=True, timeout=300)
    assert q.returncode == 0 and "SUCCESS: correct 2x2x4" in q.stderr
    for o in outs:
        os.remove(o)
    p = run([])
    assert p.returncode != 0 and "not compiled in" in p.stderr
    assert not any(os.path.exists(o) for o in outs)


def test_plans_of_different_shapes_alternate(capi):
    """A runtime-shape plan keeps working after plans and one-shot sweeps of smaller (and larger) shapes were created."""
    lo, hi = 777, 777 + 5000
    big_mkn, big_ints, big_dens = F.scaled(FX["naive_5x5x5"])
    small_mkn, small_ints, small_dens = F.scaled(FX["2x2x2_7_Strassen_kron_112"])
    big = capi.OrbitPlan(big_mkn, *big_ints, big_dens, 0, 1, SEED)
    big.run(lo, hi)
    first = big.result()
    small = capi.OrbitPlan(small_mkn, *small_ints, small_dens, 0, 1, SEED)
    small.run(lo, hi)
    small_first = small.result()
    capi.orbit_table(small_mkn, *small_ints, small_dens, 1, SEED, lo, lo + 100)
    p = 513083
    capi.orbit_sweep(small_mkn, *(residues(M, p) for M in FX["2x2x2_7_Strassen_kron_112"]), (1, 1, 1), 0, 1, SEED, lo, hi, p=p)
    big.run(lo, hi)
    assert big.result() == first
    assert big.survivors(lo, hi, nnz=first["nnz"], nno=first["nno"])[0]["index"] == first["index"]
    small.run(lo, hi)
    assert small.result() == small_first
    big.close()
    small.close()


def test_forced_parity_wide_paths(capi):
    """Triples beyond the int32 product bound (DPS-integral-12.0662, int32 entry points) and 64-bit inputs
    (DPS-intermediate-12.0695): against orbit_wide_kernel, counts and sparsity winners are identical; G2 agrees to a few ulps
    (the two kernels round G2 the same way on paper but differ in the last bit on a few per cent of the candidates)."""
    lo, hi = 2 ** 33 + 17, 2 ** 33 + 17 + 3000
    T = O.triple("2x2x2_7_DPS-integral-12.0662")
    mkn, ints, dens = F.scaled(T)
    assert capi.orbit_magnitude_bounds(mkn, *ints)[0] == 0  # the wide path
    T64 = O.triple("2x2x2_7_DPS-intermediate-12.0695")
    mkn64, ints64, dens64 = F.scaled(T64, np.int64)
    out = []
    for forced in (False, True):
        if forced:
            os.environ["PLO_ORBIT_RUNTIME_SHAPE"] = "1"
        else:
            os.environ.pop("PLO_ORBIT_RUNTIME_SHAPE", None)
        out.append((capi.orbit_table(mkn, *ints, dens, 1, SEED, lo, hi),
                    [capi.orbit_sweep(mkn, *ints, dens, ms, 1, SEED, lo, hi) for ms in (0, 3)],
                    capi.orbit_table64(mkn64, *ints64, dens64, 1, SEED, lo, hi),
                    [capi.orbit_sweep64(mkn64, *ints64, dens64, ms, 1, SEED, lo, hi) for ms in (0, 3)],
                    capi.OrbitPlan(mkn, *ints, dens, 3, 1, SEED).kernel))
    assert (out[0][4], out[1][4]) == ("orbit_wide_kernel", "orbit_rt_kernel")
    for tab, wins in ((0, 1), (2, 3)):
        (n0, o0, g0), (n1, o1, g1) = out[0][tab], out[1][tab]
        assert np.array_equal(n0, n1) and np.array_equal(o0, o1)
        np.testing.assert_allclose(g1, g0, rtol=1e-15, atol=0)
        assert out[0][wins][0] == out[1][wins][0]  # sparsity winner, exact
        a, b = out[0][wins][1], out[1][wins][1]  # G2 winner: the minimum of either table
        assert abs(a["score"] - b["score"]) <= 1e-15 * a["score"]
        assert abs(g0[b["index"] - lo] - g0.min()) <= 1e-15 * g0.min()
