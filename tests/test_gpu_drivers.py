"""GPU parity of the host-level drivers (reference CLIs restated around the kernels) vs the CPU oracle:
the whole sparsifier pipeline must return the SAME CoB and residue as the oracle's literal pipeline
(same documented pivot rule on both sides, quad loops on the GPU vs literal testLinComb on the CPU)."""
import numpy as np
import pytest

import oracle_lib as O
from plinopt_b200 import hm

pytestmark = pytest.mark.gpu

FDT = ["2x2x2_7_DPS-smallrat-12.2034_L", "2x2x2_7_Winograd_R", "2x2x2_7_DPS-accurate_P", "3x3x3_23_58_L", "3x3x6_40_R",
       "4x4x4_48_rational_L", "4x4x4_48_rational_R", "4x4x4_48_accurate_L", "3x4x7_63_rational_L", "3x4x7_63_rational_R",
       "3x4x7_63_rational_P", "4x4x4_49_156_P", "6x3x3_40_L", "cyclic"]


@pytest.mark.parametrize("name", FDT)
@pytest.mark.parametrize("q,c", [(0, 5), (7, 5)])
def test_sparsifier_matches_oracle_pipeline(capi, name, q, c):
    """bin/FDT.sh:64-66 configurations (`-c 5`, `-q 7 -c 5`): consistent factorisation, identical to the oracle's."""
    M = O.dense_fractions(name)
    CoB, Res, ok, st = capi.sparsifier(M, q, 4, c, True)
    eC, eR, eok, _ = O.sparsifier(M, q, 4, c, True)
    assert ok and eok
    assert Res == eR and CoB == eC
    assert st["searches"] > 0 and st["candidates"] >= st["searches"] * 81


def test_c1_config_trace(capi):
    """BASELINE config 1: sparsifier -c 4 data/2x2x2_7_DPS-smallrat-12.2034_L.sms."""
    M = O.dense_fractions("2x2x2_7_DPS-smallrat-12.2034_L")
    CoB, Res, ok, st = capi.sparsifier(M, 0, 4, 4, True)
    eC, eR, eok, tr = O.sparsifier(M, 0, 4, 4, True, trace=True)
    assert ok and (CoB, Res) == (eC, eR)
    # every (block, num) step of the reference loop is covered (c^4 candidate evaluations each), in far fewer device round
    # trips: all rows of an inner block come out of one launch sequence
    assert st["candidates"] == sum(t["c"] ** 4 for t in tr) and 0 < st["searches"] <= len(tr) // 4
    # Res . CoB == M exactly
    prod = [[sum(Res[i][t] * CoB[t][j] for t in range(4)) for j in range(4)] for i in range(7)]
    assert prod == M


@pytest.mark.parametrize("opts", [dict(blocksize=1, maxnumcoeff=4, initial_elimination=True), dict(blocksize=4, maxnumcoeff=6, initial_elimination=False),
                                  dict(blocksize=8, maxnumcoeff=4, initial_elimination=True)])
def test_sparsifier_flag_variants(capi, opts):
    """-b / -U variants: whole-matrix mode (blocksize <= 1), no initial LU, wide blocks (n = 8: two 4-blocks per call)."""
    M = O.dense_fractions("3x3x3_23_58_L") if opts["blocksize"] != 8 else O.dense_fractions("4x4x4_48_rational_R")
    if opts["blocksize"] == 1:
        M = [row[:6] for row in M]
    a = capi.sparsifier(M, 0, **opts)
    b = O.sparsifier(M, 0, opts["blocksize"], opts["maxnumcoeff"], opts["initial_elimination"])
    assert a[2] and (a[0], a[1]) == (b[0], b[1])


def test_c3_config_mod_p31(capi):
    """BASELINE config 3 (single GPU part): sparsifier -q 2147483647 on 4x4x4_48_rational_L, default -c 11."""
    M = O.dense_fractions("4x4x4_48_rational_L")
    q = 2147483647
    CoB, Res, ok, st = capi.sparsifier(M, q, 4, 11, True)
    eC, eR, eok, _ = O.sparsifier(M, q, 4, 11, True)
    assert ok and (CoB, Res) == (eC, eR)
    assert sum(1 for r in Res for v in r if v) < sum(1 for r in M for v in r if v)


def test_orbiter_driver(capi):
    """src/orbiter.cpp:215-360: the returned triple is the oracle's transform of the winner, passes MMchecker,
    and obeys the acceptance rule against the input (:330-331)."""
    for stem, loops in [("2x2x2_7_Winograd", 5000), ("3x3x3_23_58", 20000), ("4x4x4_48_rational", 2000)]:
        L, R, P = O.triple(stem)
        for measure in (0, 3):
            Lj, Rg, hP, rep = capi.orbiter(L, R, P, measure, 1, 77, loops)
            ref = O.orbit_sweep(L, R, P, measure, 1, 77, 0, loops, table=False)["best"]
            assert rep["best"]["index"] == ref[0] and rep["best"]["nnz"] == ref[1] and rep["best"]["nno"] == ref[2]
            assert rep["mm_verdict"] == 0
            if rep["improved"]:
                U, V, W = capi.orbit_decode(*rep["mkn"], 1, 77, rep["best"]["index"])
                assert (Lj, Rg, hP) == O.orbit_apply(L, R, P, U, V, W)
                nnz = sum(1 for M in (Lj, Rg, hP) for row in M for v in row if v != 0)
                assert nnz == rep["best"]["nnz"]
                if measure == 0:
                    assert (nnz, rep["best"]["nno"]) < (rep["init_nnz"], rep["init_nno"])
                else:
                    assert abs(O.growth_G2(Lj, Rg, hP) - rep["best"]["score"]) <= 1e-12 * rep["best"]["score"] < rep["init_score"]
            else:
                assert (Lj, Rg, hP) == (L, R, P)
    # Winograd -> a Strassen-like 14.83 point of the orbit must be found within 5000 candidates
    L, R, P = O.triple("2x2x2_7_Winograd")
    _, _, _, rep = capi.orbiter(L, R, P, 3, 1, 77, 5000)
    assert rep["improved"] and rep["best"]["score"] < 15.0


def test_mmchecker_driver(capi):
    """Makefile:60-64 mmcheck targets through the driver: Strassen over Q; DPS-accurate -m 513083 and -r 1013 2 3."""
    L, R, P = O.triple("2x2x2_7_Strassen")
    assert capi.mmchecker(L, R, P)[0] == 0
    assert capi.mmchecker(L, R, P)[1] == (36, 0)
    L, R, P = O.triple("2x2x2_7_DPS-accurate")
    assert capi.mmchecker(L, R, P, modulus=513083)[0] == 0
    assert capi.mmchecker(L, R, P, modulus=1013 ** 2 - 3)[0] == 0   # factors of 2 stripped (MMchecker.cpp:123-126)
    assert capi.mmchecker(L, R, P)[0] == 1                           # 1013 is only sqrt(3) modulo 513083
    L, R, P = O.triple("3x4x7_63_rational")
    assert capi.mmchecker(L, R, P, batch=64)[0] == 0
    assert capi.mmchecker(L, R[:-1], P)[0] == 2
    assert capi.mmchecker(L, [row[:-1] for row in R], P)[0] == 3


def test_mmchecker_over_Q_is_exact_at_the_sampled_points(capi):
    """include/plinopt_library.inl:497-528 evaluates both sides exactly over Q.  The engine decides the same equality from residues modulo
    enough word-size primes (their product exceeds twice the size of the integer D.(lhs - rhs)): a triple that is a matrix-multiplication
    algorithm modulo 2^31-1 but NOT over Q -- one entry of P shifted by 2^31-1 -- passes the single-prime check and fails the check over Q."""
    from fractions import Fraction
    L, R, P = O.triple("3x4x7_63_rational")
    v, cnt, npr = capi.mmchecker_bits(L, R, P, bitsize=32, seed=3, batch=64)
    assert v == 0 and npr >= 3          # 64 + log2(sum |P||L||R|) + log2(denominators) bits need at least three 31-bit primes
    v8, _, npr8 = capi.mmchecker_bits(L, R, P, bitsize=8, seed=3, batch=64)
    assert v8 == 0 and 1 <= npr8 < npr  # smaller coordinates, smaller integers, fewer primes
    P2 = [list(row) for row in P]
    i, j = next((i, j) for i, row in enumerate(P) for j, x in enumerate(row) if x != 0)
    P2[i][j] = Fraction(P[i][j]) + (2 ** 31 - 1)
    assert capi.mmchecker(L, R, P2, modulus=2 ** 31 - 1, batch=64)[0] == 0      # invisible modulo this prime
    v, _, npr = capi.mmchecker_bits(L, R, P2, bitsize=32, seed=3, batch=64)
    assert v == 1 and npr >= 2                                                    # the second prime sees it
    assert capi.mmchecker(L, R, P2, batch=64)[0] == 1                            # plo_mmchecker: the same decision with 32-bit coordinates


@pytest.mark.parametrize("name,k,q", [("2x2x2_7_Winograd_L", 0, 0), ("4x4x4_48_rational_L", 0, 0), ("4x4x4_48_rational_R", 20, 0),
                                      ("3x4x7_63_rational_R", 0, 0), ("3x3x3_23_58_L", 12, 0), ("4x4x4_48_rational_L", 0, 513083)])
def test_factorizer_matches_oracle_pipeline(capi, name, k, q):
    """plo_factorizer (Factorizer, plinopt_sparsify.inl:924-990): same winner, same Alt and CoB as the oracle's exact sweep
    over the same candidates, M == Alt.CoB (consistency :871-907), never worse than the trivial M = M.I (:958)."""
    M = O.dense_fractions(name)
    r, n = len(M), len(M[0])
    kk = k or n
    loops = 400
    rc, Alt, CoB, rep = capi.factorizer(M, q=q, innerdim=k, loops=loops, seed=99)
    assert rc == 0 and rep["consistent"]
    ref = O.factor_sweep(M, kk, 99, 0, loops, p=q, matrices=True)
    init = (sum(1 for row in M for v in row if v != 0), sum(1 for row in M for v in row if v != 0 and abs(v) != 1), n)
    if q == 0:
        assert rep["initial"] == init
    if ref["best"][:3] < rep["initial"]:
        assert rep["index"] == ref["best"][3] and rep["final"] == ref["best"][:3]
        assert Alt == ref["alt"] and CoB == ref["cob"]
    else:
        assert rep["index"] is None and rep["final"] == rep["initial"]
    if q == 0:
        assert [[sum(Alt[i][t] * CoB[t][j] for t in range(kk)) for j in range(n)] for i in range(r)] == M


def test_factorizer_error_codes(capi):
    M = O.dense_fractions("2x2x2_7_Winograd_L")
    assert capi.factorizer(M, innerdim=3)[0] == -1 and capi.factorizer(M, innerdim=8)[0] == -1  # :936-942
    sq = [row[:] for row in M[:4]]
    rc, Alt, CoB, rep = capi.factorizer(sq)  # square input: identity factorization (:945-951)
    assert rc == 0 and CoB == sq and Alt == [[O.Fraction(int(i == j)) for j in range(4)] for i in range(4)]
    dep = [row[:3] + [row[0]] for row in M]
    with pytest.raises(capi.PloError):
        capi.factorizer(dep)  # not full column rank: backSolver's precondition


@pytest.mark.parametrize("stem,q", [("2x2x2_7_Winograd", 2147483647), ("3x3x3_23_58", 101), ("2x2x2_7_DPS-accurate", 2 * 513083)])
def test_modular_orbiter_driver(capi, stem, q):
    """`orbiter -m q`: factors of 2 stripped (src/orbiter.cpp:421-422), search and acceptance in Z/pZ; the returned triple is the
    oracle's winner transformed in the field and is still a matrix-multiplication algorithm (:355)."""
    L, R, P = O.triple(stem)
    p = q // 2 if q % 2 == 0 else q
    loops = 3000
    Lj, Rg, hP, rep = capi.orbiter_modp(L, R, P, q, seed=5, loops=loops)
    ref = O.orbit_sweep(L, R, P, 0, 1, 5, 0, loops, p=p, table=False)["best"]
    assert (rep["best"]["index"], rep["best"]["nnz"], rep["best"]["nno"]) == ref[:3]
    assert rep["mm_verdict"] == 0
    red = lambda M: [[(v.numerator % p) * pow(v.denominator % p, -1, p) % p for v in row] for row in M]
    if rep["improved"]:
        assert rep["best"]["nnz"] <= rep["init"][0]
        nnz = sum(1 for M in (Lj, Rg, hP) for row in M for v in row if v % p)
        assert nnz == rep["best"]["nnz"]
    else:
        assert (Lj, Rg, hP) == (red(L), red(R), red(P))


@pytest.mark.parametrize("stem", ["2x2x2_7_Strassen", "2x2x2_7_Winograd", "2x2x2_7_DPS-integral-12.0662", "3x3x3_23_58", "4x4x4_48_rational", "3x4x7_63_rational"])
def test_growth_factors(capi, stem):
    """growthfactor (src/growthfactor.cpp:148-231): the eleven printed factors against the oracle's literal restatement (1e-12), and
    the classical values: Strassen gamma_inf,inf = 12, Winograd 18 (Ballard et al.), G2 as in the file names."""
    L, R, P = O.triple(stem)
    got = capi.growth_factors(L, R, P)
    ref = O.growth_factors(L, R, P)
    for name, e in zip(got, ref):
        assert abs(got[name] - e) <= 1e-12 * abs(e), name
    if stem == "2x2x2_7_Strassen":
        assert got["Ginfinf"] == 12.0 and abs(got["G2"] - (12 + 2 * 2 ** 0.5)) < 1e-12 and got["Q0"] == 8.0
    if stem == "2x2x2_7_Winograd":
        assert got["Ginfinf"] == 18.0 and abs(got["G2"] - 17.8530) < 5e-5


def test_blocksparsifier_on_c5_width_blocks(capi):
    """BASELINE config 5 size: column blocks of 32x32x32_15096_L (TM = 4 x 15096 per block: the tiled wide search kernels behind the
    one-row entry point, sparse-row eliminations on the host).  The reference's own check (bin/FDT.sh): consistent factorisation
    M == Res.CoB, and the residue is sparser.  (The whole 15096 x 1024 matrix takes 3.2 s: profiles/sparsifier_c5_r02.jsonl.)"""
    import ctypes as C
    z = hm.load_large()
    if z is None:
        pytest.skip("large fixture absent")
    rows, cols = (int(v) for v in z["L_shape"])
    ncols = 12
    num = np.zeros((rows, ncols), dtype=np.int64); den = np.ones((rows, ncols), dtype=np.int64)
    ri = np.repeat(np.arange(rows), np.diff(z["L_ptr"]))
    sel = z["L_col"] < ncols
    num[ri[sel], z["L_col"][sel]] = z["L_num"][sel]; den[ri[sel], z["L_col"][sel]] = z["L_den"][sel]
    for q in (2147483647, 0):
        cn = np.zeros((ncols, ncols), dtype=np.int64); cd = np.ones((ncols, ncols), dtype=np.int64)
        rn = np.zeros((rows, ncols), dtype=np.int64); rd = np.ones((rows, ncols), dtype=np.int64)
        ok = C.c_int(0)
        stats = np.zeros(3, dtype=np.uint64)
        f = capi.lib().plo_sparsifier
        f.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.POINTER(C.c_int), C.c_void_p, C.c_int]
        rc = f(q, rows, ncols, capi._ptr(num), capi._ptr(den), 4, 5, 1, capi._ptr(cn), capi._ptr(cd), capi._ptr(rn), capi._ptr(rd), C.byref(ok), capi._ptr(stats), -1)
        assert rc == 0, capi.lib().plo_last_error()
        assert ok.value == 1 and np.count_nonzero(rn) < np.count_nonzero(num) and stats[0] > 0
